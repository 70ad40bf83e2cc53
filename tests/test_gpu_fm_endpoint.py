"""Inference at every built attention end point (`--cnn_fm_attention`) on the B200 against the NumPy oracle: the encoder's
feature map at the end point (im_embed and Mixed_5c unchanged), and beam-3 / greedy decoding over 14 x 14 and 7 x 7 maps
at the batch sizes that select the persistent loop (8 images), the sliced / K-split per-step path (25) and the fused /
streaming attention kernels (64).  Tolerances as tests/test_gpu_parity.py: fp32 tensors 2e-4 on the f32-exact path,
1e-3 on attention maps; ids / parents / lengths bit-exact."""
import numpy as np
import pytest

from _common import comic_config, word_config, make_weights, images, fake_features, rel_err

pytestmark = pytest.mark.gpu

TOL = 2e-4
ENDPOINTS = ['MaxPool_4a_3x3', 'Mixed_4b', 'Mixed_4c', 'Mixed_4d', 'Mixed_4e', 'Mixed_4f', 'MaxPool_5a_2x2', 'Mixed_5b',
             'Mixed_5c']


@pytest.fixture(scope='module')
def torch_mod():
    import torch
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    return torch


def _engine(c, W, with_cnn=True, precision='tf32x3'):
    from comic_b200.engine import Engine
    eng = Engine(c)
    eng.bind_weights(W, with_cnn=with_cnn)
    eng.set_precision(precision)
    return eng


@pytest.fixture(scope='module')
def oracle_encoder(torch_mod):
    import inception_v1_oracle as I
    c = comic_config()
    W = make_weights(c)
    img = images(3)
    net, ep = I.inception_v1(img, W)
    return W, img, net[:, 0, 0, :], ep


@pytest.mark.parametrize('precision', ['f32', 'tf32x3'])
@pytest.mark.parametrize('endpoint', ENDPOINTS)
def test_encoder_feature_map_at_end_point(torch_mod, oracle_encoder, endpoint, precision):
    W, img, o_emb, ep = oracle_encoder
    c = comic_config(cnn_fm_attention=endpoint)
    eng = _engine(c, W, precision=precision)
    emb, fm, m5c = eng.encode(eng.to_dev(img), want_mixed5c=True)
    o_fm = ep[endpoint]
    assert fm.shape == (3, o_fm.shape[1] * o_fm.shape[2], o_fm.shape[3])
    assert rel_err(fm.cpu().numpy(), o_fm.reshape(fm.shape)) < TOL
    assert rel_err(m5c.cpu().numpy(), ep['Mixed_5c']) < TOL
    assert rel_err(emb.cpu().numpy(), o_emb) < TOL
    # without the Mixed_5c output, and over two 14 x 14 / 7 x 7 chunks (the end point's per-chunk offsets)
    emb2, fm2 = eng.encode(eng.to_dev(img))
    eng.set_option('enc_chunk_14', 2)
    emb3, fm3 = eng.encode(eng.to_dev(img))
    if precision == 'f32':
        assert torch_mod.equal(fm2, fm) and torch_mod.equal(emb2, emb)
        assert torch_mod.equal(fm3, fm) and torch_mod.equal(emb3, emb)
    else:
        assert rel_err(fm3.cpu().numpy(), fm.cpu().numpy()) < 1e-4


def test_end_point_ids_are_checked_by_the_library(torch_mod):
    """comic_set_fm_endpoint refuses an id it does not build, a config whose feature map is not the end point's, and a
    call after the handle was sized."""
    import ctypes as C
    from comic_b200.engine import Engine
    eng = Engine(comic_config(cnn_fm_attention='Mixed_4c'))
    with pytest.raises(ValueError):                                        # sized by comic_set_fm_endpoint's caller
        n = C.c_size_t()
        eng._check(eng.lib.comic_workspace_bytes(eng._h, 0, 1, 1, 1, C.byref(n)))
        eng._check(eng.lib.comic_set_fm_endpoint(eng._h, 2))
    eng = Engine(comic_config(cnn_fm_attention='Mixed_4c'))
    with pytest.raises(NotImplementedError):
        eng._check(eng.lib.comic_set_fm_endpoint(eng._h, 9))
    with pytest.raises(ValueError, match='fm_channels 512'):
        eng._check(eng.lib.comic_set_fm_endpoint(eng._h, 5))              # Mixed_4f is [14 x 14, 832]


DECODE = {
    'Mixed_4c_tied': lambda: comic_config(cnn_fm_attention='Mixed_4c'),
    'Mixed_4e_none': lambda: comic_config(cnn_fm_attention='Mixed_4e', cnn_fm_projection='none'),          # 66 a head
    'MaxPool_4a_independent': lambda: comic_config(cnn_fm_attention='MaxPool_4a_3x3', cnn_fm_projection='independent'),
    'MaxPool_4a_none': lambda: comic_config(cnn_fm_attention='MaxPool_4a_3x3', cnn_fm_projection='none'),  # 60 a head
    'Mixed_5b_tied': lambda: comic_config(cnn_fm_attention='Mixed_5b'),
    'Mixed_5c_none': lambda: comic_config(cnn_fm_attention='Mixed_5c', cnn_fm_projection='none'),          # VAL 1024
    'word_MaxPool_5a': lambda: word_config(n_words=1000, cnn_fm_attention='MaxPool_5a_2x2'),
}


def _features(c, B, seed):
    from comic_b200 import weights as wts
    d = wts.Dims(c)
    W = make_weights(c, include_cnn=False)
    im, fm = fake_features(B, C=d.C, M=d.M, seed=seed)
    return W, im, fm


@pytest.mark.parametrize('B', [8, 25, 64])
@pytest.mark.parametrize('name', list(DECODE))
def test_beam3_matches_oracle(torch_mod, name, B):
    import comic_oracle as O
    c = DECODE[name]()
    W, im, fm = _features(c, B, seed=B)
    eng = _engine(c, W, with_cnn=False)
    max_it = 8
    ref = O.beam_search_decode(O.Decoder(W, c), im, fm, 3, 0.0, max_it)
    keys, values = eng.project_fm(eng.to_dev(fm))
    c0, h0 = eng.rnn_init(eng.to_dev(im))
    n0 = eng.launch_count()
    r = eng.decode_beam(keys, values, c0, h0, 3, 0.0, max_it)
    if B == 8 and name.endswith('_tied'):
        assert eng.launch_count() - n0 < 16, 'persistent decode loop was not used'
    T = int(r['T'].item())
    assert T == ref['T']
    np.testing.assert_array_equal(r['step_ids'][:T].cpu().numpy(), ref['step_ids'])
    np.testing.assert_array_equal(r['parent_ids'][:T].cpu().numpy(), ref['parent_ids'])
    np.testing.assert_array_equal(r['predicted_ids'][:T].cpu().numpy(), ref['predicted_ids'])
    np.testing.assert_array_equal(r['lengths'].cpu().numpy(), ref['lengths'])
    np.testing.assert_allclose(r['scores'][:T].cpu().numpy(), ref['scores'], rtol=1e-4, atol=1e-4)
    _, _, am = O.post_process_beam(ref, c.attn_num_heads, 3)
    assert rel_err(r['attn'][:, :, :T].cpu().numpy(), am) < 1e-3


@pytest.mark.parametrize('B', [8, 25])
@pytest.mark.parametrize('name', list(DECODE))
def test_greedy_matches_oracle(torch_mod, name, B):
    import comic_oracle as O
    c = DECODE[name]()
    W, im, fm = _features(c, B, seed=B + 1)
    eng = _engine(c, W, with_cnn=False)
    ref = O.greedy_decode(O.Decoder(W, c), im, fm, 10)
    keys, values = eng.project_fm(eng.to_dev(fm))
    c0, h0 = eng.rnn_init(eng.to_dev(im))
    r = eng.decode_greedy(keys, values, c0, h0, 10)
    T = int(r['T'].item())
    assert T == ref['T']
    np.testing.assert_array_equal(r['ids'][:T].cpu().numpy(), ref['ids'])
    assert rel_err(r['logits'][:T].cpu().numpy(), ref['logits']) < 1e-3
    _, _, am = O.post_process_plain(ref['logits'], ref['ids'], ref['alignment_history'], c.attn_num_heads)
    assert rel_err(r['attn'][:, :, :T].cpu().numpy(), am) < 1e-3


@pytest.mark.parametrize('endpoint', ['Mixed_4c', 'Mixed_5b'])
def test_caption_model_end_to_end(torch_mod, endpoint):
    """images -> encoder -> beam-3 through CaptionModel (the inference surface) equals the oracle's captions."""
    import comic_oracle as O
    import inception_v1_oracle as I
    from comic_b200 import configuration as conf
    from comic_b200.model import CaptionModel
    c = conf.make_config(infer_max_length=4, cnn_fm_attention=endpoint)
    W = make_weights(c, seed=3)
    img = images(2, seed=4)
    m = CaptionModel(c, 'infer', batch_ops=[img], weights=W)
    preds, attn = m.infer_output
    emb, fm, _ = I.encoder(img, W, c)
    ref = O.beam_search_decode(O.Decoder(W, c), emb, fm, 3, 0.0)
    _, ids, am = O.post_process_beam(ref, 8, 3)
    assert np.array_equal(preds, ids)
    assert rel_err(attn, am) < 1e-3

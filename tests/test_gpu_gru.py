"""GRU decoder cell (rnn_name=GRU) on the B200 against the NumPy oracle (tests/gru_oracle.py): the init step, one
wrapper step (with and without the training masks), beam search and greedy decode on the FFMA and tensor paths, and
the repack of the weights bound by pointer."""
import numpy as np
import pytest

from _common import comic_config, word_config, make_weights, fake_features, images, rel_err
import comic_oracle as O
import gru_oracle as GO

TOL = 2e-4

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def torch_mod():
    import torch
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    return torch


CONFIGS = {
    'comic256': lambda **kw: comic_config(rnn_name='GRU', **kw),
    'project_hidden': lambda **kw: comic_config(rnn_name='GRU', rnn_init_method='project_hidden', **kw),
    'dot_sigmoid_ctx_h4': lambda **kw: comic_config(rnn_name='GRU', attn_alignment_method='dot', attn_probability_fn='sigmoid',
                                                    attn_context_layer=True, cnn_fm_projection='independent', attn_num_heads=4,
                                                    **kw),
    'word_none_h1': lambda **kw: word_config(n_words=1000, rnn_name='GRU', **kw),
}


def _engine(c, W, precision='tf32x3', with_cnn=False):
    from comic_b200.engine import Engine
    eng = Engine(c)
    eng.bind_weights(W, with_cnn=with_cnn)
    eng.set_precision(precision)
    return eng


@pytest.mark.parametrize('precision', ['f32', 'tf32x3'])
@pytest.mark.parametrize('name,B,k', [('comic256', 3, 3), ('project_hidden', 3, 3), ('dot_sigmoid_ctx_h4', 2, 3),
                                      ('word_none_h1', 3, 3), ('comic256', 48, 3), ('word_none_h1', 48, 3)])
def test_gru_decode_step_matches_oracle(torch_mod, name, B, k, precision):
    """rnn_init + one wrapper step; 144 rows put both GRU GEMMs on the tcgen05 path (tf32x3)."""
    c = CONFIGS[name]()
    W = make_weights(c, include_cnn=False)
    eng = _engine(c, W, precision)
    im, fm = fake_features(B)
    dec = GO.GRUDecoder(W, c)
    dec.setup_memory(O.tile_batch(fm, k))
    _, h0 = dec.init_state(O.tile_batch(im, k))
    state = dec.zero_state(dec.init_state(O.tile_batch(im, k)))
    rng = np.random.default_rng(11)
    state['attention'] = rng.standard_normal(state['attention'].shape).astype(np.float32) * 0.3
    state['h'] = np.tanh(state['h'] + rng.standard_normal(state['h'].shape).astype(np.float32) * 0.1)
    toks = rng.integers(0, dec.V, size=(B * k,)).astype(np.int32)
    if c.token_type == 'radix':
        toks[0] = -1
    cell_out, ns, al = dec.call(dec.embed(toks), state)
    logits = dec.output_layer(cell_out)

    keys, values = eng.project_fm(eng.to_dev(fm))
    gc0, gh0 = eng.rnn_init(eng.to_dev(im))
    assert gc0 is None
    assert rel_err(gh0.cpu().numpy(), h0[::k]) < TOL
    r = eng.decode_step(keys, values, B, k, eng.to_dev(toks), None, eng.to_dev(state['h']), eng.to_dev(state['attention']))
    assert r['c'] is None
    assert rel_err(r['h'].cpu().numpy(), ns['h']) < TOL
    assert rel_err(r['logits'].cpu().numpy(), logits) < TOL
    assert rel_err(r['alignments'].cpu().numpy(), al) < TOL
    assert rel_err(r['attention'].cpu().numpy(), ns['attention']) < TOL


def test_gru_decode_step_train_masks(torch_mod):
    """Input / output dropout of the DropoutWrapper and attention-map dropout with explicit masks, init step included."""
    c = CONFIGS['comic256']()
    W = make_weights(c, include_cnn=False)
    eng = _engine(c, W)
    B = 4
    im, fm = fake_features(B)
    dec = GO.GRUDecoder(W, c)
    dec.setup_memory(fm)
    rng = np.random.default_rng(2)
    keeps = (0.65, 0.65, 0.9)
    init_mask = (rng.uniform(size=(B, 768)) < keeps[0]).astype(np.float32)
    _, h0 = dec.init_state(im, init_mask, keeps[0])
    state = dec.zero_state(dec.init_state(im, init_mask, keeps[0]))
    state['attention'] = rng.standard_normal(state['attention'].shape).astype(np.float32) * 0.3
    toks = rng.integers(0, 258, size=(B,)).astype(np.int32)
    in_mask = (rng.uniform(size=(B, 768)) < keeps[0]).astype(np.float32)
    out_mask = (rng.uniform(size=(B, 512)) < keeps[1]).astype(np.float32)
    att_mask = (rng.uniform(size=(B, 8, 196)) < keeps[2]).astype(np.float32)
    cell_out, ns, al = dec.call(dec.embed(toks), state, in_mask, out_mask, att_mask, *keeps)
    logits = dec.output_layer(cell_out)
    keys, values = eng.project_fm(eng.to_dev(fm))
    _, gh0 = eng.rnn_init(eng.to_dev(im), eng.to_dev(init_mask), keeps[0])
    assert rel_err(gh0.cpu().numpy(), h0) < TOL
    r = eng.decode_step(keys, values, B, 1, eng.to_dev(toks), None, eng.to_dev(state['h']),
                        eng.to_dev(state['attention']), eng.to_dev(in_mask), eng.to_dev(out_mask),
                        eng.to_dev(att_mask.reshape(B, -1)), keeps)
    assert rel_err(r['h'].cpu().numpy(), ns['h']) < TOL          # state h is undropped
    assert rel_err(r['logits'].cpu().numpy(), logits) < TOL      # logits use the dropped output
    assert rel_err(r['alignments'].cpu().numpy(), al) < TOL
    assert rel_err(r['attention'].cpu().numpy(), ns['attention']) < TOL


def _beam_vs_oracle(eng, W, c, B, k, max_it, seed=0):
    im, fm = fake_features(B, seed=seed + 3)
    ref = O.beam_search_decode(GO.GRUDecoder(W, c), im, fm, k, 0.0, max_it)
    keys, values = eng.project_fm(eng.to_dev(fm))
    c0, h0 = eng.rnn_init(eng.to_dev(im))
    n0 = eng.launch_count()
    r = eng.decode_beam(keys, values, c0, h0, k, 0.0, max_it)
    T = int(r['T'].item())
    assert T == ref['T']
    assert eng.launch_count() - n0 >= 5 * T                       # per-step path: no persistent loop for the GRU
    np.testing.assert_array_equal(r['step_ids'][:T].cpu().numpy(), ref['step_ids'])
    np.testing.assert_array_equal(r['parent_ids'][:T].cpu().numpy(), ref['parent_ids'])
    np.testing.assert_array_equal(r['predicted_ids'][:T].cpu().numpy(), ref['predicted_ids'])
    np.testing.assert_array_equal(r['lengths'].cpu().numpy(), ref['lengths'])
    np.testing.assert_allclose(r['scores'][:T].cpu().numpy(), ref['scores'], rtol=1e-4, atol=1e-4)
    _, _, am = O.post_process_beam(ref, c.attn_num_heads, k)
    assert rel_err(r['attn'][:, :, :T].cpu().numpy(), am) < 1e-3


@pytest.mark.parametrize('precision', ['f32', 'tf32x3'])
@pytest.mark.parametrize('name,B,max_it', [('comic256', 4, 12), ('comic256', 8, 10), ('comic256', 25, 8),
                                           ('comic256', 64, 5), ('project_hidden', 4, 8), ('dot_sigmoid_ctx_h4', 3, 6)])
def test_gru_beam_search_matches_oracle(torch_mod, name, B, max_it, precision):
    """4 images: FFMA GEMMs; 8 x 3 rows: what the persistent loop would take for the LSTM; 25 images: K-split tensor
    GEMMs; 64 images: tensor path with the streaming attention kernel."""
    c = CONFIGS[name]()
    W = make_weights(c, include_cnn=False)
    _beam_vs_oracle(_engine(c, W, precision), W, c, B, 3, max_it)


def test_gru_beam_search_word_model_v10000(torch_mod):
    c = word_config(n_words=10000, rnn_name='GRU')
    W = make_weights(c, include_cnn=False)
    _beam_vs_oracle(_engine(c, W), W, c, 4, 3, 6)


@pytest.mark.parametrize('precision', ['f32', 'tf32x3'])
def test_gru_greedy_matches_oracle(torch_mod, precision):
    c = CONFIGS['comic256']()
    W = make_weights(c, include_cnn=False)
    eng = _engine(c, W, precision)
    im, fm = fake_features(5, seed=3)
    ref = O.greedy_decode(GO.GRUDecoder(W, c), im, fm, 12)
    keys, values = eng.project_fm(eng.to_dev(fm))
    c0, h0 = eng.rnn_init(eng.to_dev(im))
    r = eng.decode_greedy(keys, values, c0, h0, 12)
    T = int(r['T'].item())
    assert T == ref['T']
    np.testing.assert_array_equal(r['ids'][:T].cpu().numpy(), ref['ids'])
    assert rel_err(r['logits'][:T].cpu().numpy(), ref['logits']) < TOL
    _, _, am = O.post_process_plain(ref['logits'], ref['ids'], ref['alignment_history'], 8)
    assert rel_err(r['attn'][:, :, :T].cpu().numpy(), am) < 1e-3


def test_gru_refresh_packed_follows_weights_updated_in_place(torch_mod):
    """The four GRU variables are bound by pointer: after an in-place update (what the optimiser does to the Trainer's
    flat buffer) comic_refresh_packed rebuilds the gate panel and the tensor-path packs from them, and a decode equals
    one of an engine bound fresh to the updated weights, bit for bit."""
    torch = torch_mod
    c = CONFIGS['comic256']()
    W = make_weights(c, include_cnn=False)
    B, k, max_it = 25, 3, 6
    im, fm = fake_features(B, seed=7)
    eng = _engine(c, W)
    rng = np.random.default_rng(4)
    W2 = dict(W)
    for n in W:
        if '/gru_cell/' in n:
            W2[n] = (W[n] + rng.standard_normal(W[n].shape).astype(np.float32) * 0.05).astype(np.float32)
            eng._dev_weights[n].copy_(torch.as_tensor(W2[n]))
    eng.refresh_packed()

    def run(e):
        keys, values = e.project_fm(e.to_dev(fm))
        c0, h0 = e.rnn_init(e.to_dev(im))
        r = e.decode_beam(keys, values, c0, h0, k, 0.0, max_it)
        return r['predicted_ids'].cpu().numpy(), r['scores'].cpu().numpy(), r['attn'].cpu().numpy()
    got, want = run(eng), run(_engine(c, W2))
    for a, b in zip(got, want):
        np.testing.assert_array_equal(a, b)


def test_gru_caption_model_end_to_end(torch_mod):
    """images -> CaptionModel('infer') with a GRU config vs the oracle encoder + GRU beam search."""
    import inception_v1_oracle as I
    from comic_b200.model import CaptionModel
    c = CONFIGS['comic256'](infer_max_length=6)
    W = make_weights(c)
    img = images(3, seed=8)
    preds, attn = CaptionModel(c, 'infer', batch_ops=[img], weights=W).infer_output
    o_emb, o_fm, _ = I.encoder(img, W, c)
    ref = O.beam_search_decode(GO.GRUDecoder(W, c), o_emb, o_fm, 3, 0.0)
    _, ids, am = O.post_process_beam(ref, 8, 3)
    np.testing.assert_array_equal(preds, ids)
    assert rel_err(attn, am) < 1e-3


def test_gru_engine_refusals(torch_mod):
    from comic_b200.engine import ComicError, Engine
    with pytest.raises(ComicError, match='rnn_name=LN_LSTM is not built'):
        Engine(comic_config(rnn_name='LN_LSTM'))
    c = CONFIGS['comic256']()
    W = make_weights(c, include_cnn=False)
    W.pop(GO.O.DEC + 'rnn_init_input/gru_cell/candidate/kernel')
    with pytest.raises(ValueError):                                # comic_bind_gru_candidate: null kernel
        Engine(c).bind_weights(W, with_cnn=False)

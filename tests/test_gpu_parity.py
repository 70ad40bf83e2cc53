"""GPU parity tests: the CUDA path (through the C ABI) against the NumPy oracle
on the same seeded inputs.  Tolerances: fp32 tensors 1e-3 relative (north_star)
-- the f32-exact path is held to 2e-4; ids / parents / lengths bit-exact."""
import numpy as np
import pytest

from _common import comic_config, word_config, make_weights, images, fake_features, rel_err

pytestmark = pytest.mark.gpu

TOL = 2e-4


@pytest.fixture(scope='module')
def torch_mod():
    import torch
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    return torch


def _engine(c, W, with_cnn=True, precision='tf32x3', fused=None):
    """fused: True = one-CTA-per-image fused attention at any batch; False = sliced kernels (both on the
    one-launch-per-op path); 'persistent' = the whole decode loop as one cooperative kernel (the
    default for <= 32 rows); None = engine defaults."""
    from comic_b200.engine import Engine
    eng = Engine(c)
    eng.bind_weights(W, with_cnn=with_cnn)
    eng.set_precision(precision)
    if fused in (True, False):
        eng.set_option('fused_attn_min_images', 1 if fused else 1 << 30)
        eng.set_option('persistent_max_rows', 0)
    return eng


def _check_path(eng, fused, launches_before, max_it):
    """The persistent path enqueues O(1) kernels per decode call, the per-step path >= 5 per step."""
    n = eng.launch_count() - launches_before
    if fused == 'persistent':
        assert n < 16, 'persistent decode loop was not used (%d launches)' % n
    elif fused in (True, False):
        assert n >= 5 * max_it


@pytest.mark.parametrize('precision', ['f32', 'tf32x3'])
@pytest.mark.parametrize('M,N,K', [(24, 2048, 1280), (7, 64, 36), (300, 132, 147), (1536, 772, 512),
                                   (129, 68, 520), (64, 2048, 768), (1000, 448, 528), (4096, 64, 32),
                                   (256, 2048, 1280)])
def test_gemm_f32(torch_mod, M, N, K, precision):
    """The dense kernel alone: FFMA path and tcgen05 3xTF32 path (M >= 128) vs fp64."""
    torch = torch_mod
    c = comic_config()
    eng = _engine(c, make_weights(c, include_cnn=False), with_cnn=False, precision=precision)
    rng = np.random.default_rng(M + N + K)
    A = rng.standard_normal((M, K)).astype(np.float32)
    Bm = rng.standard_normal((K, N)).astype(np.float32)
    bias = rng.standard_normal((N,)).astype(np.float32)
    out = eng.gemm(eng.to_dev(A), eng.to_dev(Bm), eng.to_dev(bias)).cpu().numpy()
    ref = A.astype(np.float64) @ Bm.astype(np.float64) + bias
    # FFMA: fp32 round-off only.  3xTF32: dropped lo*lo term (2^-22) plus the tensor core's
    # truncating fp32 accumulation, measured ~6e-6 at K = 1280.
    assert rel_err(out, ref) < (1e-5 if precision == 'f32' else 5e-5)


@pytest.mark.parametrize('precision', ['f32', 'tf32x3'])
def test_encoder_matches_oracle(torch_mod, precision):
    import inception_v1_oracle as I
    c = comic_config()
    W = make_weights(c)
    eng = _engine(c, W, precision=precision)
    img = images(3)
    emb, fm, m5c = eng.encode(eng.to_dev(img), want_mixed5c=True)
    o_emb, o_fm, ep = I.encoder(img, W, c)
    assert fm.shape == (3, 196, 832) and emb.shape == (3, 1024)
    assert rel_err(fm.cpu().numpy(), o_fm) < TOL
    assert rel_err(m5c.cpu().numpy(), ep['Mixed_5c']) < TOL
    assert rel_err(emb.cpu().numpy(), o_emb) < TOL


def test_encoder_chunking_batch_independent(torch_mod):
    """Images are independent units: a batch of 70 (two chunks) == singles.  Bit-identical
    on the FFMA path; the tensor path switches kernels with the row count (M < 128 -> FFMA),
    so it is compared at tolerance."""
    c = comic_config()
    W = make_weights(c)
    img = images(70, seed=5)
    eng = _engine(c, W, precision='f32')
    for name, n in (('enc_chunk_stem', 64), ('enc_chunk_28', 48), ('enc_chunk_14', 40)):   # 64+6, 48+22, 40+30
        eng.set_option(name, n)
    emb, fm = eng.encode(eng.to_dev(img))
    emb1, fm1 = eng.encode(eng.to_dev(img[67:68]))
    assert torch_mod.equal(fm[67:68], fm1)
    assert torch_mod.equal(emb[67:68], emb1)
    eng.set_precision('tf32x3')
    emb2, fm2 = eng.encode(eng.to_dev(img))
    assert rel_err(fm2.cpu().numpy(), fm.cpu().numpy()) < 1e-4
    assert rel_err(emb2.cpu().numpy(), emb.cpu().numpy()) < 1e-4
    # tensor path, stem conv: 4x4 stride-1 conv over the space-to-depth bf16-plane image (default) vs the
    # 7x7 stride-2 gather from the NHWC4 fp32 image -- the same products in a different summation order
    eng.set_option('stem_s2d', 0)
    emb5, fm5 = eng.encode(eng.to_dev(img))
    assert rel_err(fm5.cpu().numpy(), fm2.cpu().numpy()) < 5e-5
    assert rel_err(emb5.cpu().numpy(), emb2.cpu().numpy()) < 5e-5
    eng.set_option('stem_s2d', 2)


CONFIGS = {
    'comic256': lambda: comic_config(),
    'word_none_h1': lambda: word_config(n_words=1000),
    'independent_h4': lambda: comic_config(cnn_fm_projection='independent', attn_num_heads=4),
    'dot_sigmoid': lambda: comic_config(attn_alignment_method='dot', attn_probability_fn='sigmoid'),
    'legacy': lambda: comic_config(legacy=True),
    'context_layer': lambda: comic_config(attn_context_layer=True, cnn_fm_projection='none'),
}


@pytest.mark.parametrize('fused', [False, True])
@pytest.mark.parametrize('name', list(CONFIGS))
def test_decode_step_matches_oracle(torch_mod, name, fused):
    import comic_oracle as O
    torch = torch_mod
    c = CONFIGS[name]()
    W = make_weights(c, include_cnn=False)
    eng = _engine(c, W, with_cnn=False, fused=fused)
    B, k = 3, 3
    im, fm = fake_features(B)
    dec = O.Decoder(W, c)
    dec.setup_memory(O.tile_batch(fm, k))
    c0, h0 = dec.init_state(O.tile_batch(im, k))
    state = dec.zero_state((c0, h0))
    rng = np.random.default_rng(11)
    state['attention'] = rng.standard_normal(state['attention'].shape).astype(np.float32) * 0.3
    state['c'] = state['c'] + rng.standard_normal(state['c'].shape).astype(np.float32) * 0.1
    state['h'] = np.tanh(state['h'] + rng.standard_normal(state['h'].shape).astype(np.float32) * 0.1)
    toks = rng.integers(0, dec.V, size=(B * k,)).astype(np.int32)
    if c.token_type == 'radix':
        toks[0] = -1                     # PAD -> one-hot zero row
    cell_out, new_state, al = dec.call(dec.embed(toks), state)
    logits = dec.output_layer(cell_out)

    fm_d = eng.to_dev(fm)
    keys, values = eng.project_fm(fm_d)
    assert rel_err(keys.cpu().numpy(), dec.keys[::k]) < TOL
    gc0, gh0 = eng.rnn_init(eng.to_dev(im))
    assert rel_err(gc0.cpu().numpy(), c0[::k]) < TOL
    assert rel_err(gh0.cpu().numpy(), h0[::k]) < TOL
    r = eng.decode_step(keys, values, B, k, eng.to_dev(toks), eng.to_dev(state['c']), eng.to_dev(state['h']),
                        eng.to_dev(state['attention']))
    assert rel_err(r['c'].cpu().numpy(), new_state['c']) < TOL
    assert rel_err(r['h'].cpu().numpy(), new_state['h']) < TOL
    assert rel_err(r['logits'].cpu().numpy(), logits) < TOL
    assert rel_err(r['alignments'].cpu().numpy(), al) < TOL
    assert rel_err(r['attention'].cpu().numpy(), new_state['attention']) < TOL
    a = r['alignments'].cpu().numpy().reshape(B * k, c.attn_num_heads, -1)
    np.testing.assert_allclose(a.sum(-1), 1.0, atol=1e-5)       # alpha sums to 1 per head


@pytest.mark.parametrize('name', ['comic256', 'word_none_h1'])
def test_decode_step_large_rows_tensor_path(torch_mod, name):
    """N = 144 rows: gate / logits|query GEMMs run on the tcgen05 3xTF32 kernel with
    the beam-state row indirection and the 3-segment A operand."""
    import comic_oracle as O
    c = CONFIGS[name]()
    W = make_weights(c, include_cnn=False)
    eng = _engine(c, W, with_cnn=False)
    B, k = 48, 3
    im, fm = fake_features(B)
    dec = O.Decoder(W, c)
    dec.setup_memory(O.tile_batch(fm, k))
    c0, h0 = dec.init_state(O.tile_batch(im, k))
    state = dec.zero_state((c0, h0))
    rng = np.random.default_rng(5)
    state['attention'] = rng.standard_normal(state['attention'].shape).astype(np.float32) * 0.3
    toks = rng.integers(0, dec.V, size=(B * k,)).astype(np.int32)
    cell_out, ns, al = dec.call(dec.embed(toks), state)
    logits = dec.output_layer(cell_out)
    keys, values = eng.project_fm(eng.to_dev(fm))
    r = eng.decode_step(keys, values, B, k, eng.to_dev(toks), eng.to_dev(state['c']), eng.to_dev(state['h']),
                        eng.to_dev(state['attention']))
    assert rel_err(r['h'].cpu().numpy(), ns['h']) < TOL
    assert rel_err(r['logits'].cpu().numpy(), logits) < TOL
    assert rel_err(r['alignments'].cpu().numpy(), al) < TOL
    assert rel_err(r['attention'].cpu().numpy(), ns['attention']) < TOL


@pytest.mark.parametrize('fused', [False, True])
def test_decode_step_train_masks(torch_mod, fused):
    """DropoutWrapper in/out masks + attention-map dropout with explicit masks."""
    import comic_oracle as O
    c = comic_config()
    W = make_weights(c, include_cnn=False)
    eng = _engine(c, W, with_cnn=False, fused=fused)
    B = 4
    im, fm = fake_features(B)
    dec = O.Decoder(W, c)
    dec.setup_memory(fm)
    rng = np.random.default_rng(2)
    keeps = (0.65, 0.65, 0.9)
    init_mask = (rng.uniform(size=(B, 768)) < keeps[0]).astype(np.float32)
    c0, h0 = dec.init_state(im, init_mask, keeps[0])
    state = dec.zero_state((c0, h0))
    state['attention'] = rng.standard_normal(state['attention'].shape).astype(np.float32) * 0.3
    toks = rng.integers(0, 258, size=(B,)).astype(np.int32)
    in_mask = (rng.uniform(size=(B, 768)) < keeps[0]).astype(np.float32)
    out_mask = (rng.uniform(size=(B, 512)) < keeps[1]).astype(np.float32)
    att_mask = (rng.uniform(size=(B, 8, 196)) < keeps[2]).astype(np.float32)
    cell_out, ns, al = dec.call(dec.embed(toks), state, in_mask, out_mask, att_mask, *keeps)
    logits = dec.output_layer(cell_out)
    keys, values = eng.project_fm(eng.to_dev(fm))
    gc0, gh0 = eng.rnn_init(eng.to_dev(im), eng.to_dev(init_mask), keeps[0])
    assert rel_err(gc0.cpu().numpy(), c0) < TOL
    r = eng.decode_step(keys, values, B, 1, eng.to_dev(toks), eng.to_dev(state['c']), eng.to_dev(state['h']),
                        eng.to_dev(state['attention']), eng.to_dev(in_mask), eng.to_dev(out_mask),
                        eng.to_dev(att_mask.reshape(B, -1)), keeps)
    assert rel_err(r['h'].cpu().numpy(), ns['h']) < TOL          # state h is undropped
    assert rel_err(r['logits'].cpu().numpy(), logits) < TOL      # logits use the dropped output
    assert rel_err(r['alignments'].cpu().numpy(), al) < TOL
    assert rel_err(r['attention'].cpu().numpy(), ns['attention']) < TOL


def _beam_state(rng, B, k, V, with_finished):
    log_probs = -rng.uniform(0, 10, size=(B, k)).astype(np.float32)
    finished = np.zeros((B, k), bool)
    lengths = rng.integers(0, 9, size=(B, k)).astype(np.int64)
    if with_finished:
        finished = rng.uniform(size=(B, k)) < 0.4
    return log_probs, finished, lengths


@pytest.mark.parametrize('B,k,V,lpw,fin', [(5, 3, 258, 0.0, False), (4, 3, 258, 0.0, True),
                                           (3, 7, 258, 0.7, True), (2, 3, 10000, 0.0, True),
                                           (1, 1, 300, 0.0, False), (6, 5, 64, 1.0, True),
                                           (3, 4, 5000, 0.7, True), (2, 7, 3000, 0.0, False),
                                           (70, 3, 258, 0.0, True), (65, 3, 258, 0.7, True), (64, 1, 300, 0.0, False)])
def test_beam_step_bit_exact(torch_mod, B, k, V, lpw, fin):
    """K10 given identical total log-probs: ids / parents / lengths / finished
    bit-exact, ties -> lower flat index."""
    import comic_oracle as O
    torch = torch_mod
    c = comic_config()
    eng = _engine(c, make_weights(c, include_cnn=False), with_cnn=False)
    rng = np.random.default_rng(B * 100 + k)
    # coarse grid of logits so that exact ties occur and log-softmax differences are far above 1 ulp
    logits = (rng.integers(-8, 8, size=(B, k, V)) * 0.5).astype(np.float32)
    eos = V - 1
    lp, finished, lengths = _beam_state(rng, B, k, V, fin)
    if not fin:
        lp[:, 1:] = -np.inf; lp[:, 0] = 0          # the init state of BeamSearchDecoder.initialize
        finished[:, 1:] = True
        lengths[:] = 0
    top, word, parent, new_lp, new_fin, new_len, total = O.beam_search_step(
        logits, lp.copy(), finished.copy(), lengths.copy(), k, eos, lpw)
    d_lp, d_fin, d_len = eng.to_dev(lp), eng.to_dev(finished.astype(np.uint8)), eng.to_dev(lengths)
    g_top, g_word, g_parent = eng.beam_step(eng.to_dev(logits), d_lp, d_fin, d_len, eos, lpw)
    # device log-softmax (expf/logf) may differ from NumPy by an ulp: ids must agree wherever the
    # oracle's margin to the next candidate is not a float tie-break artefact.
    np.testing.assert_array_equal(g_word.cpu().numpy(), word)
    np.testing.assert_array_equal(g_parent.cpu().numpy(), parent)
    np.testing.assert_array_equal(d_fin.cpu().numpy().astype(bool), new_fin)
    np.testing.assert_array_equal(d_len.cpu().numpy(), new_len)
    np.testing.assert_allclose(g_top.cpu().numpy(), top, rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(d_lp.cpu().numpy(), new_lp, rtol=1e-5, atol=1e-5)


@pytest.mark.parametrize('B,k,V,lpw', [(6, 3, 10000, 0.0), (4, 5, 7001, 0.7), (3, 8, 4000, 0.0), (5, 3, 10000, 0.7)])
def test_beam_step_large_vocabulary_threshold_selection(torch_mod, B, k, V, lpw):
    """Word vocabularies with ordinary (tie-free) logits: the block's score threshold keeps a handful of the k x V
    candidates and the exact top-k is drawn from those (search_steps.cuh); the coarse-grid cases of
    test_beam_step_bit_exact overflow the candidate list instead and take the k-pass fallback."""
    import comic_oracle as O
    c = comic_config()
    eng = _engine(c, make_weights(c, include_cnn=False), with_cnn=False)
    rng = np.random.default_rng(1000 + B * 10 + k)
    logits = (rng.standard_normal((B, k, V)) * 3).astype(np.float32)
    eos = V - 1
    lp, finished, lengths = _beam_state(rng, B, k, V, True)
    top, word, parent, new_lp, new_fin, new_len, total = O.beam_search_step(
        logits, lp.copy(), finished.copy(), lengths.copy(), k, eos, lpw)
    d_lp, d_fin, d_len = eng.to_dev(lp), eng.to_dev(finished.astype(np.uint8)), eng.to_dev(lengths)
    g_top, g_word, g_parent = eng.beam_step(eng.to_dev(logits), d_lp, d_fin, d_len, eos, lpw)
    np.testing.assert_array_equal(g_word.cpu().numpy(), word)
    np.testing.assert_array_equal(g_parent.cpu().numpy(), parent)
    np.testing.assert_array_equal(d_fin.cpu().numpy().astype(bool), new_fin)
    np.testing.assert_array_equal(d_len.cpu().numpy(), new_len)
    np.testing.assert_allclose(g_top.cpu().numpy(), top, rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(d_lp.cpu().numpy(), new_lp, rtol=1e-5, atol=1e-5)


def test_gather_tree_bit_exact(torch_mod):
    import comic_oracle as O
    c = comic_config()
    eng = _engine(c, make_weights(c, include_cnn=False), with_cnn=False)
    rng = np.random.default_rng(9)
    T, B, k, eos = 13, 6, 4, 257
    step_ids = rng.integers(0, 256, size=(T, B, k)).astype(np.int32)
    step_ids[rng.uniform(size=step_ids.shape) < 0.08] = eos
    parents = rng.integers(0, k, size=(T, B, k)).astype(np.int32)
    msl = np.array([13, 0, 5, 20, 1, 9], np.int32)
    ref = O.gather_tree(step_ids, parents, msl, eos)
    out = eng.gather_tree(eng.to_dev(step_ids), eng.to_dev(parents), eng.to_dev(msl), eos)
    np.testing.assert_array_equal(out.cpu().numpy(), ref)


def _decode_inputs(c, B, seed=0):
    W = make_weights(c, include_cnn=False)
    im, fm = fake_features(B, seed=seed + 3)
    return W, im, fm


@pytest.mark.parametrize('fused', [False, True, 'persistent'])
@pytest.mark.parametrize('name,B,k,max_it', [('comic256', 4, 3, 14), ('word_none_h1', 3, 3, 8),
                                             ('comic256', 2, 7, 10), ('independent_h4', 2, 2, 6),
                                             ('comic256', 8, 3, 60), ('comic256', 1, 1, 5), ('comic256', 10, 3, 9)])
def test_beam_search_matches_oracle(torch_mod, name, B, k, max_it, fused):
    import comic_oracle as O
    c = CONFIGS[name]()
    W, im, fm = _decode_inputs(c, B)
    eng = _engine(c, W, with_cnn=False, fused=fused)
    ref = O.beam_search_decode(O.Decoder(W, c), im, fm, k, 0.0, max_it)
    keys, values = eng.project_fm(eng.to_dev(fm))
    c0, h0 = eng.rnn_init(eng.to_dev(im))
    n0 = eng.launch_count()
    r = eng.decode_beam(keys, values, c0, h0, k, 0.0, max_it)
    _check_path(eng, fused, n0, max_it)
    T = int(r['T'].item())
    assert T == ref['T']
    np.testing.assert_array_equal(r['step_ids'][:T].cpu().numpy(), ref['step_ids'])
    np.testing.assert_array_equal(r['parent_ids'][:T].cpu().numpy(), ref['parent_ids'])
    np.testing.assert_array_equal(r['predicted_ids'][:T].cpu().numpy(), ref['predicted_ids'])
    np.testing.assert_array_equal(r['lengths'].cpu().numpy(), ref['lengths'])
    np.testing.assert_allclose(r['scores'][:T].cpu().numpy(), ref['scores'], rtol=1e-4, atol=1e-4)
    _, _, am = O.post_process_beam(ref, c.attn_num_heads, k)
    assert rel_err(r['attn'][:, :, :T].cpu().numpy(), am) < 1e-3


@pytest.mark.parametrize('fused', [True, 'persistent'])
def test_beam_search_eos_and_early_stop(torch_mod, fused):
    """Bias the output layer towards EOS so beams finish: exercises _mask_probs,
    length bookkeeping, gather_tree EOS back-fill and the all-finished stop."""
    import comic_oracle as O
    from comic_b200 import weights as wts
    c = comic_config()
    W, im, fm = _decode_inputs(c, 5, seed=4)
    b = W[wts.DEC + 'output_projection/bias'].copy()
    b[257] += 3.2
    W[wts.DEC + 'output_projection/bias'] = b
    eng = _engine(c, W, with_cnn=False, fused=fused)
    ref = O.beam_search_decode(O.Decoder(W, c), im, fm, 3, 0.0, 40)
    keys, values = eng.project_fm(eng.to_dev(fm))
    c0, h0 = eng.rnn_init(eng.to_dev(im))
    r = eng.decode_beam(keys, values, c0, h0, 3, 0.0, 40)
    T = int(r['T'].item())
    assert ref['T'] < 40, 'test should stop early'
    assert T == ref['T']
    np.testing.assert_array_equal(r['predicted_ids'][:T].cpu().numpy(), ref['predicted_ids'])
    np.testing.assert_array_equal(r['parent_ids'][:T].cpu().numpy(), ref['parent_ids'])
    np.testing.assert_array_equal(r['lengths'].cpu().numpy(), ref['lengths'])
    _, _, am = O.post_process_beam(ref, 8, 3)
    assert rel_err(r['attn'][:, :, :T].cpu().numpy(), am) < 1e-3


@pytest.mark.parametrize('fused', [False, True, 'persistent'])
def test_greedy_matches_oracle(torch_mod, fused):
    import comic_oracle as O
    c = comic_config()
    W, im, fm = _decode_inputs(c, 5)
    eng = _engine(c, W, with_cnn=False, fused=fused)
    ref = O.greedy_decode(O.Decoder(W, c), im, fm, 12)
    keys, values = eng.project_fm(eng.to_dev(fm))
    c0, h0 = eng.rnn_init(eng.to_dev(im))
    n0 = eng.launch_count()
    r = eng.decode_greedy(keys, values, c0, h0, 12)
    _check_path(eng, fused, n0, 12)
    T = int(r['T'].item())
    assert T == ref['T']
    np.testing.assert_array_equal(r['ids'][:T].cpu().numpy(), ref['ids'])
    assert rel_err(r['logits'][:T].cpu().numpy(), ref['logits']) < TOL
    _, _, am = O.post_process_plain(ref['logits'], ref['ids'], ref['alignment_history'], 8)
    assert rel_err(r['attn'][:, :, :T].cpu().numpy(), am) < 1e-3


def test_fast_tanh_mode_within_north_star_tolerance(torch_mod):
    """precision 'fast' (tanh.approx.f32 in the LN-tanh) stays inside the 1e-3 bound."""
    import comic_oracle as O
    c = comic_config()
    W = make_weights(c, include_cnn=False)
    eng = _engine(c, W, with_cnn=False, precision='fast', fused=True)
    B, k = 4, 3
    im, fm = fake_features(B)
    dec = O.Decoder(W, c)
    dec.setup_memory(O.tile_batch(fm, k))
    state = dec.zero_state(dec.init_state(O.tile_batch(im, k)))
    rng = np.random.default_rng(3)
    toks = rng.integers(0, dec.V, size=(B * k,)).astype(np.int32)
    cell_out, ns, al = dec.call(dec.embed(toks), state)
    keys, values = eng.project_fm(eng.to_dev(fm))
    r = eng.decode_step(keys, values, B, k, eng.to_dev(toks), eng.to_dev(state['c']), eng.to_dev(state['h']),
                        eng.to_dev(state['attention']))
    assert rel_err(r['alignments'].cpu().numpy(), al) < 1e-3
    assert rel_err(r['attention'].cpu().numpy(), ns['attention']) < 1e-3


def test_golden_decoder_beam_fixture_gpu(torch_mod):
    """The committed fixture tests/golden/decoder_beam_comic256.npz (oracle output, frozen)."""
    import os
    import make_golden as G
    g = np.load(os.path.join(os.path.dirname(G.__file__), 'decoder_beam_comic256.npz'))
    c = comic_config()
    W = G.golden_weights(c, False)
    im, fm = G.decoder_inputs(4, 77)
    for fused in (False, True):
        eng = _engine(c, W, with_cnn=False, fused=fused)
        keys, values = eng.project_fm(eng.to_dev(fm))
        c0, h0 = eng.rnn_init(eng.to_dev(im))
        r = eng.decode_beam(keys, values, c0, h0, 3, 0.0, 10)
        np.testing.assert_array_equal(r['predicted_ids'].cpu().numpy(), g['predicted_ids'])
        np.testing.assert_array_equal(r['parent_ids'].cpu().numpy(), g['parent_ids'])
        np.testing.assert_array_equal(r['lengths'].cpu().numpy(), g['lengths'])
        assert rel_err(r['scores'].cpu().numpy(), g['scores']) < 1e-4
        assert rel_err(r['attn'].cpu().numpy(), g['attn_top']) < 1e-3


def test_golden_encoder_fixture_gpu(torch_mod):
    import os
    import make_golden as G
    g = np.load(os.path.join(os.path.dirname(G.__file__), 'encoder_2img.npz'))
    c = comic_config()
    W = G.golden_weights(c, True)
    rng = np.random.default_rng(5)
    img = rng.uniform(-1, 1, (2, 224, 224, 3)).astype(np.float32)
    for precision in ('f32', 'tf32x3'):
        eng = _engine(c, W, precision=precision)
        emb, fm = eng.encode(eng.to_dev(img))
        fm = fm.cpu().numpy()
        assert rel_err(emb.cpu().numpy(), g['im_embed']) < TOL
        assert rel_err(fm[:, ::7, ::13], g['fm_sample']) < TOL
        # checksum of the whole map: the tensor-core path accumulates with truncation (round toward
        # zero) inside the MMA, a systematic ~4e-5 shrink after 20 layers; FFMA rounds to nearest
        bias = abs(float(fm.astype(np.float64).sum()) - float(g['fm_sum'])) / float(g['fm_sum'])
        assert bias < (1e-5 if precision == 'f32' else 2e-4), (precision, bias)


def test_caption_model_end_to_end(torch_mod):
    """images -> CaptionModel('infer').infer_output vs oracle encoder+beam search."""
    import comic_oracle as O
    import inception_v1_oracle as I
    from comic_b200.model import CaptionModel
    c = comic_config(infer_max_length=6)           # 12 radix steps
    W = make_weights(c)
    img = images(3, seed=8)
    m = CaptionModel(c, 'infer', batch_ops=[img], weights=W)
    preds, attn = m.infer_output
    o_emb, o_fm, _ = I.encoder(img, W, c)
    ref = O.beam_search_decode(O.Decoder(W, c), o_emb, o_fm, 3, 0.0)
    _, ids, am = O.post_process_beam(ref, 8, 3)
    np.testing.assert_array_equal(preds, ids)
    assert attn.shape == am.shape
    assert rel_err(attn, am) < 1e-3


def test_run_stream_pipeline_matches_run(torch_mod):
    """CaptionModel.run_stream (H2D / compute / D2H overlapped over 3 streams) returns, batch by batch and
    bit for bit, what the blocking `run` returns -- pinned host batches, pageable ones and an empty loop."""
    from comic_b200.model import CaptionModel
    torch = torch_mod
    c = comic_config(infer_max_length=4)
    W = make_weights(c)
    m = CaptionModel(c, 'infer', weights=W)
    batches = [images(3, seed=s) for s in (1, 2, 3, 4, 5)]
    want = []
    for b in batches:
        p, a = m.run(b)
        want.append((p.copy(), a.copy()))
    hosts = [torch.from_numpy(b).pin_memory() if i % 2 == 0 else b for i, b in enumerate(batches)]
    n = 0
    for (p, a), (wp, wa) in zip(m.run_stream(iter(hosts)), want):
        np.testing.assert_array_equal(p, wp)
        np.testing.assert_array_equal(a, wa)
        n += 1
    assert n == len(batches)
    assert list(m.run_stream([])) == []
    # a second pass reuses the slots; a single batch drains correctly
    (p, a), = list(m.run_stream([hosts[0]]))
    np.testing.assert_array_equal(p, want[0][0])


def test_run_inference_driver_on_engine(torch_mod, tmp_path):
    """inference.run_inference (src/infer_fn.py:76-184) over the CUDA engine: captions in the json are
    id_to_caption of what the blocking `run` decodes for the same images, whole batches only."""
    import json
    from comic_b200 import inference as inf
    from comic_b200.model import CaptionModel
    from comic_b200.scst import id_to_caption
    c = comic_config(infer_max_length=4)
    c.batch_size_infer = 3
    c.save_attention_maps = True
    c.infer_save_path = str(tmp_path)
    m = CaptionModel(c, 'infer', weights=make_weights(c))
    batches = [images(3, seed=s) for s in (1, 2, 3)]
    files = ['COCO_val2014_%012d.jpg' % i for i in range(8)]            # 8 files -> 2 whole batches of 3
    want = [cap for b in batches[:2] for cap in id_to_caption(m.run(b)[0], c)]
    raw, coco, _ = inf.run_inference(c, 'model_compact-77', m, files, iter(batches))
    assert [e['caption'] for e in coco] == want and [e['image_id'] for e in coco] == list(range(6))
    assert json.load(open(tmp_path / 'captions___77.json')) == coco
    np.testing.assert_array_equal(raw['attention'][files[4]], m.run(batches[1])[1][1])


@pytest.mark.parametrize('B,H,W,out_hw', [(2, 37, 53, (224, 224)), (1, 480, 640, (224, 224)), (3, 256, 256, (224, 224)),
                                          (1, 500, 333, (300, 200)), (2, 224, 224, (224, 224))])
def test_preprocess_eval_bit_exact(torch_mod, B, H, W, out_hw):
    """comic_preprocess_eval (uint8 -> resize 256 bilinear -> crop / pad -> (x - 0.5) * 2, fused) against the NumPy
    restatement of inception_preprocessing_radix.py:229-235, 270-273: same fp32 operations, bit-exact."""
    import inception_v1_oracle as I
    torch = torch_mod
    c = comic_config()
    eng = _engine(c, make_weights(c, include_cnn=False), with_cnn=False)
    x = np.random.default_rng(B * 1000 + H + W).integers(0, 256, size=(B, H, W, 3), dtype=np.uint8)
    got = eng.preprocess_eval(torch.from_numpy(x).to(eng.device), out_hw).cpu().numpy()
    np.testing.assert_array_equal(got, I.preprocess_eval(x, out_hw))
    with pytest.raises(ValueError):
        eng.preprocess_eval(torch.zeros((1, 8, 8, 3), device=eng.device))


def test_errors(torch_mod):
    from comic_b200.engine import Engine
    with pytest.raises(ValueError):
        Engine(comic_config(attn_alignment_method='add'))        # src/model_base.py:133-138
    c = comic_config()
    eng = Engine(c)
    with pytest.raises(Exception):
        eng.project_fm(eng.f32(2, 196, 832))                     # weights not bound


def test_cli_drivers_run(torch_mod, capsys):
    """`python -m comic_b200.cli infer|train` (the reference's infer.py / train.py flag surface) on synthetic batches."""
    from comic_b200 import cli
    assert cli.main(['infer', '--batch_size_infer', '3', '--infer_max_length', '3', '--synthetic_batches', '2']) == 0
    assert 'captions/s' in capsys.readouterr().out
    assert cli.main(['train', '--train_mode', 'decoder', '--batch_size_train', '4', '--synthetic_steps', '2']) == 0
    out = capsys.readouterr().out
    assert 'steps/s' in out and 'step    2' in out


@pytest.mark.parametrize('case', ['STEP', 'STEP_WITH_EOS'])
def test_beam_step_kernel_reproduces_tf19_unit_test(torch_mod, case):
    """The CUDA beam step on TensorFlow r1.9's own test vectors (tests/golden/tf19_vectors.py)."""
    import os
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden'))
    import tf19_vectors as TV
    c = comic_config()
    eng = _engine(c, make_weights(c, include_cnn=False), with_cnn=False)
    v = getattr(TV, case)
    d_lp = eng.to_dev(TV.initial_log_probs())
    d_fin = eng.to_dev(v['finished'].astype(np.uint8))
    d_len = eng.to_dev(v['lengths'])
    _top, word, parent = eng.beam_step(eng.to_dev(v['logits']), d_lp, d_fin, d_len, TV.END_TOKEN, TV.LENGTH_PENALTY)
    np.testing.assert_array_equal(word.cpu().numpy(), v['predicted_ids'])
    np.testing.assert_array_equal(parent.cpu().numpy(), v['parent_ids'])
    np.testing.assert_array_equal(d_len.cpu().numpy(), v['next_lengths'])
    np.testing.assert_array_equal(d_fin.cpu().numpy().astype(bool), v['next_finished'])


def test_gather_tree_kernel_reproduces_tf19_unit_test(torch_mod):
    import os
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden'))
    import tf19_vectors as TV
    c = comic_config()
    eng = _engine(c, make_weights(c, include_cnn=False), with_cnn=False)
    g = TV.GATHER_TREE
    out = eng.gather_tree(eng.to_dev(g['step_ids']), eng.to_dev(g['parent_ids']), eng.to_dev(g['max_sequence_lengths']),
                          g['end_token'])
    np.testing.assert_array_equal(out.cpu().numpy(), g['expected'])


def test_rnn_decoder_training_matches_oracle(torch_mod):
    """rops.rnn_decoder_training (common/ops_rnn.py:183-243): ragged lengths, impute_finished, padding by the last step."""
    import comic_oracle as O
    from comic_b200 import rops
    c = comic_config()
    W = make_weights(c, include_cnn=False)
    eng = _engine(c, W, with_cnn=False)
    B, T = 4, 9
    im, fm = fake_features(B, seed=23)
    rng = np.random.default_rng(6)
    ids = rng.integers(0, 256, size=(B, T)).astype(np.int32)
    lens = np.array([7, 3, 5, 1], np.int32)
    ref = O.training_decode(O.Decoder(W, c), im, fm, ids, lens)
    d_im, d_fm = eng.to_dev(im), eng.to_dev(fm)
    am = rops.MultiHeadAddLN(c.rnn_size, d_fm, c.cnn_fm_projection, c.attn_num_heads, engine=eng)
    cell = rops.MultiHeadAttentionWrapperV3(context_layer=c.attn_context_layer, cell=c.rnn_name, attention_mechanism=am,
                                            initial_cell_state=rops.LSTMStateTuple(*eng.rnn_init(d_im)))
    with pytest.raises(ValueError):
        rops.rnn_decoder_training(cell, ids.T, None, B, lens)
    cell.im_embed = d_im
    out_ids, rnn_out, state = rops.rnn_decoder_training(cell, ids.T, None, B, lens)
    assert rnn_out.shape == (T, B, 258) and state.time == ref['T_run'] == 7
    assert rel_err(rnn_out.cpu().numpy(), ref['logits']) < TOL
    np.testing.assert_array_equal(out_ids.cpu().numpy(), ref['ids'])
    hist = ref['alignment_history'].reshape(ref['T_run'], B, 8, 196).transpose(1, 2, 0, 3)
    assert rel_err(state.alignment_history.cpu().numpy(), hist) < 1e-3


@pytest.mark.parametrize('B,H,W', [(3, 240, 320), (2, 480, 640), (2, 100, 75)])
def test_preprocess_train_bit_exact(torch_mod, B, H, W):
    """comic_preprocess_train (resize 256 -> flip -> crop at the given corner -> standardise) against the NumPy
    restatement of preprocess_for_train with the same draws."""
    import inception_v1_oracle as I
    from comic_b200.train import random_crop_flip
    torch = torch_mod
    c = comic_config()
    eng = _engine(c, make_weights(c, include_cnn=False), with_cnn=False)
    rng = np.random.default_rng(H + W)
    x = rng.integers(0, 256, (B, H, W, 3), dtype=np.uint8)
    crop, flip = random_crop_flip(B, rng=rng)
    crop[0] = (0, 32)                                # the corners of the offset range
    crop[-1] = (32, 0)
    flip[0], flip[-1] = 1, 0
    got = eng.preprocess_train(torch.from_numpy(x).to(eng.device), crop, flip).cpu().numpy()
    np.testing.assert_array_equal(got, I.preprocess_train(x, crop, flip))
    with pytest.raises(ValueError):
        eng.preprocess_train(torch.from_numpy(x).to(eng.device), np.array([[0, 33]] * B), flip)

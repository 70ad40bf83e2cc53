"""The encoder and the beam decode against the oracles at the batch the benchmark decodes (bench.py: 512 images per GPU,
1,536 beam rows, 60 steps, the default encoder chunks 256 / 512 / 512, the device step replayed as a CUDA graph).

The kernels pick their launch variants from the row count and the SM count, so the small batches of the other parity
tests never reach several of the variants the benchmark runs (gemm_tc.cuh: launch_gemm_tc, pick_bn):
  - the resident-weight-panel convolutions (gemm_bf16x3_bres_kernel) need N <= 64 and at least 2 x SMs M tiles: the
    14 x 14 Branch_3 1 x 1 convs of Mixed_4b-4e (K = 480 / 512, bres<2, 8>) from 193 images per chunk on 148 SMs, the
    28 x 28 Branch_3 convs of Mixed_3b / 3c (bres<4, 4>) from 49;
  - convolutions take 256-wide tiles, several per persistent CTA, once a launch is more than a wave (128-wide below);
  - the stem's second 256-image chunk exists only for B > 256;
  - at 1,536 rows pick_bn's cost rule gives the LSTM gate GEMM 176-wide tiles, [logits | query] 128 (the word model's,
    V = 10,000: 256, 504 tiles, several per CTA through both TMEM accumulators) and the GRU gate GEMM 128; at the
    <= 192 rows of the other tests these are all 64 or 176.
test_launch_variants_at_the_bench_shape restates those rules and asserts that the shapes below reach them on this
device.  Tolerances are those of the smaller tests (encoder 2e-4, decode scores 2e-4, attention maps 1e-3, ids / parents
exact except at audited oracle near-ties), but taken per image: one wrong tile would vanish in a whole-batch maximum.

Run with -s for the launch table, the worst errors and each phase's wall time."""
import resource
import time

import numpy as np
import pytest

from _common import comic_config, word_config, make_weights, images, fake_features
from test_gpu_parity_large import margin_audit

pytestmark = pytest.mark.gpu

B = 512                      # bench.py --batch default
BEAM = 3
ENC_CHUNKS = (256, 512, 512)  # comic_internal.cuh enc_chunk: stem / 28 x 28 blocks / 14 x 14 + 7 x 7 blocks
ENC_TOL = 2e-4
BM, BK = 128, 64             # gemm_tc.cuh M tile and K block


@pytest.fixture(scope='module')
def torch_mod():
    import torch
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    return torch


@pytest.fixture(scope='module')
def sms(torch_mod):
    return torch_mod.cuda.get_device_properties(0).multi_processor_count


class _phase(object):
    """Prints the wall time of a block and the process's peak host memory so far."""

    def __init__(self, what):
        self.what = what

    def __enter__(self):
        self.t0 = time.perf_counter()

    def __exit__(self, *exc):
        print('[%6.1f s, peak host RSS %.1f GB] %s' % (time.perf_counter() - self.t0,
                                                       resource.getrusage(resource.RUSAGE_SELF).ru_maxrss / 2 ** 20,
                                                       self.what))


# ---------------------------------------------------------------------------
# Launch rules of gemm_tc.cuh, restated
# ---------------------------------------------------------------------------
def _cdiv(a, b):
    return -(-a // b)


def pick_bn(M, N, sms, small_ok):
    """gemm_tc.cuh pick_bn."""
    if N <= 64:
        return 64
    if N <= 128:
        return 128
    mt = _cdiv(M, BM)
    if small_ok and mt * _cdiv(N, 256) < sms:
        return min((256, 176, 128, 64), key=lambda bn: _cdiv(mt * _cdiv(N, bn), sms) * (bn + 48))   # first minimum wins
    if mt * _cdiv(N, 256) < sms and mt * _cdiv(N, 128) <= sms:
        return 128
    return 256


def conv_variant(M, N, K, KH, Cin, sms):
    """launch_gemm_tc<1> (im2col convolution) -> (variant, tiles)."""
    mt = _cdiv(M, BM)
    if 256 < N <= 352 and K >= 512:
        return '176', mt * _cdiv(N, 176)
    if N == 192 and KH == 3 and Cin == 64:
        return '192', mt
    bn = pick_bn(M, N, sms, False)
    if bn == 64 and mt >= 2 * sms:
        nkb = _cdiv(K, BK)
        for stages, nkres in ((4, 4), (3, 6), (2, 8)):
            if nkb <= nkres:
                return 'bres<%d,%d>' % (stages, nkres), mt
    return str(bn), mt * _cdiv(N, bn)


def gemm_variant(M, N, K, sms, ksplit_ok):
    """launch_gemm_tc<0 / 4> of a dense GEMM -> (variant, tiles); ksplit_ok: the caller applies tc_ksplit
    (comic_internal.cuh tc_ksplit_shape), whose launches take 128-wide tiles."""
    if ksplit_ok:
        tiles = _cdiv(M, 128) * _cdiv(N, 128)
        ks = max(min(sms // tiles, _cdiv(K, 64) // 2, 8), 1)
        if ks >= 2:
            return 'splitK%d,128' % ks, tiles * ks
    bn = pick_bn(M, N, sms, True)
    return str(bn), _cdiv(M, BM) * _cdiv(N, bn)


def encoder_launches(nimg, sms):
    """[(launch, M, N, K, variant, tiles)] of the tensor-path encoder on one chunk of each stage (encoder.cu
    encoder_forward, fp32 activations), keyed by the chunk sizes the default plan gives `nimg` images."""
    from comic_b200 import weights as wts
    cs, c3, c4 = (min(nimg, c) for c in ENC_CHUNKS)
    out = [('Conv2d_1a_7x7 (stem halo, chunk %d)' % cs, cs * 12544, 64, 256, 'bres<3,4>', cs * 98)]
    for name, S, nb, K, KH, cin, n in (('Conv2d_2b_1x1', 56, cs, 64, 1, 64, 64), ('Conv2d_2c_3x3', 56, cs, 576, 3, 64, 192)):
        out.append((name, nb * S * S, n, K) + conv_variant(nb * S * S, n, K, KH, cin, sms))
    for blk in wts.BLOCKS:
        if len(blk) == 3:
            continue
        name, cin, b0, b1a, b1b, b2a, b2b, b3 = blk
        S, nb = (28, c3) if name.startswith('Mixed_3') else (14, c4) if name.startswith('Mixed_4') else (7, c4)
        M = nb * S * S
        ng = b0 + b1a + b2a
        out.append((name + ' [b0|b1a|b2a] 1x1', M, ng, cin) + gemm_variant(M, ng, cin, sms, False))
        out.append((name + ' Branch_1 3x3', M, b1b, 9 * b1a) + conv_variant(M, b1b, 9 * b1a, 3, b1a, sms))
        out.append((name + ' Branch_2 3x3', M, b2b, 9 * b2a) + conv_variant(M, b2b, 9 * b2a, 3, b2a, sms))
        out.append((name + ' Branch_3 1x1', M, b3, cin) + conv_variant(M, b3, cin, 1, cin, sms))
    return out


def decoder_launches(c, nimg, sms):
    """[(launch, M, N, K, variant, tiles)] of one beam-3 decode step's tensor-path GEMMs (decoder.cu run_step /
    run_gru_cell / step_tail with the default options: LSTM gate GEMM from the loader warps, [logits | query] from the
    TMA-staged planes; the GRU's GEMMs all from the loader warps)."""
    from comic_b200 import weights as wts
    d = wts.Dims(c)
    M, KX, LQ = nimg * BEAM, d.W + d.A + d.R, _cdiv(d.V, 4) * 4 + d.R
    if c.rnn_name == 'GRU':
        return [('GRU gate GEMM', M, 3 * d.R, KX) + gemm_variant(M, 3 * d.R, KX, sms, True),
                ('GRU candidate GEMM', M, d.R, d.R) + gemm_variant(M, d.R, d.R, sms, True),
                ('[logits | query]', M, LQ, d.R) + gemm_variant(M, LQ, d.R, sms, M <= 128)]
    return [('LSTM gate GEMM', M, 4 * d.R, KX) + gemm_variant(M, 4 * d.R, KX, sms, True),
            ('[logits | query] (TMA planes)', M, LQ, d.R) + gemm_variant(M, LQ, d.R, sms, False)]


def _find(rows, prefix):
    hit = [r for r in rows if r[0].startswith(prefix)]
    assert len(hit) == 1, prefix
    return hit[0]


def test_launch_variants_at_the_bench_shape(sms):
    """The 512-image shapes of this file reach the launch variants named in the module docstring on this device."""
    enc = encoder_launches(B, sms)
    dec = {name: decoder_launches(c, B, sms) for name, c in (('comic256', comic_config()), ('GRU', comic_config(rnn_name='GRU')),
                                                             ('word V=10000', word_config(n_words=10000)))}
    print('\nlaunch variants at %d images / %d beam rows on %d SMs' % (B, B * BEAM, sms))
    print('%-44s %8s %6s %6s %-12s %6s' % ('launch', 'M', 'N', 'K', 'variant', 'tiles'))
    for title, rows in [('encoder', enc)] + [('decoder ' + k, v) for k, v in dec.items()]:
        print('-- ' + title)
        for r in rows:
            print('%-44s %8d %6d %6d %-12s %6d' % r)

    why = ' on this device (%d SMs): the 512-image tests below do not reach this path' % sms
    for blk in ('Mixed_4b', 'Mixed_4c', 'Mixed_4d', 'Mixed_4e'):
        r = _find(enc, blk + ' Branch_3')
        assert r[4] == 'bres<2,8>', '%s takes %s%s' % (r[0], r[4], why)
    for blk in ('Mixed_3b', 'Mixed_3c'):
        r = _find(enc, blk + ' Branch_3')
        assert r[4] == 'bres<4,4>', '%s takes %s%s' % (r[0], r[4], why)
    r = _find(enc, 'Mixed_5c Branch_1')
    assert r[4] == '256' and r[5] > sms, '%s takes %s x %d tiles%s' % (r[0], r[4], r[5], why)
    assert B > ENC_CHUNKS[0], 'no second stem chunk'
    r = _find(dec['comic256'], 'LSTM gate GEMM')
    assert r[4] == '176', '%s takes %s%s' % (r[0], r[4], why)
    r = _find(dec['comic256'], '[logits | query]')
    assert r[4] == '128', '%s takes %s%s' % (r[0], r[4], why)
    r = _find(dec['word V=10000'], '[logits | query]')
    assert r[4] == '256' and r[5] > sms, '%s takes %s x %d tiles%s' % (r[0], r[4], r[5], why)
    r = _find(dec['GRU'], 'GRU gate GEMM')
    assert r[4] == '128', '%s takes %s%s' % (r[0], r[4], why)


# ---------------------------------------------------------------------------
# 1. Encoder at 512 images, default chunks and precision
# ---------------------------------------------------------------------------
def _per_image_err(got, ref):
    """max |got - ref| / max |ref| over each image's tensor."""
    n = got.shape[0]
    g = got.reshape(n, -1).astype(np.float64)
    r = ref.reshape(n, -1).astype(np.float64)
    return np.abs(g - r).max(axis=1) / (np.abs(r).max(axis=1) + 1e-30)


def _where(b):
    """Chunk position of image b in the default plan, and its M tiles at 28 x 28 / 14 x 14."""
    cs, c3, c4 = ENC_CHUNKS
    p3, p4 = b % c3, b % c4
    return ('stem chunk %d; 28x28 chunk %d image %d (M tiles %d-%d); 14x14 chunk %d image %d (M tiles %d-%d)'
            % (b // cs, b // c3, p3, p3 * 784 // BM, (p3 * 784 + 783) // BM, b // c4, p4, p4 * 196 // BM,
               (p4 * 196 + 195) // BM))


@pytest.fixture(scope='module')
def enc512(torch_mod):
    """The engine (CNN bound, engine defaults) and its encoding of images(512, seed=41)."""
    from comic_b200.engine import Engine
    c = comic_config()
    W = make_weights(c)
    img = images(B, seed=41)
    eng = Engine(c)
    eng.bind_weights(W, with_cnn=True)
    dev = eng.to_dev(img)
    with _phase('GPU encode, %d images' % B):
        emb, fm, m5c = eng.encode(dev, want_mixed5c=True)
        out = dict(emb=emb.cpu().numpy(), fm=fm.cpu().numpy(), m5c=m5c.cpu().numpy())
    return dict(c=c, W=W, img=img, dev=dev, eng=eng, out=out)


def test_encoder_512_images_matches_oracle_per_image(enc512):
    import inception_v1_oracle as I
    img, W, c, got = enc512['img'], enc512['W'], enc512['c'], enc512['out']
    ref = dict(emb=[], fm=[], m5c=[])
    with _phase('oracle encoder, %d images in host chunks of 32' % B):
        for b0 in range(0, B, 32):
            emb, fm, ep = I.encoder(img[b0:b0 + 32], W, c)
            ref['emb'].append(emb)
            ref['fm'].append(fm)
            ref['m5c'].append(ep['Mixed_5c'])
    for key in ('fm', 'emb', 'm5c'):
        err = _per_image_err(got[key], np.concatenate(ref[key]))
        b = int(np.argmax(err))
        print('encoder %-4s worst per-image error %.2e at image %d (%s)' % (key, err[b], b, _where(b)))
        assert err[b] <= ENC_TOL, '%s: image %d is %.2e from the oracle (%s); %d images over %.0e' % (
            key, b, err[b], _where(b), int((err > ENC_TOL).sum()), ENC_TOL)


def test_encoder_300_images_partial_second_stem_chunk(enc512, sms):
    """300 images: stem chunks 256 + 44, one 28 x 28 and one 14 x 14 chunk of 300.  On 148 SMs every launch keeps the
    variant it has at 512 images (same tile widths, resident panels still >= 2 x SMs M tiles), and a row's result does
    not depend on the tile it lands in, so the outputs equal the 512-image ones bit for bit."""
    changed = [(a[0], a[4], b[4]) for a, b in zip(encoder_launches(B, sms), encoder_launches(300, sms)) if a[4] != b[4]]
    print('launch variants that differ between 512 and 300 images: %s' % changed)
    eng, got = enc512['eng'], enc512['out']
    with _phase('GPU encode, 300 images'):
        emb, fm, m5c = eng.encode(enc512['dev'][:300], want_mixed5c=True)
    for key, t in (('fm', fm), ('emb', emb), ('m5c', m5c)):
        a = t.cpu().numpy()
        err = _per_image_err(a, got[key][:300])
        b = int(np.argmax(err))
        print('300 vs 512 images, %-4s: worst per-image difference %.2e at image %d, bit-identical: %s'
              % (key, err[b], b, np.array_equal(a, got[key][:300])))
        assert err[b] <= 5e-5, '%s: image %d (%s) differs by %.2e between the 300- and 512-image calls' % (
            key, b, _where(b), err[b])
        if not changed:
            assert np.array_equal(a, got[key][:300]), key


# ---------------------------------------------------------------------------
# 2-4. Beam-3 decodes at 1,536 rows against the oracle
# ---------------------------------------------------------------------------
# name -> (config, max_it, steps checked on all 512 images, size of the image sample checked over every step)
DECODE_CASES = {
    'comic256': (lambda: comic_config(), 60, 6, 32),
    'word_v10000': (lambda: word_config(n_words=10000), 30, 3, 24),
    'gru': (lambda: comic_config(rnn_name='GRU'), 60, 3, 24),
}


def _sample(n):
    """n images spread over the batch, both ends of each 256-image half included."""
    idx = np.unique(np.r_[np.linspace(0, B - 1, n - 2).round().astype(int), 255, 256])
    assert len(idx) == n and {0, 255, 256, 511} <= set(idx.tolist())
    return idx


def _oracle_decoder(c, W, dtype=np.float32):
    import comic_oracle as O
    import gru_oracle as GO
    return GO.GRUDecoder(W, c, dtype) if c.rnn_name == 'GRU' else O.Decoder(W, c, dtype)


@pytest.mark.parametrize('name', sorted(DECODE_CASES))
def test_decode_step_1536_rows_matches_fp64_oracle(torch_mod, name):
    """One wrapper step on 1,536 rows -- the decode's GEMM variants, with the [logits | query] GEMM reading h from the
    loader warps -- against the oracle in float64, per image: new state, logits, alignments and context.  Beam scores
    are sums of log-probabilities and barely move when one GEMM tile is off by 1e-3 relative; the state does."""
    import comic_oracle as O
    from comic_b200 import weights as wts
    from comic_b200.engine import Engine
    c = DECODE_CASES[name][0]()
    W = make_weights(c, include_cnn=False)
    im, fm = fake_features(B, seed=53)
    N, gru = B * BEAM, c.rnn_name == 'GRU'
    dec = _oracle_decoder(c, W, np.float64)
    rng = np.random.default_rng(59)
    c0, h0 = dec.init_state(O.tile_batch(im, BEAM))
    state = dict(c=c0, h=np.tanh(h0 + 0.1 * rng.standard_normal(h0.shape)),              # beams of an image differ
                 attention=0.3 * rng.standard_normal((N, wts.Dims(c).A)), time=0)
    for k in ('c', 'h', 'attention'):
        state[k] = state[k].astype(np.float32).astype(np.float64)                      # the inputs the GPU gets
    toks = rng.integers(0, dec.V, size=N).astype(np.int32)
    ref = dict(h=[], c=[], attention=[], alignments=[], logits=[])
    with _phase('oracle %s, one step on %d rows in float64' % (name, N)):
        for b0 in range(0, B, 128):                                                     # rows are independent
            rows = slice(b0 * BEAM, (b0 + 128) * BEAM)
            dec.setup_memory(O.tile_batch(fm[b0:b0 + 128], BEAM))
            out, ns, al = dec.call(dec.embed(toks[rows]), {k: v if k == 'time' else v[rows] for k, v in state.items()})
            for k, v in (('h', ns['h']), ('c', ns['c']), ('attention', ns['attention']), ('alignments', al),
                         ('logits', dec.output_layer(out))):
                ref[k].append(v)
    eng = Engine(c)
    eng.bind_weights(W, with_cnn=False)
    keys, values = eng.project_fm(eng.to_dev(fm))
    f32 = lambda x: eng.to_dev(x.astype(np.float32))
    r = eng.decode_step(keys, values, B, BEAM, eng.to_dev(toks), None if gru else f32(state['c']), f32(state['h']),
                        f32(state['attention']))
    for k in (('h', 'logits', 'alignments', 'attention') if gru else ('c', 'h', 'logits', 'alignments', 'attention')):
        err = _per_image_err(r[k].cpu().numpy().reshape(B, -1), np.concatenate(ref[k]).reshape(B, -1))
        b = int(np.argmax(err))
        print('%s step, %-10s worst per-image error %.2e (image %d)' % (name, k, err[b], b))
        assert err[b] < 2e-4, '%s: image %d (rows %d-%d) is %.2e from the oracle' % (k, b, 3 * b, 3 * b + 2, err[b])


@pytest.fixture(scope='module', params=sorted(DECODE_CASES))
def decoded(request, torch_mod):
    """One engine-default beam-3 decode of fake_features(512) per case, as host arrays."""
    from comic_b200.engine import Engine, executed_steps
    name = request.param
    make, max_it, head, n_sample = DECODE_CASES[name]
    c = make()
    W = make_weights(c, include_cnn=False)
    im, fm = fake_features(B, seed=43)
    eng = Engine(c)
    eng.bind_weights(W, with_cnn=False)
    with _phase('GPU decode %s, %d images x %d steps' % (name, B, max_it)):
        keys, values = eng.project_fm(eng.to_dev(fm))
        c0, h0 = eng.rnn_init(eng.to_dev(im))
        n0 = eng.launch_count()
        r = eng.decode_beam(keys, values, c0, h0, BEAM, 0.0, max_it)
        T = executed_steps(r['T'])
        launches = eng.launch_count() - n0
        r = {k: v.cpu().numpy() for k, v in r.items()}
    del eng, keys, values, c0, h0
    torch_mod.cuda.empty_cache()
    return dict(name=name, c=c, W=W, im=im, fm=fm, r=r, T=T, launches=launches, max_it=max_it, head=head,
                n_sample=n_sample)


def _audit(ref, got, k, what):
    """ids / parents of `got` (restricted to the oracle's images and T steps) against the oracle, identical except at
    audited near-ties; scores of the other images to 2e-4.  Returns the images that match."""
    n_same, near, bad = margin_audit(ref, got['step_ids'], got['parent_ids'], k)
    n = ref['step_ids'].shape[1]
    assert not bad, '%s: divergence away from a near-tie (image, step, relative gap): %s' % (what, bad[:10])
    keep = np.array(sorted(set(range(n)) - {x[0] for x in near}))
    T = ref['T']
    ref_s = ref['scores'][:, keep].astype(np.float64)
    ratio = np.abs(got['scores'][:T][:, keep] - ref_s) / (2e-4 + 2e-4 * np.abs(ref_s))
    t, j, _ = np.unravel_index(int(np.argmax(ratio)), ratio.shape)
    print('%s: %d / %d images identical over %d steps, %d near-tie divergences %s; worst score error %.2f x tolerance '
          '(step %d, image %d)' % (what, n_same, n, T, len(near), near[:5], ratio.max(), t, keep[j]))
    np.testing.assert_allclose(got['scores'][:T][:, keep], ref['scores'][:, keep], rtol=2e-4, atol=2e-4, err_msg=what)
    assert n_same >= 0.9 * n, what
    return keep


def test_beam_decode_512_images_first_steps(decoded):
    """Every image of the 1,536-row decode over its first steps (steps are causal: the first steps of the long run are
    those of a short oracle run)."""
    import comic_oracle as O
    d = decoded
    assert d['launches'] >= 5 * d['max_it'], 'expected the one-launch-per-op large-batch path (%d launches)' % d['launches']
    assert d['T'] >= d['head']
    with _phase('oracle %s, %d images x %d steps' % (d['name'], B, d['head'])):
        ref = O.beam_search_decode(_oracle_decoder(d['c'], d['W']), d['im'], d['fm'], BEAM, 0.0, d['head'],
                                   return_trace=True)
    assert ref['T'] == d['head']
    _audit(ref, d['r'], BEAM, '%s, all %d images, first %d steps' % (d['name'], B, d['head']))


def test_beam_decode_512_images_all_steps_on_a_sample(decoded):
    """A sample of the images over the whole decode: the oracle run on those images alone (beam search keeps images
    independent) against their rows of the 512-image result -- ids, parents, gathered ids, lengths, scores, maps."""
    import comic_oracle as O
    d = decoded
    idx = _sample(d['n_sample'])
    with _phase('oracle %s, %d images x %d steps' % (d['name'], len(idx), d['max_it'])):
        ref = O.beam_search_decode(_oracle_decoder(d['c'], d['W']), d['im'][idx], d['fm'][idx], BEAM, 0.0, d['max_it'],
                                   return_trace=True)
    T = ref['T']
    assert T <= d['T']                      # the batch runs until its last image finishes
    r = d['r']
    got = {k: r[k][:T][:, idx] for k in ('step_ids', 'parent_ids', 'predicted_ids', 'scores')}
    what = '%s, %d-image sample, %d steps' % (d['name'], len(idx), T)
    keep = _audit(ref, got, BEAM, what)
    np.testing.assert_array_equal(got['predicted_ids'][:, keep], ref['predicted_ids'][:, keep], err_msg=what)
    np.testing.assert_array_equal(r['lengths'][idx][keep], ref['lengths'][keep], err_msg=what)
    _, _, am = O.post_process_beam(ref, d['c'].attn_num_heads, BEAM)
    attn = r['attn'][idx][keep][:, :, :T].astype(np.float64)
    err = _per_image_err(attn, am[keep])
    j = int(np.argmax(err))
    print('%s: worst top-beam attention map error %.2e (image %d)' % (what, err[j], idx[keep][j]))
    assert err[j] < 1e-3, '%s: attention maps of image %d are %.2e from the oracle' % (what, idx[keep][j], err[j])


# ---------------------------------------------------------------------------
# 5. The benchmark's replayed device step, and the pipelined loop, at 512 images
# ---------------------------------------------------------------------------
FIELDS = ('step_ids', 'parent_ids', 'predicted_ids', 'lengths', 'scores', 'attn')


def test_graph_replay_of_the_bench_step_is_bit_identical(enc512, torch_mod):
    """bench.py's step_device: encode -> project -> init -> 60-step decode through Engine.graphed, called three times on
    one device batch (eager, capture + replay, replay); every output of the replays equals the eager call's."""
    from comic_b200.engine import executed_steps
    eng, c, dev = enc512['eng'], enc512['c'], enc512['dev']
    T = c.infer_max_length * 2

    def step_eager(x):
        emb, fm = eng.encode(x)
        keys, values = eng.project_fm(fm)
        c0, h0 = eng.rnn_init(emb)
        return eng.decode_beam(keys, values, c0, h0, BEAM, c.infer_length_penalty_weight, T)

    with _phase('GPU bench step x 3 through Engine.graphed, %d images' % B):
        outs = []
        for i in range(3):
            r = eng.graphed('bench_step_test', step_eager, dev)
            n = executed_steps(r['T'])
            outs.append((n, {k: (r[k] if k in ('lengths', 'attn') else r[k][:n]).clone() for k in FIELDS}))
            if i == 1:
                replayed = eng.replayed_launches
    assert eng._graphs['bench_step_test']['graph'] is not None
    assert eng.replayed_launches > replayed > 0
    (n0, eager), rest = outs[0], outs[1:]
    print('bench step: %d steps, %d launches per replay' % (n0, eng._graphs['bench_step_test']['launches']))
    for i, (n, o) in enumerate(rest, 2):
        assert n == n0, 'call %d' % i
        for k in FIELDS:
            a, b = (o[k], eager[k]) if k != 'attn' else (o[k][:, :, :n0], eager[k][:, :, :n0])
            assert torch_mod.equal(a, b), 'call %d: %s differs from the eager call' % (i, k)


def test_run_stream_512_image_batches_matches_run(enc512):
    """CaptionModel.run_stream over six uint8 batches of 512 images (each of its two input slots runs eager, captures,
    replays) returns, batch by batch, what CaptionModel.run returns."""
    from comic_b200.model import CaptionModel
    c, W = enc512['c'], enc512['W']
    m = CaptionModel(c, 'infer', batch_ops=None, weights=W)
    rng = np.random.default_rng(47)
    u8 = [rng.integers(0, 256, (B, 240, 320, 3), dtype=np.uint8) for _ in range(6)]
    with _phase('CaptionModel.run, 6 x %d images' % B):
        refs = [tuple(a.copy() for a in m.run(x)) for x in u8]
    with _phase('CaptionModel.run_stream, 6 x %d images' % B):
        n = 0
        for i, (p, a) in enumerate(m.run_stream(iter(u8))):
            np.testing.assert_array_equal(p, refs[i][0], err_msg='batch %d ids' % i)
            np.testing.assert_array_equal(a, refs[i][1], err_msg='batch %d attention maps' % i)
            n += 1
    assert n == 6 and refs[0][0].shape[0] == B
    g = [e for k, e in m.engine._graphs.items() if k[0] == 'run_stream']
    assert len(g) == 2 and all(e['graph'] is not None for e in g) and m.engine.replayed_launches > 0

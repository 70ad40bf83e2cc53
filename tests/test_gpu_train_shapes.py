"""The training backward at the batch shapes the training benchmark runs (scripts/bench_train.py): 32 rows x 41 steps for
decoder / cnn_finetune, 10 images x 3 hypotheses for scst, against fp64 autograd of tests/torch_ref.py.

csrc/train.cu picks its work splits from the batch size, so the 4-row cases of test_gpu_train.py never reach them:
  - the attention backward runs one CTA per (image, position slice), S = clamp(2 x SMs / B, 1, 28) slices.  Below 11 rows
    S = 28 cuts the 196 positions evenly (7 each); at 32 rows (148 SMs) S = 9 and attn_bwd_dalpha(_vec)_kernel cuts them
    by ceiling division (8 x 22 + 20) while attn_bwd_ln_kernel / attn_bwd_dot_kernel use floor division (21 / 22);
  - the weight-gradient GEMMs (K = (T_run + 1) x B rows) split K from 128 rows on, and the per-step skinny GEMMs change
    tile configuration at 33 rows;
  - the teacher-forced forward takes attn_fused_kernel from 48 images on and, in 'split' precision, the tensor path for
    its gate / [logits | query] GEMMs from 64 rows on;
  - the InceptionV1 backward takes the tcgen05 dgrad and a pixel-split wgrad on the 7 x 7 layers from 3 images on.
Each decoder case names the slice count S it reaches; its row count is derived from the device's SM count so that it
does.  Tolerances are relative to each tensor's largest entry: 'f32' 1e-4 (torch's own fp32 autograd is 6.6e-7 from
fp64 at 32 x 41), 'split' 1e-3 (bf16x3 GEMMs)."""
import gc

import numpy as np
import pytest

from _common import comic_config, word_config, make_weights, images, fake_features, rel_err

pytestmark = pytest.mark.gpu

M_POS = 196


@pytest.fixture(scope='module')
def torch_mod():
    import torch
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    return torch


@pytest.fixture(scope='module')
def sms(torch_mod):
    return torch_mod.cuda.get_device_properties(0).multi_processor_count


def _slices(B, sms):
    """attn_slices() of csrc/train.cu."""
    return min(max((2 * sms) // B, 1), 28)


def _rows_for_slices(S, sms):
    """A row count whose attention backward runs S position slices: just above the SM count for S = 1, the largest
    row count with 2 x SMs / B >= S otherwise (32 rows for S = 9 on 148 SMs, the benchmark's batch)."""
    return sms + 2 if S == 1 else (2 * sms) // S


def _captions(c, B, L, lengths, rng):
    """[B, L] int32 captions: <GO>, tokens, <EOS>, padding -1.  lengths 'full': every row executes L - 1 steps (the
    benchmark's batches); 'ragged': the row lengths spread evenly over 1 .. L - 1 in random row order."""
    V = 258 if c.token_type == 'radix' else len(c.itow)
    go, eos = (256, 257) if c.token_type == 'radix' else (c.wtoi['<GO>'], c.wtoi['<EOS>'])
    T = L - 1
    if lengths == 'full':
        lens = np.full(B, T)
    else:
        lens = rng.permutation(1 + (np.arange(B) * (T - 1)) // max(B - 1, 1))
    caps = np.full((B, L), -1, np.int32)
    for b in range(B):
        n = int(lens[b]) - 1                            # tokens before <EOS>
        caps[b, 0] = go
        caps[b, 1:1 + n] = rng.integers(0, V - 2, size=n)
        caps[b, 1 + n] = eos
    return caps


def _reference(c, W, im, fm, caps, masks, keeps, rewards):
    """fp64 autograd of the torch restatement; the graph is freed before returning (~9 GB at 32 x 41)."""
    import torch_ref as TR
    P = TR.to_params(W)
    tot, xe, mp, reg, aux = TR.training_loss(P, c, im, fm, caps, masks, keeps, rewards, fm_requires_grad=True)
    tot.backward()
    ref = dict(loss=np.array([float(v.detach()) for v in (tot, xe, mp, reg)]),
               logits=aux['logits'].detach().numpy(), attn=aux['attn'].detach().numpy(),
               grads={k: v.grad.numpy() for k, v in P.items()},
               dfm=aux['fm'].grad.numpy(), dim=aux['im'].grad.numpy())
    del P, tot, xe, mp, reg, aux
    gc.collect()
    return ref


TRAIN_CFG = {
    'decoder': lambda: comic_config(train_mode='decoder'),
    'scst': lambda: comic_config(train_mode='scst'),
    'dot': lambda: comic_config(train_mode='decoder', attn_alignment_method='dot'),
    'sigmoid': lambda: comic_config(train_mode='decoder', attn_probability_fn='sigmoid'),
    'context_layer': lambda: comic_config(train_mode='decoder', attn_context_layer=True),
    'independent_h4': lambda: comic_config(train_mode='decoder', cnn_fm_projection='independent', attn_num_heads=4),
    'project_hidden': lambda: comic_config(train_mode='decoder', rnn_init_method='project_hidden'),
    'word_none_h1': lambda: word_config(n_words=300, train_mode='decoder'),
    'rnn_size_256': lambda: comic_config(train_mode='decoder', rnn_size=256),
    'rnn_size_1024': lambda: comic_config(train_mode='decoder', rnn_size=1024),
}

# id -> (config, slice count S or fixed row count, steps, lengths, hypotheses per image (scst), precisions)
DECODER_CASES = {
    'bench_S9_32x41': ('decoder', dict(S=9), 41, 'full', 1, ('f32', 'split')),
    'ragged_S9_32x41': ('decoder', dict(S=9), 41, 'ragged', 1, ('f32',)),
    'scst_S9_10x3x41': ('scst', dict(S=9), 41, 'ragged', 3, ('f32',)),
    'S1_150x4': ('decoder', dict(S=1), 4, 'ragged', 1, ('f32', 'split')),
    'S3_98x6': ('decoder', dict(S=3), 6, 'ragged', 1, ('f32',)),
    'S22_13x8': ('decoder', dict(S=22), 8, 'ragged', 1, ('f32',)),
    'rows48_S6_6': ('decoder', dict(rows=48), 6, 'ragged', 1, ('split',)),
    'rows64_S4_6': ('decoder', dict(rows=64), 6, 'ragged', 1, ('split',)),
    'dot_S9_32x21': ('dot', dict(S=9), 21, 'ragged', 1, ('f32',)),
    'sigmoid_S9_32x21': ('sigmoid', dict(S=9), 21, 'ragged', 1, ('f32',)),
    'context_layer_S9_32x21': ('context_layer', dict(S=9), 21, 'ragged', 1, ('f32',)),
    'independent_h4_S9_32x21': ('independent_h4', dict(S=9), 21, 'ragged', 1, ('f32',)),
    'project_hidden_S9_32x21': ('project_hidden', dict(S=9), 21, 'ragged', 1, ('f32',)),
    'word_none_h1_S9_32x21': ('word_none_h1', dict(S=9), 21, 'ragged', 1, ('f32',)),
    'rnn_size_256_S9_32x21': ('rnn_size_256', dict(S=9), 21, 'ragged', 1, ('f32',)),
    'rnn_size_1024_S9_32x21': ('rnn_size_1024', dict(S=9), 21, 'ragged', 1, ('f32',)),
}

TOL = {'f32': dict(loss=1e-5, fwd=2e-4, grad=1e-4), 'split': dict(loss=1e-4, fwd=2e-4, grad=1e-3)}


def _case_inputs(c, B, T, lengths, tile, seed):
    rng = np.random.default_rng(seed)
    W = make_weights(c, include_cnn=False)
    im, fm = fake_features(B // tile, seed=seed + 1)
    if tile > 1:                                        # scst_step repeats each image's encoder outputs per hypothesis
        im, fm = np.tile(im, (tile, 1)), np.tile(fm, (tile, 1, 1))
    caps = _captions(c, B, T + 1, lengths, rng)
    rewards = None
    if c.train_mode == 'scst':
        rewards = rng.standard_normal(B).astype(np.float32)
        rewards[::5] = 0.0                               # sampled = greedy caption: zero advantage
    return W, im, fm, caps, rewards


@pytest.mark.parametrize('case', list(DECODER_CASES))
def test_training_backward_matches_fp64_autograd(torch_mod, sms, case):
    """Losses, logits, attention maps, every decoder gradient and d loss / d (fm, im_embed) -- resolved per image and
    position, so a position that an attention-backward slice drops or counts twice shows there directly."""
    from comic_b200.train import Trainer
    from comic_b200 import weights as wts
    cfg, shape, T, lengths, tile, precisions = DECODER_CASES[case]
    c = TRAIN_CFG[cfg]()
    if 'S' in shape:
        S = shape['S']
        B = _rows_for_slices(S, sms) // tile * tile
        assert _slices(B, sms) == S, (B, sms)
    else:
        B = shape['rows']
    W, im, fm, caps, rewards = _case_inputs(c, B, T, lengths, tile, seed=B + T)
    tr = Trainer(c, W, with_cnn=False)
    eng = tr.engine
    masks, keeps = tr.make_masks(B, T, seed=1000 + B)  # on the device, as Trainer.step draws them
    hmasks = {k: v.cpu().numpy() for k, v in masks.items()}
    if 'att' in hmasks:
        hmasks['att'] = hmasks['att'].reshape(T, B, c.attn_num_heads, M_POS)
    ref = _reference(c, W, im, fm, caps, hmasks, keeps, rewards)
    fm_d, im_d = eng.to_dev(fm), eng.to_dev(im)
    failures = []
    for prec in precisions:
        tol = TOL[prec]
        eng.set_precision(prec)
        out = tr.forward_backward(fm_d, im_d, caps, rewards, masks, keeps, want_logits=True, want_attn=True)
        assert out['T_run'] == T
        err = {}
        loss = out['loss'].cpu().numpy().astype(np.float64)
        for i, name in enumerate(('total', 'xe', 'map', 'reg')):
            err['loss/' + name] = (abs(loss[i] - ref['loss'][i]) / max(abs(ref['loss'][i]), 1e-30), tol['loss'])
        err['logits'] = (rel_err(out['logits'].cpu().numpy().transpose(1, 0, 2), ref['logits']), tol['fwd'])
        err['attn'] = (rel_err(out['attn'].cpu().numpy(), ref['attn']), tol['fwd'])
        for vname in wts.decoder_shapes(c):
            g = tr.gradient(vname).cpu().numpy().reshape(ref['grads'][vname].shape)
            err[vname] = (rel_err(g, ref['grads'][vname]), tol['grad'])
        dfm, dim = eng.train_encoder_grads(B, T)
        err['d fm'] = (rel_err(dfm.cpu().numpy(), ref['dfm']), tol['grad'])
        err['d im_embed'] = (rel_err(dim.cpu().numpy(), ref['dim']), tol['grad'])
        grads = {k: v for k, v in err.items() if not k.startswith(('loss/', 'logits', 'attn'))}
        worst = max(grads, key=lambda k: grads[k][0])
        print('\n%s [%s] B=%d S=%d T=%d: worst gradient %s %.2e, d fm %.2e, logits %.2e, attn %.2e, xe %.2e'
              % (case, prec, B, _slices(B, sms), T, worst, grads[worst][0], err['d fm'][0], err['logits'][0],
                 err['attn'][0], err['loss/xe'][0]))
        failures += [(prec, k, e, t) for k, (e, t) in err.items() if not e < t]
    assert not failures, failures


def test_cuda_graph_replay_at_the_bench_shape_is_bit_identical(torch_mod, sms):
    """32 x 41 full-length rows, 'split' precision, dropout: two eager calls agree bit for bit, and the CUDA-graph
    replays (third call on) reproduce them -- the fixed-order reductions hold at the split-K / S = 9 plans too."""
    from comic_b200.train import Trainer
    c = TRAIN_CFG['decoder']()
    B, T = 32, 41
    W, im, fm, caps, _ = _case_inputs(c, B, T, 'full', 1, seed=5)
    runs = {}
    for graphed in (False, True):
        tr = Trainer(c, W, with_cnn=False)
        tr.cuda_graph = graphed
        eng = tr.engine
        eng.set_precision('split')
        fm_d, im_d = eng.to_dev(fm), eng.to_dev(im)
        masks, keeps = tr.make_masks(B, T, seed=77)
        got = []
        for _ in range(4 if graphed else 2):
            out = tr.forward_backward(fm_d, im_d, caps, None, masks, keeps)
            got.append((out['loss'].clone(), tr.grads.clone()))
        if graphed:
            assert tr.replayed_launches > 0
        runs[graphed] = got
    (l0, g0), (l1, g1) = runs[False]
    assert torch_mod.equal(l0, l1) and torch_mod.equal(g0, g1), 'two eager calls differ'
    for i, (l, g) in enumerate(runs[True]):
        assert torch_mod.equal(l, l0) and torch_mod.equal(g, g0), 'graphed call %d differs from eager' % i


# ---------------------------------------------------------------------------------------------------------------------
# cnn_finetune at 32 images.  fp64 autograd cannot check the CNN gradients at this size: ReLU / max-pool mask flips put
# torch's own fp32 autograd 6.5e-3 away from fp64 there.  The backward is linear in the cotangents and sums over images,
# and the f32 forward tape is batch-invariant bit for bit, so the 32-image backward must equal the sum of sixteen
# 2-image backwards -- the configuration test_gpu_train_cnn.py pins to fp64 -- on the same images and cotangents.
# ---------------------------------------------------------------------------------------------------------------------
# about 10x what a B200 (148 SMs, 1,000 W limit) measured: f32 9.5e-7 (summation order only), split 4.6e-5 (bf16x3 dgrad);
# one pixel of the last image left out of the 7 x 7 layers' wgrad moves them by 7.5e-3
N_IMG, PAIR = 32, 2
CNN_TOL = {'f32': 1e-5, 'split': 5e-4}


@pytest.fixture(scope='module')
def cnn_pairs(torch_mod):
    """Trainer, inputs, and the 2-image tapes and fp64-accumulated gradient sums (f32 precision)."""
    from comic_b200.train import Trainer
    torch = torch_mod
    c = comic_config(train_mode='cnn_finetune')
    tr = Trainer(c, make_weights(c, seed=11))
    eng = tr.engine
    eng.set_precision('f32')
    rng = np.random.default_rng(9)
    img = eng.to_dev(images(N_IMG, seed=5))
    Gf = eng.to_dev(rng.standard_normal((N_IMG, M_POS, 832)).astype(np.float32))
    Ge = eng.to_dev(rng.standard_normal((N_IMG, 1024)).astype(np.float32))
    lo = tr.n_decoder_flat
    total = torch.zeros(tr.n_flat - lo, dtype=torch.float64, device=eng.device)
    embs, fms = [], []
    for i in range(0, N_IMG, PAIR):
        sl = slice(i, i + PAIR)
        emb, fm = eng.encode_train(img[sl])
        embs.append(emb.clone())
        fms.append(fm.clone())
        tr.grads.zero_()
        eng.encode_bwd(img[sl], Gf[sl], Ge[sl], tr.cnn_grad_w, tr.cnn_grad_b)
        total += tr.grads[lo:].double()
    return dict(tr=tr, img=img, Gf=Gf, Ge=Ge, emb=torch.cat(embs), fm=torch.cat(fms), total=total)


@pytest.mark.parametrize('precision', ['f32', 'split'])
def test_cnn_backward_at_32_images_is_the_sum_of_2_image_backwards(torch_mod, cnn_pairs, precision):
    """'split' runs the backward GEMMs on the tcgen05 bf16x3 path over the f32 tape (the 7 x 7 layers' dgrad takes it at
    32 images, not at 2), compared with the f32 sum."""
    from comic_b200 import weights as wts
    k = cnn_pairs
    tr, eng = k['tr'], k['tr'].engine
    eng.set_precision('f32')
    emb, fm = eng.encode_train(k['img'])
    assert torch_mod.equal(fm, k['fm']) and torch_mod.equal(emb, k['emb']), \
        'the 32-image tape differs from the 2-image tapes (ReLU / pool masks may differ)'
    eng.set_precision(precision)
    tr.grads.zero_()
    eng.encode_bwd(k['img'], k['Gf'], k['Ge'], tr.cnn_grad_w, tr.cnn_grad_b)
    lo = tr.n_decoder_flat
    got = tr.grads[lo:].double().cpu().numpy()
    want = k['total'].cpu().numpy()
    worst = {}
    for sc, *_ in wts.cnn_conv_list():
        for name in (wts.CNN + sc + '/weights', wts.CNN + sc + '/BatchNorm/beta'):
            o, n, _ = tr.offsets[name]
            worst[name] = rel_err(got[o - lo:o - lo + n], want[o - lo:o - lo + n])
    name = max(worst, key=worst.get)
    print('\ncnn_finetune 32 images [%s] vs sum of 2-image backwards: worst %s %.2e' % (precision, name, worst[name]))
    bad = {n: v for n, v in worst.items() if not v < CNN_TOL[precision]}
    assert not bad, bad


# ---------------------------------------------------------------------------------------------------------------------
# Inference at rnn_size 256 / 1024: the persistent decode loop and the streaming attention kernel are R = 512 only, so
# these sizes run the per-step kernels, and from 48 images on attn_fused_kernel<256 | 1024>.
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('B', [4, 50])
@pytest.mark.parametrize('R', [256, 1024])
def test_beam_search_at_rnn_size_matches_oracle(torch_mod, R, B):
    import comic_oracle as O
    from comic_b200.engine import Engine
    c = comic_config(rnn_size=R)
    W = make_weights(c, include_cnn=False)
    im, fm = fake_features(B, seed=R + B)
    k, max_it = 3, 8
    ref = O.beam_search_decode(O.Decoder(W, c), im, fm, k, 0.0, max_it)
    eng = Engine(c)
    eng.bind_weights(W, with_cnn=False)
    eng.set_precision('f32')
    keys, values = eng.project_fm(eng.to_dev(fm))
    c0, h0 = eng.rnn_init(eng.to_dev(im))
    r = eng.decode_beam(keys, values, c0, h0, k, 0.0, max_it)
    T = int(r['T'].item())
    assert T == ref['T']
    np.testing.assert_array_equal(r['step_ids'][:T].cpu().numpy(), ref['step_ids'])
    np.testing.assert_array_equal(r['parent_ids'][:T].cpu().numpy(), ref['parent_ids'])
    np.testing.assert_array_equal(r['predicted_ids'][:T].cpu().numpy(), ref['predicted_ids'])
    np.testing.assert_array_equal(r['lengths'].cpu().numpy(), ref['lengths'])
    np.testing.assert_allclose(r['scores'][:T].cpu().numpy(), ref['scores'], rtol=1e-4, atol=1e-4)
    _, _, am = O.post_process_beam(ref, c.attn_num_heads, k)
    err = rel_err(r['attn'][:, :, :T].cpu().numpy(), am)
    print('\nbeam search rnn_size %d, %d images: attention maps %.2e' % (R, B, err))
    assert err < 2e-4

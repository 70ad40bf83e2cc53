"""Training at attention end points other than Mixed_4f on the B200: decoder-mode / scst losses and every decoder
gradient (and d loss / d (fm, im_embed)) against fp64 autograd at 14 x 14 and 7 x 7 maps for tied, independent and
unprojected values; the cnn_finetune InceptionV1 backward with the feature-map gradient entering at the end point;
end-to-end scst, --legacy and cnn_finetune steps; CUDA-graph replay; a falling loss.  Tolerances as
tests/test_gpu_train.py (decoder 1e-3) and tests/test_gpu_train_cnn.py (CNN 5e-3, see its docstring)."""
import numpy as np
import pytest

from _common import comic_config, word_config, make_weights, images, rel_err
import fm_endpoint_ref as FR

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def torch_mod():
    import torch
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    return torch


CASES = {
    'Mixed_4c_tied_dropout': (lambda: comic_config(train_mode='decoder', cnn_fm_attention='Mixed_4c'), True, False),
    'Mixed_4e_none': (lambda: comic_config(train_mode='decoder', cnn_fm_attention='Mixed_4e', cnn_fm_projection='none'),
                      True, False),
    'MaxPool_4a_independent_h4': (lambda: comic_config(train_mode='decoder', cnn_fm_attention='MaxPool_4a_3x3',
                                                       cnn_fm_projection='independent', attn_num_heads=4), True, False),
    'Mixed_5b_tied_dropout': (lambda: comic_config(train_mode='decoder', cnn_fm_attention='Mixed_5b'), True, False),
    'Mixed_5c_none': (lambda: comic_config(train_mode='decoder', cnn_fm_attention='Mixed_5c', cnn_fm_projection='none'),
                      True, False),
    'MaxPool_5a_independent_scst': (lambda: comic_config(train_mode='scst', cnn_fm_attention='MaxPool_5a_2x2',
                                                         cnn_fm_projection='independent'), True, True),
    'word_Mixed_5b_ctx': (lambda: word_config(n_words=300, train_mode='decoder', cnn_fm_attention='Mixed_5b',
                                              attn_context_layer=True), True, False),
}


def _dev_masks(eng, masks):
    if masks is None:
        return None
    return dict(init_in=eng.to_dev(masks['init_in']), inp=eng.to_dev(masks['inp']), out=eng.to_dev(masks['out']),
                att=eng.to_dev(masks['att'].reshape(masks['att'].shape[0], masks['att'].shape[1], -1)))


@pytest.mark.parametrize('name,B', [(n, 3) for n in CASES] + [('Mixed_4c_tied_dropout', 48), ('Mixed_5c_none', 48)])
def test_gradients_match_autograd(torch_mod, name, B):
    """B = 3: sliced attention kernels, B * 49 odd; B = 48: the fused attention kernel and the tensor-path GEMMs."""
    import torch_ref as TR
    from comic_b200.train import Trainer
    from comic_b200 import weights as wts
    mk, dropout, scst = CASES[name]
    c = mk()
    W, im, fm, caps, masks, keeps = FR.train_case(c, B=B, L=8, seed=3, dropout=dropout)
    rewards = np.random.default_rng(1).uniform(-1, 1, B).astype(np.float32) if scst else None
    P = TR.to_params(W)
    tot, xe, mp, reg, aux = TR.training_loss(P, c, im, fm, caps, masks, keeps, rewards, fm_requires_grad=True)
    tot.backward()
    tr = Trainer(c, W, with_cnn=False)
    eng = tr.engine
    eng.set_precision('f32')
    out = tr.forward_backward(eng.to_dev(fm), eng.to_dev(im), caps, rewards, _dev_masks(eng, masks), keeps,
                              want_logits=True, want_attn=True)
    loss = out['loss'].cpu().numpy()
    assert abs(loss[1] - float(xe)) < 1e-4 * max(1.0, abs(float(xe)))
    assert abs(loss[0] - float(tot)) < 1e-4 * max(1.0, abs(float(tot)))
    assert rel_err(out['attn'].cpu().numpy(), aux['attn'].detach().numpy()) < 2e-4
    worst = {}
    for vname in wts.decoder_shapes(c):
        g = tr.gradient(vname).cpu().numpy().reshape(P[vname].shape)
        worst[vname] = rel_err(g, P[vname].grad.numpy())
    bad = {k: v for k, v in worst.items() if not v < 1e-3}
    assert not bad, (bad, worst)
    dfm, demb = eng.train_encoder_grads(B, out['T_run'])
    assert rel_err(dfm.cpu().numpy(), aux['fm'].grad.numpy()) < 1e-3
    assert rel_err(demb.cpu().numpy(), aux['im'].grad.numpy()) < 1e-3


def _cnn_grad_names():
    from comic_b200 import weights as wts
    out = []
    for sc, *_ in wts.cnn_conv_list():
        out += [wts.CNN + sc + '/weights', wts.CNN + sc + '/BatchNorm/beta']
    return out


def _layer_above(name, endpoint):
    """Whether the variable `name` belongs to a layer after `endpoint` in the network (it never sees d loss / d fm)."""
    from comic_b200 import weights as wts
    order = [b[0] for b in wts.BLOCKS]
    scope = name[len(wts.CNN):].split('/')[0]
    return scope in order and order.index(scope) > order.index(endpoint)


@pytest.mark.parametrize('endpoint', ['Mixed_4c', 'MaxPool_4a_3x3', 'Mixed_5b', 'Mixed_5c'])
def test_cnn_backward_takes_dfm_at_the_end_point(torch_mod, endpoint):
    """loss = <fm, Gf> + <im_embed, Ge> with fixed random cotangents, against fp64 autograd of the torch restatement.

    Where dfm enters is checked exactly: with Ge = 0 every conv-kernel / BN-beta gradient of a layer after the end point
    is zero and every other one is not.  The values are held to what fp32 arithmetic allows on the case: torch's OWN fp32
    autograd of the same lines differs from its fp64 autograd by up to 2.5e-2 at these end points on 2-image cases (ReLU /
    max-pool masks flipped by rounding; measured over six weight / image seeds), so the 95th percentile of the 114
    per-tensor errors must stay within max(5e-3, 2x torch fp32's) and the worst below 3e-2, while a misplaced or missing
    dfm moves every tensor below the end point by O(1)."""
    import torch_ref as TR
    from comic_b200.train import Trainer
    from comic_b200 import weights as wts
    torch = torch_mod
    c = comic_config(train_mode='cnn_finetune', cnn_fm_attention=endpoint)
    d = wts.Dims(c)
    W = make_weights(c, seed=11)
    img = images(2, seed=5)
    rng = np.random.default_rng(9)
    Gf = rng.standard_normal((2, d.M, d.C)).astype(np.float32)
    Ge = rng.standard_normal((2, 1024)).astype(np.float32)
    grads, outs = {}, {}
    for dt in (torch.float64, torch.float32):
        P = TR.cnn_params(W, dtype=dt)
        emb, fm = FR.encoder_forward(P, img, endpoint)
        ((fm * torch.as_tensor(Gf, dtype=dt)).sum() + (emb * torch.as_tensor(Ge, dtype=dt)).sum()).backward()
        grads[dt] = {n: P[n].grad.double().numpy() for n in _cnn_grad_names()}
        outs[dt] = (emb.detach().numpy(), fm.detach().numpy())
    emb, fm = outs[torch.float64]
    ref = grads[torch.float64]
    floor = np.quantile([rel_err(grads[torch.float32][n], ref[n]) for n in ref], 0.95)
    tr = Trainer(c, W)
    eng = tr.engine
    eng.set_precision('f32')
    d_img = eng.to_dev(img)
    emb_d, fm_d = eng.encode_train(d_img)
    assert rel_err(fm_d.cpu().numpy(), fm) < 2e-4
    assert rel_err(emb_d.cpu().numpy(), emb) < 2e-4
    tr.grads.zero_()
    eng.encode_bwd(d_img, eng.to_dev(Gf), eng.to_dev(Ge), tr.cnn_grad_w, tr.cnn_grad_b)
    worst = {n: rel_err(tr.gradient(n).cpu().numpy(), ref[n]) for n in ref}
    errs = np.array(sorted(worst.values()))
    assert errs[-1] < 3e-2 and np.quantile(errs, 0.95) < max(5e-3, 2 * floor), \
        (floor, sorted(worst.items(), key=lambda kv: -kv[1])[:8])
    g1 = tr.grads.clone()
    tr.grads.zero_()
    eng.encode_bwd(d_img, eng.to_dev(Gf), eng.to_dev(Ge), tr.cnn_grad_w, tr.cnn_grad_b)
    assert torch.equal(g1, tr.grads)                        # fixed-order reductions: bit-reproducible
    tr.grads.zero_()
    eng.encode_bwd(d_img, eng.to_dev(Gf), eng.to_dev(np.zeros_like(Ge)), tr.cnn_grad_w, tr.cnn_grad_b)
    for n in _cnn_grad_names():
        nz = bool(tr.gradient(n).abs().max() > 0)
        assert nz != _layer_above(n, endpoint), n


def test_cnn_finetune_steps_at_a_7x7_end_point(torch_mod):
    from comic_b200.train import Trainer
    c = comic_config(train_mode='cnn_finetune', cnn_fm_attention='Mixed_5c', max_step=100)
    W = make_weights(c, seed=5)
    _, _, _, caps, _, _ = FR.train_case(c, B=2, L=7, seed=4, dropout=False)
    tr = Trainer(c, W)
    img = tr.engine.to_dev(images(2, seed=3))
    before = tr.params.clone()
    losses = [float(tr.step(img, caps, lr=1e-3)['loss'][1]) for _ in range(3)]
    assert all(np.isfinite(losses)) and losses[-1] < losses[0], losses
    assert not torch_mod.equal(before, tr.params)


def test_scst_step_at_a_7x7_end_point(torch_mod):
    from comic_b200 import scst as S
    from comic_b200.train import Trainer
    c = comic_config(train_mode='scst', scst_beam_size=3, n_words=1000, max_step=50, cnn_fm_attention='Mixed_5b')
    W = make_weights(c)
    B = 2
    rng = np.random.default_rng(0)
    refs = [[' '.join('w%d' % w for w in rng.integers(0, 997, size=10)) for _ in range(5)] for _ in range(B)]
    df = {'document_frequency': S.compute_doc_freq(refs), 'ref_len': B}
    scorer = S.CaptionScorer(df, dict(ciderD=c.scst_weight_ciderD, bleu=c.scst_weight_bleu))
    tr = Trainer(c, W)
    before = tr.params.clone()
    out = S.scst_step(tr, scorer, tr.engine.to_dev(images(B, seed=12)), refs, seed=3, lr=1e-3)
    assert np.isfinite(out['rewards']).all()
    assert np.isfinite(out['loss'].cpu().numpy()).all()
    assert tr.global_step == 1 and not torch_mod.equal(before, tr.params)


def test_legacy_decoder_step_at_mixed_5b(torch_mod):
    from comic_b200.train import Trainer
    from comic_b200 import weights as wts
    c = comic_config(train_mode='decoder', legacy=True, max_step=100, cnn_fm_attention='Mixed_5b')
    W = make_weights(c, seed=5)
    _, _, _, caps, _, _ = FR.train_case(c, B=2, L=7, seed=4, dropout=False)
    tr = Trainer(c, W)
    img = tr.engine.to_dev(images(2, seed=3))
    w0 = tr.variable(wts.ENC + 'im_embed/weight').clone()
    losses = [float(tr.step(img, caps, lr=1e-2)['loss'][1]) for _ in range(3)]
    assert all(np.isfinite(losses)) and losses[-1] < losses[0], losses
    assert float((tr.variable(wts.ENC + 'im_embed/weight') - w0).abs().max()) > 0


@pytest.mark.parametrize('endpoint', ['Mixed_4e', 'Mixed_5b'])
def test_cuda_graph_replay_is_bit_identical_and_loss_falls(torch_mod, endpoint):
    from comic_b200.train import Trainer
    c = comic_config(train_mode='decoder', max_step=100, cnn_fm_attention=endpoint)
    W, im, fm, caps, _, _ = FR.train_case(c, B=5, L=8, seed=7, dropout=False)
    runs = {}
    for graphed in (False, True):
        tr = Trainer(c, W, with_cnn=False)
        tr.cuda_graph = graphed
        eng = tr.engine
        got = []
        for i in range(5):
            fm_d, im_d = eng.to_dev(fm * (1.0 + 0.1 * i)), eng.to_dev(im * (1.0 + 0.1 * i))
            masks, keeps = tr.make_masks(5, int((caps[:, 1:] >= 0).sum(1).max()), 100 + i)
            out = tr.forward_backward(fm_d, im_d, caps, None, masks, keeps)
            got.append((out['loss'].clone(), tr.grads.clone()))
        if graphed:
            assert any(e['graph'] is not None for e in tr._graphs.values())
        runs[graphed] = got
    for (l0, g0), (l1, g1) in zip(runs[False], runs[True]):
        assert torch_mod.equal(l0, l1) and torch_mod.equal(g0, g1)
    tr = Trainer(c, W, with_cnn=False)
    fm_d, im_d = tr.engine.to_dev(fm), tr.engine.to_dev(im)
    losses = []
    for _ in range(6):
        losses.append(float(tr.forward_backward(fm_d, im_d, caps)['loss'][1].item()))
        tr.apply_gradients(lr=5e-3)
    assert all(np.isfinite(losses)) and losses[-1] < losses[0] - 0.05, losses

"""GPU parity of GRU training (csrc/train.cu, rnn_name=GRU): losses and every decoder-variable gradient against fp64
autograd of the torch restatement with the GRU cell (tests/gru_oracle.training_loss, pinned to the NumPy oracle's forward
in tests/test_gru_host.py), with the tolerances of tests/test_gpu_train.py."""
import numpy as np
import pytest

from _common import comic_config, word_config, rel_err
from test_oracle_known_answers import _train_case
import gru_oracle as GO

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def torch_mod():
    import torch
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    return torch


CASES = {
    'xe_dropout': (lambda: comic_config(rnn_name='GRU', train_mode='decoder'), True, False),
    'scst_dropout': (lambda: comic_config(rnn_name='GRU', train_mode='scst'), True, True),
    'xe_nodrop': (lambda: comic_config(rnn_name='GRU', train_mode='decoder'), False, False),
    'project_hidden': (lambda: comic_config(rnn_name='GRU', train_mode='decoder', rnn_init_method='project_hidden'), True, False),
    'dot_sigmoid_ctx_indep_h4': (lambda: comic_config(rnn_name='GRU', train_mode='scst', attn_alignment_method='dot',
                                                      attn_probability_fn='sigmoid', attn_context_layer=True,
                                                      cnn_fm_projection='independent', attn_num_heads=4), True, True),
    'word_none_h1': (lambda: word_config(n_words=300, rnn_name='GRU', train_mode='decoder'), True, False),
}
REWARDS = np.array([0.4, -0.3, 1.2, 0.05], np.float32)


def _dev_masks(eng, masks):
    if masks is None:
        return None
    return dict(init_in=eng.to_dev(masks['init_in']), inp=eng.to_dev(masks['inp']), out=eng.to_dev(masks['out']),
                att=eng.to_dev(masks['att'].reshape(masks['att'].shape[0], masks['att'].shape[1], -1)))


@pytest.mark.parametrize('name', list(CASES))
def test_gru_gradients_match_autograd(torch_mod, name):
    import torch_ref as TR
    from comic_b200.train import Trainer
    from comic_b200 import weights as wts
    mk, dropout, scst = CASES[name]
    c = mk()
    W, im, fm, caps, masks, keeps = _train_case(c, B=4, L=8, seed=3, dropout=dropout)
    rewards = REWARDS if scst else None
    P = TR.to_params(W)
    tot, xe, mp, reg, aux = GO.training_loss(P, c, im, fm, caps, masks, keeps, rewards)
    tot.backward()
    tot, xe, mp = (float(v.detach()) for v in (tot, xe, mp))
    tr = Trainer(c, W, with_cnn=False)
    eng = tr.engine
    eng.set_precision('f32')
    out = tr.forward_backward(eng.to_dev(fm), eng.to_dev(im), caps, rewards, _dev_masks(eng, masks), keeps, want_logits=True,
                              want_attn=True)
    loss = out['loss'].cpu().numpy()
    assert abs(loss[1] - xe) < 1e-4 * max(1.0, abs(xe))
    assert abs(loss[2] - mp) < 1e-4 * max(1e-3, abs(mp))
    assert abs(loss[0] - tot) < 1e-4 * max(1.0, abs(tot))
    assert rel_err(out['logits'].cpu().numpy().transpose(1, 0, 2), aux['logits'].detach().numpy()) < 2e-4
    assert rel_err(out['attn'].cpu().numpy(), aux['attn'].detach().numpy()) < 2e-4
    worst = {}
    for vname in wts.decoder_shapes(c):
        ref = P[vname].grad.numpy()
        worst[vname] = rel_err(tr.gradient(vname).cpu().numpy().reshape(ref.shape), ref)
    assert any('gru_cell/candidate/kernel' in k for k in worst)
    bad = {k: v for k, v in worst.items() if not v < 1e-3}
    assert not bad, (bad, worst)


@pytest.mark.parametrize('name', ['xe_dropout', 'project_hidden'])
def test_gru_encoder_output_gradients_match_autograd(torch_mod, name):
    """comic_train_encoder_grads (cnn_finetune's input to the CNN backward) through the GRU init step."""
    import torch_ref as TR
    from comic_b200.train import Trainer
    mk, dropout, scst = CASES[name]
    c = mk()
    W, im, fm, caps, masks, keeps = _train_case(c, B=4, L=8, seed=3, dropout=dropout)
    P = TR.to_params(W)
    tot, _, _, _, aux = GO.training_loss(P, c, im, fm, caps, masks, keeps, None, fm_requires_grad=True)
    tot.backward()
    tr = Trainer(c, W, with_cnn=False)
    eng = tr.engine
    eng.set_precision('f32')
    out = tr.forward_backward(eng.to_dev(fm), eng.to_dev(im), caps, None, _dev_masks(eng, masks), keeps)
    dfm, demb = eng.train_encoder_grads(4, out['T_run'])
    assert rel_err(dfm.cpu().numpy(), aux['fm'].grad.numpy()) < 1e-3
    assert rel_err(demb.cpu().numpy(), aux['im'].grad.numpy()) < 1e-3


def test_gru_training_48_rows_fused_attention_and_tensor_path(torch_mod):
    """48 rows in the default precision (fused attention, K-split tensor GEMMs writing the GRU tape) against the sliced
    all-FFMA f32 run: same losses and gradients within the bf16x3 budget."""
    from comic_b200.train import Trainer
    c = comic_config(rnn_name='GRU', train_mode='decoder')
    W, im, fm, caps, masks, keeps = _train_case(c, B=48, L=7, seed=9, dropout=True)
    res = []
    for prec, min_images in (('split', 1), ('f32', 10000)):
        tr = Trainer(c, W, with_cnn=False)
        eng = tr.engine
        eng.set_precision(prec)
        eng.set_option('fused_attn_min_images', min_images)
        out = tr.forward_backward(eng.to_dev(fm), eng.to_dev(im), caps, None, _dev_masks(eng, masks), keeps, want_logits=True)
        res.append((out['loss'].cpu().numpy(), out['logits'].cpu().numpy(), tr.grads.cpu().numpy().copy()))
    (l1, lg1, g1), (l2, lg2, g2) = res
    np.testing.assert_allclose(l1, l2, rtol=1e-4, atol=1e-6)
    assert rel_err(lg1, lg2) < 2e-4
    assert rel_err(g1, g2) < 1e-3


def test_gru_cuda_graph_replay_of_fwd_bwd_is_bit_identical(torch_mod):
    from comic_b200.train import Trainer
    c = comic_config(rnn_name='GRU', train_mode='decoder', max_step=100)
    W, im, fm, caps, _, _ = _train_case(c, B=5, L=8, seed=7, dropout=False)
    runs = {}
    for graphed in (False, True):
        tr = Trainer(c, W, with_cnn=False)
        tr.cuda_graph = graphed
        eng = tr.engine
        got = []
        for i in range(5):
            scale = 1.0 + 0.1 * i
            masks, keeps = tr.make_masks(5, int((caps[:, 1:] >= 0).sum(1).max()), 100 + i)
            out = tr.forward_backward(eng.to_dev(fm * scale), eng.to_dev(im * scale), caps, None, masks, keeps)
            got.append((out['loss'].clone(), tr.grads.clone()))
        if graphed:
            assert any(e['graph'] is not None for e in tr._graphs.values())
        runs[graphed] = got
    for (l0, g0), (l1, g1) in zip(runs[False], runs[True]):
        assert torch_mod.equal(l0, l1) and torch_mod.equal(g0, g1)


def test_gru_training_steps_reduce_loss_and_decode_follows_the_update(torch_mod):
    """Adam steps on one batch lower the loss; after the last step a decode on the trainer's engine (weights updated in
    place, panels repacked) equals a decode of a fresh engine bound to the updated variables."""
    from comic_b200.engine import Engine
    from comic_b200.train import Trainer
    from comic_b200 import weights as wts
    c = comic_config(rnn_name='GRU', train_mode='decoder', max_step=100)
    W, im, fm, caps, _, _ = _train_case(c, B=6, L=9, seed=5, dropout=False)
    tr = Trainer(c, W, with_cnn=False)
    eng = tr.engine
    fm_d, im_d = eng.to_dev(fm), eng.to_dev(im)
    losses = []
    for _ in range(6):
        out = tr.forward_backward(fm_d, im_d, caps)
        losses.append(float(out['loss'][1].item()))
        tr.apply_gradients(lr=5e-3)
    assert losses[-1] < losses[0] - 0.05, losses
    W2 = {n: tr.variable(n).cpu().numpy().reshape(np.shape(W[n])) for n in wts.decoder_shapes(c)}
    assert not np.array_equal(W2[wts.cell_scope(c) + 'candidate/kernel'], W[wts.cell_scope(c) + 'candidate/kernel'])
    fresh = Engine(c)
    fresh.bind_weights(W2, with_cnn=False)

    def run(e):
        keys, values = e.project_fm(fm_d)
        c0, h0 = e.rnn_init(im_d)
        r = e.decode_beam(keys, values, c0, h0, 3, 0.0, 8)
        return r['predicted_ids'].cpu().numpy(), r['scores'].cpu().numpy()
    for a, b in zip(run(eng), run(fresh)):
        np.testing.assert_array_equal(a, b)

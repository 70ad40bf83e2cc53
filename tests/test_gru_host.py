"""GRU decoder cell (rnn_name=GRU) on the host: the cell equation against TF r1.9's testGRUCell, the oracle decoder
built on it, variable names / shapes / initialisers, checkpoint round trip and the CLI flag."""
import numpy as np
import pytest

from _common import comic_config, make_weights, fake_features, rel_err
import comic_oracle as O
import gru_oracle as GO
import tf19_gru_vectors as TFV
from comic_b200 import checkpoint as ck
from comic_b200 import cli
from comic_b200 import weights as wts

GRU = wts.DEC + 'rnn_init_input/gru_cell/'


@pytest.mark.parametrize('case', range(len(TFV.CASES)))
def test_gru_cell_reproduces_tf19_unit_test(case):
    x, expected = TFV.CASES[case]
    X = x.shape[1] + TFV.UNITS
    Kg = np.full((X, 2 * TFV.UNITS), TFV.KERNEL_INIT, np.float32)
    Kc = np.full((X, TFV.UNITS), TFV.KERNEL_INIT, np.float32)
    bg = np.full((2 * TFV.UNITS,), TFV.GATES_BIAS, np.float32)
    bc = np.full((TFV.UNITS,), TFV.CANDIDATE_BIAS, np.float32)
    h = GO.gru_cell(x, TFV.H, Kg, bg, Kc, bc)
    np.testing.assert_allclose(h, expected, atol=1e-6)


def test_gru_variables_shapes_and_parameter_count():
    c = comic_config(rnn_name='GRU')
    sh = wts.decoder_shapes(c)
    R, XH = c.rnn_size, c.rnn_word_size + c.rnn_size + c.rnn_size       # COMIC-256: A = R (tied projection)
    assert sh[GRU + 'gates/kernel'] == (XH, 2 * R) and sh[GRU + 'gates/bias'] == (2 * R,)
    assert sh[GRU + 'candidate/kernel'] == (XH, R) and sh[GRU + 'candidate/bias'] == (R,)
    assert not any('basic_lstm_cell' in n for n in sh)
    # 4,297,987 (LSTM, README) - 2,623,488 (LSTM kernel + bias) + 1,967,616 (GRU kernels + biases)
    assert wts.count_params(sh) == 3642115
    ph = wts.decoder_shapes(comic_config(rnn_name='GRU', rnn_init_method='project_hidden'))
    assert wts.DEC + 'gru_cell/gates/kernel' in ph and wts.DEC + 'rnn_initial_state/weight' in ph
    assert wts.cell_scope(comic_config(rnn_name='GRU', rnn_init_method='project_hidden')) == wts.DEC + 'gru_cell/'
    # the LSTM model is untouched
    assert wts.count_params(wts.decoder_shapes(comic_config())) == 4297987


def test_gru_initialisers():
    c = comic_config(rnn_name='GRU')
    W = wts.init_weights(c, include_cnn=False)
    np.testing.assert_array_equal(W[GRU + 'gates/bias'], 1.0)           # GRUCell's constant 1.0 gate bias
    np.testing.assert_array_equal(W[GRU + 'candidate/bias'], 0.0)
    lim = np.sqrt(6.0 / sum(W[GRU + 'gates/kernel'].shape))               # Xavier
    assert 0 < np.abs(W[GRU + 'gates/kernel']).max() <= lim
    P = wts.perturb_for_parity(W)
    assert np.std(P[GRU + 'gates/bias']) > 0 and np.std(P[GRU + 'candidate/bias']) > 0


@pytest.mark.parametrize('init', ['first_input', 'project_hidden'])
def test_gru_oracle_decoder_steps(init):
    """GRUDecoder.call is MultiHeadAttentionWrapperV3 over gru_cell; the init state follows _get_rnn_init."""
    c = comic_config(rnn_name='GRU', rnn_init_method=init)
    W = make_weights(c, include_cnn=False)
    dec = GO.GRUDecoder(W, c)
    B = 3
    im, fm = fake_features(B)
    dec.setup_memory(fm)
    _, h0 = dec.init_state(im)
    s = dec.cell_scope
    if init == 'project_hidden':
        np.testing.assert_allclose(h0, im @ W[wts.DEC + 'rnn_initial_state/weight'], rtol=1e-5)
    else:
        x0 = im @ W[wts.DEC + 'rnn_init_input/projection/weight']
        R = c.rnn_size
        u0 = O.sigmoid(x0 @ W[s + 'gates/kernel'][:x0.shape[1], R:] + W[s + 'gates/bias'][R:])
        c0 = np.tanh(x0 @ W[s + 'candidate/kernel'][:x0.shape[1]] + W[s + 'candidate/bias'])
        np.testing.assert_allclose(h0, (1 - u0) * c0, rtol=1e-4, atol=1e-6)
    state = dec.zero_state(dec.init_state(im))
    toks = np.array([1, 5, 9], np.int32)
    out, ns, _ = dec.call(dec.embed(toks), state)
    x = np.concatenate([dec.embed(toks), state['attention']], axis=1)
    ref = GO.gru_cell(x, h0, W[s + 'gates/kernel'], W[s + 'gates/bias'], W[s + 'candidate/kernel'], W[s + 'candidate/bias'])
    np.testing.assert_allclose(out, ref, rtol=1e-6)
    np.testing.assert_array_equal(out, ns['h'])
    # the oracle's search loops run unchanged on the GRU decoder
    res = O.beam_search_decode(GO.GRUDecoder(W, c), im, fm, 3, 0.0, 4)
    assert res['predicted_ids'].shape[1:] == (B, 3)


def test_gru_checkpoint_round_trip(tmp_path):
    c = comic_config(rnn_name='GRU')
    W = wts.init_weights(c, seed=5, include_cnn=False)
    prefix = str(tmp_path / 'run' / 'model_compact-3')
    rng = np.random.default_rng(0)
    trained = {k: (np.asarray(v) + rng.standard_normal(np.shape(v)).astype(np.float32) * 0.01).astype(np.float32)
               for k, v in W.items()}
    ck.write_v2(prefix, trained, with_data_crc=False)
    shapes = ck.variable_shapes(prefix)
    assert shapes[GRU + 'gates/kernel'] == [1280, 1024] and shapes[GRU + 'candidate/bias'] == [512]
    c.checkpoint_path, c.resume_training, c.checkpoint_exclude_scopes = str(tmp_path / 'run'), True, ''
    got, info = ck.restore_weights(c, W)
    assert info['mode'] == 'resume'
    for k in W:
        np.testing.assert_array_equal(got[k], trained[k])


def test_cli_accepts_gru():
    """--rnn_name is a train.py flag (inference reads it from the run's config.pkl)."""
    args = cli.create_train_parser().parse_args(['--rnn_name', 'GRU'])
    assert cli.config_from_train_args(args).rnn_name == 'GRU'


def test_ln_lstm_still_refused():
    """LN_LSTM is not built: the wrapper refuses it before touching a device (Engine: tests/test_gpu_gru.py)."""
    from comic_b200 import rops
    with pytest.raises(NotImplementedError, match='Only `LSTM` and `GRU`'):
        rops.MultiHeadAttentionWrapperV3(cell='LN_LSTM', attention_mechanism=object())


@pytest.mark.parametrize('mode', ['xe', 'scst'])
@pytest.mark.parametrize('init', ['first_input', 'project_hidden'])
def test_torch_gru_training_reference_matches_oracle_forward(init, mode):
    """The fp64 autograd reference of GRU training (gru_oracle.training_loss) computes the oracle's teacher-forced decode
    and loss, dropout masks included."""
    import torch_ref as TR
    from test_oracle_known_answers import _train_case
    c = comic_config(rnn_name='GRU', rnn_init_method=init)
    W, im, fm, caps, masks, keeps = _train_case(c)
    dec = GO.GRUDecoder(W, c, np.float64)
    inputs, targets, wmask, lens = O.process_inputs(caps, c.token_type)
    m64 = {k: v.astype(np.float64) for k, v in masks.items()}
    r = O.training_decode(dec, im.astype(np.float64), fm.astype(np.float64), inputs, lens, m64, keeps)
    _, _, am = O.post_process_plain(r['logits'], r['ids'], r['alignment_history'], c.attn_num_heads)
    rewards = None if mode == 'xe' else np.array([0.3, -0.2, 1.1])
    Wd = {k: v for k, v in W.items() if k.startswith('Model/decoder')}
    tot, xe, mp, reg = O.caption_loss(r['logits'].transpose(1, 0, 2), targets, wmask.astype(np.float64), am, Wd, c, rewards)
    P = TR.to_params(W)
    t_tot, t_xe, t_map, t_reg, aux = GO.training_loss(P, c, im, fm, caps, masks, keeps, rewards)
    assert rel_err(aux['logits'].detach().numpy(), r['logits']) < 1e-9
    assert rel_err(aux['attn'].detach().numpy(), am) < 1e-9
    assert abs(float(t_xe) - float(xe)) < 1e-9 * max(1, abs(float(xe)))
    assert abs(float(t_tot) - float(tot)) < 1e-9 * max(1, abs(float(tot)))
    t_tot.backward()
    g = P[dec.cell_scope + 'candidate/kernel'].grad
    assert g is not None and bool(g.abs().sum() > 0)
    assert TR._lstm.__name__ == '_lstm'                               # the hook is restored

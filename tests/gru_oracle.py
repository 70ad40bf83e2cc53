"""ORACLE (test infrastructure, not product code) -- the GRU decoder cell, restated in NumPy beside
oracle/comic_oracle.py.

The cell is TF r1.9 `rnn_cell_impl.GRUCell` (`tf.contrib.rnn.GRUCell`), created in src/model_base.py:622-629 when
c.rnn_name == 'GRU':

    [r, u] = sigmoid([x, h] . gates/kernel + gates/bias)          gates/kernel [W+A+R, 2R], r first
    c      = tanh([x, r*h] . candidate/kernel + candidate/bias)   candidate/kernel [W+A+R, R]
    h'     = u*h + (1-u)*c                                        output == new state (a tensor)

`GRUDecoder` is `comic_oracle.Decoder` with this cell in place of BasicLSTMCell.  The Decoder calls its cell through
`Decoder.lstm(x, c_prev, h_prev)`; the GRU passes `c` through unchanged, so the state dicts keep a `c` entry that no
GRU computation reads, and `beam_search_decode`, `greedy_decode` and `training_decode` run on it unmodified.  The
initial state (src/model_base.py:651-689) follows from the same hook: first_input runs the cell once on the projected
im_embed from a zero state, project_hidden is h0 = im_embed . rnn_initial_state/weight.

PARITY UNPINNED as the rest of the oracle (DESIGN.md §2); the cell equation itself is pinned by TF's own testGRUCell
vectors (tests/golden/tf19_gru_vectors.py).
"""
import copy

import numpy as np

import comic_oracle as O


def gru_cell(x, h, Kg, bg, Kc, bc):
    """One GRUCell step: x [N, X], h [N, R] -> h' [N, R]."""
    g = O.sigmoid(np.concatenate([x, h], axis=1) @ Kg + bg)
    r, u = np.split(g, 2, axis=1)
    c = np.tanh(np.concatenate([x, r * h], axis=1) @ Kc + bc)
    return u * h + (1 - u) * c


class GRUDecoder(O.Decoder):
    """The attention-GRU decoder of one sequence batch (MultiHeadAttentionWrapperV3 over GRUCell)."""

    def __init__(self, W, config, dtype=np.float32):
        if config.rnn_name != 'GRU':
            raise ValueError('GRUDecoder restates rnn_name=GRU')
        lstm_view = copy.copy(config)
        lstm_view.rnn_name = 'LSTM'                  # Decoder.__init__ checks the name only; every other field is shared
        super(GRUDecoder, self).__init__(W, lstm_view, dtype)
        self.c = config
        self.cell_scope = O.DEC + ('rnn_init_input/gru_cell/' if config.rnn_init_method == 'first_input'
                                   else 'gru_cell/')

    def lstm(self, x, c_prev, h_prev):
        s = self.cell_scope
        h_new = gru_cell(x, h_prev, self.W[s + 'gates/kernel'], self.W[s + 'gates/bias'],
                         self.W[s + 'candidate/kernel'], self.W[s + 'candidate/bias'])
        return c_prev, h_new


def _torch_gru(P, c, x, c_prev, h_prev):
    import torch
    s = O.DEC + ('rnn_init_input/gru_cell/' if c.rnn_init_method == 'first_input' else 'gru_cell/')
    g = torch.sigmoid(torch.cat([x, h_prev], 1) @ P[s + 'gates/kernel'] + P[s + 'gates/bias'])
    r, u = g.chunk(2, 1)
    cand = torch.tanh(torch.cat([x, r * h_prev], 1) @ P[s + 'candidate/kernel'] + P[s + 'candidate/bias'])
    return c_prev, u * h_prev + (1 - u) * cand


def training_loss(P, c, *args, **kw):
    """tests/torch_ref.training_loss (fp64 autograd reference of the training forward + loss) with the GRU cell.
    torch_ref calls its cell through `_lstm(P, c, x, c_prev, h_prev)`; the GRU takes that hook for the duration of the
    call and passes c through unchanged, as GRUDecoder does."""
    import torch_ref as TR
    cell = TR._lstm
    TR._lstm = _torch_gru
    try:
        return TR.training_loss(P, c, *args, **kw)
    finally:
        TR._lstm = cell

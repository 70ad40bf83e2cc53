"""Weight container for the COMIC hot path (SURVEY.md §8a W-table).

Holds every tensor of the reference graph under the reference's TF variable
names with the reference's shapes, as numpy fp32 arrays (host side).  The CUDA
engine packs them into its own HBM layout at bind time (`engine.py`).

Reference sites:
  decoder variables   src/model_base.py:531-554 (word projections), :606-689
                      (cell + init), common/ops_rnn.py:441-442,470,545-561
  encoder variables   common/nets/inception_v1.py:29-266 (57 convs),
                      common/nets/inception_utils.py:56-66 (BN: no gamma)
  initialisers        src/model_base.py:823-831 (xavier), inception_v1.py:26
                      (truncated_normal(0.01)), ops_rnn.py:559 (T = 5.0)
"""
from __future__ import annotations

import numpy as np

DEC = 'Model/decoder/rnn_decoder/'
ENC = 'Model/encoder/'
CNN = 'Model/encoder/cnn/InceptionV1/'

# ---------------------------------------------------------------------------
# InceptionV1 layer table (common/nets/inception_v1.py:70-265).
# Each inception block: (name, c_in, b0, b1a, b1b, b2a, b2b, b3)
# ---------------------------------------------------------------------------
STEM = [
    # (kind, name, k, stride, c_in, c_out)
    ('conv', 'Conv2d_1a_7x7', 7, 2, 3, 64),      # inception_v1.py:70
    ('maxpool', 'MaxPool_2a_3x3', 3, 2, 64, 64),  # :75
    ('conv', 'Conv2d_2b_1x1', 1, 1, 64, 64),     # :80
    ('conv', 'Conv2d_2c_3x3', 3, 1, 64, 192),    # :85
    ('maxpool', 'MaxPool_3a_3x3', 3, 2, 192, 192),  # :90
]
BLOCKS = [
    ('Mixed_3b', 192, 64, 96, 128, 16, 32, 32),     # :95-111
    ('Mixed_3c', 256, 128, 128, 192, 32, 96, 64),   # :113-129
    ('MaxPool_4a_3x3', 3, 2),                         # :131-132
    ('Mixed_4b', 480, 192, 96, 208, 16, 48, 64),    # :136-152
    ('Mixed_4c', 512, 160, 112, 224, 24, 64, 64),   # :154-170
    ('Mixed_4d', 512, 128, 128, 256, 24, 64, 64),   # :172-188
    ('Mixed_4e', 512, 112, 144, 288, 32, 64, 64),   # :190-206
    ('Mixed_4f', 528, 256, 160, 320, 32, 128, 128),  # :208-224
    ('MaxPool_5a_2x2', 2, 2),                         # :226-227
    ('Mixed_5b', 832, 256, 160, 320, 32, 128, 128),  # :231-247
    ('Mixed_5c', 832, 384, 192, 384, 48, 128, 128),  # :249-265
]


def block_conv_scopes(name):
    """Scopes of the six convs of one inception block, in reference order.
    Mixed_5b's Branch_2 3x3 is scoped `Conv2d_0a_3x3` (inception_v1.py:240)."""
    b2b = 'Conv2d_0a_3x3' if name == 'Mixed_5b' else 'Conv2d_0b_3x3'
    return [name + '/Branch_0/Conv2d_0a_1x1',
            name + '/Branch_1/Conv2d_0a_1x1',
            name + '/Branch_1/Conv2d_0b_3x3',
            name + '/Branch_2/Conv2d_0a_1x1',
            name + '/Branch_2/' + b2b,
            name + '/Branch_3/Conv2d_0b_1x1']


def cnn_conv_list():
    """[(scope, k, stride, c_in, c_out)] for all 57 convs."""
    out = []
    for s in STEM:
        if s[0] == 'conv':
            out.append((s[1], s[2], s[3], s[4], s[5]))
    for b in BLOCKS:
        if len(b) == 3:
            continue
        name, cin, b0, b1a, b1b, b2a, b2b, b3 = b
        sc = block_conv_scopes(name)
        out += [(sc[0], 1, 1, cin, b0), (sc[1], 1, 1, cin, b1a),
                (sc[2], 3, 1, b1a, b1b), (sc[3], 1, 1, cin, b2a),
                (sc[4], 3, 1, b2a, b2b), (sc[5], 1, 1, cin, b3)]
    return out


def fm_channels(endpoint):
    for b in BLOCKS:
        if b[0] == endpoint and len(b) > 3:
            return b[2] + b[4] + b[6] + b[7]
    raise ValueError('Unknown feature-map end point %s' % endpoint)


# ---------------------------------------------------------------------------
# Model dimensions derived from a config (src/model_base.py:40-46, 611-615).
# ---------------------------------------------------------------------------
class Dims(object):
    def __init__(self, c):
        self.R = int(c.rnn_size)
        self.W = int(c.rnn_word_size)
        self.H = int(c.attn_num_heads)
        self.C = fm_channels(c.cnn_fm_attention)
        self.E = 1024
        self.M = 196
        self.fm_projection = c.cnn_fm_projection        # None|'tied'|'independent'
        self.context_layer = bool(c.attn_context_layer)
        if self.fm_projection is None and not self.context_layer:
            self.A = self.C                              # model_base.py:611-612
        else:
            self.A = self.R
        # width of the value tensor the context is taken over (ops_rnn.py:460-477)
        self.VAL = self.C if self.fm_projection is None else self.R
        if c.token_type == 'radix':
            self.V = int(c.radix_base) + 2               # model_base.py:42-43
        else:
            self.V = len(c.itow)                         # :45
        self.legacy = bool(c.legacy)
        self.init_method = c.rnn_init_method
        self.token_type = c.token_type


def decoder_shapes(c):
    """name -> shape for all decoder variables (SURVEY §8a W-table)."""
    d = Dims(c)
    sh = {}
    if d.init_method == 'first_input':
        sh[DEC + 'rnn_init_input/projection/weight'] = (d.E, d.W + d.A)
    else:
        sh[DEC + 'rnn_initial_state/weight'] = (d.E, d.R)
    cs = cell_scope(c)
    if c.rnn_name == 'GRU':                      # TF r1.9 GRUCell: gates [r, u], candidate
        sh[cs + 'gates/kernel'] = (d.W + d.A + d.R, 2 * d.R)
        sh[cs + 'gates/bias'] = (2 * d.R,)
        sh[cs + 'candidate/kernel'] = (d.W + d.A + d.R, d.R)
        sh[cs + 'candidate/bias'] = (d.R,)
    else:
        sh[cs + 'kernel'] = (d.W + d.A + d.R, 4 * d.R)
        sh[cs + 'bias'] = (4 * d.R,)
    sh[DEC + 'memory_layer/kernel'] = (d.C, d.R)
    if d.fm_projection == 'independent':
        sh[DEC + 'value_layer/kernel'] = (d.C, d.R)
    att = DEC + 'multi_add_attention/'
    sh[att + 'query_layer/kernel'] = (d.R, d.R)
    sh[att + 'attention_v'] = (d.R,)
    sh[att + 'LN_tanh/beta'] = (d.R,)
    sh[att + 'LN_tanh/gamma'] = (d.R,)
    sh[DEC + 'softmax_temperature'] = ()
    if d.context_layer:
        sh[DEC + 'a_layer/kernel'] = (d.VAL, d.R)
    sh[DEC + 'output_projection/kernel'] = (d.R, d.V)
    sh[DEC + 'output_projection/bias'] = (d.V,)
    sh[DEC + 'embedding_map'] = (d.V, d.W)
    return sh


def encoder_head_shapes(c):
    """Legacy-only encoder head (src/model_base.py:80-91); not part of the
    README's decoder parameter counts."""
    sh = {}
    if c.legacy:
        sh[ENC + 'LN_tanh/beta'] = (1024,)
        sh[ENC + 'LN_tanh/gamma'] = (1024,)
        sh[ENC + 'im_embed/weight'] = (1024, 1024)
    return sh


def cell_scope(c):
    """Variable scope of the decoder cell (src/model_base.py:622-629): `basic_lstm_cell` (LSTM) or `gru_cell` (GRU),
    under `rnn_init_input/` when the first_input init step created it."""
    cell = 'gru_cell/' if c.rnn_name == 'GRU' else 'basic_lstm_cell/'
    return DEC + ('rnn_init_input/' if c.rnn_init_method == 'first_input' else '') + cell


def cnn_shapes():
    sh = {}
    for scope, k, _s, cin, cout in cnn_conv_list():
        sh[CNN + scope + '/weights'] = (k, k, cin, cout)
        sh[CNN + scope + '/BatchNorm/beta'] = (cout,)
        sh[CNN + scope + '/BatchNorm/moving_mean'] = (cout,)
        sh[CNN + scope + '/BatchNorm/moving_variance'] = (cout,)
    return sh


def count_params(shapes):
    return int(sum(int(np.prod(s)) for s in shapes.values()))


def _xavier(rng, shape):
    """slim.xavier_initializer (uniform): +-sqrt(6/(fan_in+fan_out)); for a
    rank-1 shape TF uses fan_in = fan_out = shape[0]."""
    if len(shape) == 0:
        fan_in = fan_out = 1
    elif len(shape) == 1:
        fan_in = fan_out = shape[0]
    elif len(shape) == 2:
        fan_in, fan_out = shape
    else:
        rf = int(np.prod(shape[:-2]))
        fan_in, fan_out = shape[-2] * rf, shape[-1] * rf
    lim = np.sqrt(6.0 / (fan_in + fan_out))
    return rng.uniform(-lim, lim, size=shape).astype(np.float32)


def init_weights(c, seed=48964896, cnn_init='he', include_cnn=True):
    """Seeded random-init weights with the reference's initialisers.

    cnn_init: 'reference' = truncated_normal(0.01) conv weights, BN mu=0,
    var=1, beta=0 (activations collapse towards 0, SURVEY §8a); 'he' =
    variance-preserving He-normal conv weights so that parity checks on the
    feature map are meaningful.
    """
    rng = np.random.default_rng(seed)
    w = {}
    shapes = dict(decoder_shapes(c))
    shapes.update(encoder_head_shapes(c))
    for name, shape in shapes.items():
        if name.endswith('gru_cell/gates/bias'):
            w[name] = np.ones(shape, np.float32)           # GRUCell: constant 1.0 gate bias
        elif name.endswith('basic_lstm_cell/bias') or name.endswith('gru_cell/candidate/bias') \
                or name.endswith('LN_tanh/beta') or name.endswith('output_projection/bias'):
            w[name] = np.zeros(shape, np.float32)
        elif name.endswith('LN_tanh/gamma'):
            w[name] = np.ones(shape, np.float32)
        elif name.endswith('softmax_temperature'):
            w[name] = np.array(5.0, np.float32)
        else:
            w[name] = _xavier(rng, shape)
    if include_cnn:
        for scope, k, _s, cin, cout in cnn_conv_list():
            shape = (k, k, cin, cout)
            if cnn_init == 'reference':
                x = rng.standard_normal(size=shape) * 0.01
                x = np.clip(x, -0.02, 0.02)      # truncated at 2 sigma
            else:
                x = rng.standard_normal(size=shape) * np.sqrt(2.0 / (k * k * cin))
            w[CNN + scope + '/weights'] = x.astype(np.float32)
            w[CNN + scope + '/BatchNorm/beta'] = np.zeros((cout,), np.float32)
            w[CNN + scope + '/BatchNorm/moving_mean'] = np.zeros((cout,), np.float32)
            w[CNN + scope + '/BatchNorm/moving_variance'] = np.ones((cout,), np.float32)
    return w


def perturb_for_parity(w, seed=7):
    """Make zero/one-initialised tensors non-trivial (biases, LN beta/gamma, BN
    statistics) so that parity tests exercise every term of the graph."""
    rng = np.random.default_rng(seed)
    out = dict(w)
    for k, v in w.items():
        if k.endswith('/bias') or k.endswith('LN_tanh/beta'):
            out[k] = (rng.standard_normal(v.shape) * 0.1).astype(np.float32)
        elif k.endswith('LN_tanh/gamma'):
            out[k] = (1.0 + rng.standard_normal(v.shape) * 0.1).astype(np.float32)
        elif k.endswith('BatchNorm/beta'):
            out[k] = (rng.standard_normal(v.shape) * 0.1).astype(np.float32)
        elif k.endswith('moving_mean'):
            out[k] = (rng.standard_normal(v.shape) * 0.1).astype(np.float32)
        elif k.endswith('moving_variance'):
            out[k] = rng.uniform(0.5, 1.5, v.shape).astype(np.float32)
    return out

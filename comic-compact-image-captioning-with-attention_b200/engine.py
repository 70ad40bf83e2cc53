"""ctypes binding of libcomic_b200.so (include/comic_b200.h).

PyTorch is used for device memory, the caching allocator and the current
stream only; every FLOP of the hot path runs in the library's hand-written
sm_100a kernels.  There is no CPU or eager fallback: if the library is missing
or no CUDA device is present, constructing an `Engine` raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import weights as wts

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libcomic_b200.so')
NUM_CONVS = 57

FM_PROJ = {None: 0, 'none': 0, 'tied': 1, 'independent': 2}
ALIGN = {'add_LN': 0, 'dot': 1}
PROB = {'softmax': 0, 'sigmoid': 1}
INIT = {'first_input': 0, 'project_hidden': 1}
CELL = {'LSTM': 0, 'GRU': 1}                   # COMIC_CELL_*


class ComicCfg(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        'rnn_size', 'word_size', 'num_heads', 'fm_channels', 'fm_positions', 'embed_size', 'vocab',
        'fm_projection', 'context_layer', 'init_method', 'alignment', 'prob_fn', 'embed_lookup',
        'legacy', 'go_id', 'eos_id')]


_FP = C.c_void_p


class ComicWeights(C.Structure):
    _fields_ = [(n, _FP) for n in (
        'lstm_kernel', 'lstm_bias', 'init_weight', 'memory_kernel', 'value_kernel', 'query_kernel',
        'attention_v', 'ln_gamma', 'ln_beta', 'temperature', 'a_layer', 'out_kernel', 'out_bias',
        'embedding_map', 'enc_ln_gamma', 'enc_ln_beta', 'enc_embed_weight')] + [
        ('conv_w', _FP * NUM_CONVS), ('bn_beta', _FP * NUM_CONVS), ('bn_mean', _FP * NUM_CONVS),
        ('bn_var', _FP * NUM_CONVS)]


class ComicTrainMasks(C.Structure):
    _fields_ = [('init_in', _FP), ('inp', _FP), ('out', _FP), ('att', _FP),
                ('in_keep', C.c_float), ('out_keep', C.c_float), ('att_keep', C.c_float)]


GRAD_FIELDS = ('lstm_kernel', 'lstm_bias', 'init_weight', 'memory_kernel', 'value_kernel', 'query_kernel',
               'attention_v', 'ln_gamma', 'ln_beta', 'temperature', 'out_kernel', 'out_bias', 'embedding_map', 'a_layer',
               'cand_kernel', 'cand_bias')


class ComicDecoderGrads(C.Structure):
    _fields_ = [(n, _FP) for n in GRAD_FIELDS]


class ComicCnnGrads(C.Structure):
    _fields_ = [('conv_w', _FP * NUM_CONVS), ('bn_beta', _FP * NUM_CONVS)]


class ComicConvDesc(C.Structure):
    _fields_ = [('k', C.c_int32), ('stride', C.c_int32), ('c_in', C.c_int32), ('c_out', C.c_int32)]


class ComicError(RuntimeError):
    pass


_lib = None

# (name, restype, argtypes) for every symbol include/comic_b200.h declares.
_I, _F, _SZ, _P = C.c_int, C.c_float, C.c_size_t, C.c_void_p
SIGNATURES = {
    'comic_last_error': (C.c_char_p, []),
    'comic_version': (C.c_char_p, []),
    'comic_conv_table': (C.POINTER(ComicConvDesc), []),
    'comic_create': (_I, [C.POINTER(ComicCfg), C.POINTER(_P)]),
    'comic_destroy': (_I, [_P]),
    'comic_packed_bytes': (_I, [_P, C.POINTER(_SZ)]),
    'comic_bind_weights': (_I, [_P, C.POINTER(ComicWeights), _I, _P, _SZ, _P]),
    'comic_set_rnn_cell': (_I, [_P, _I]),
    'comic_bind_gru_candidate': (_I, [_P, _P, _P]),
    'comic_workspace_bytes': (_I, [_P, _I, _I, _I, _I, C.POINTER(_SZ)]),
    'comic_encode_fwd': (_I, [_P, _P, _I, _P, _P, _P, _P, _SZ, _P]),
    'comic_preprocess_eval': (_I, [_P, _P, _I, _I, _I, _I, _I, _P, _P]),
    'comic_project_fm': (_I, [_P, _P, _I, _P, _P, _P]),
    'comic_rnn_init': (_I, [_P, _P, _I, _P, _P, _P, _F, _P, _SZ, _P]),
    'comic_decode_step': (_I, [_P, _P, _P, _I, _I, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P,
                               _F, _F, _F, _P, _SZ, _P]),
    'comic_decode_greedy': (_I, [_P, _P, _P, _P, _P, _I, _I, _P, _P, _P, _P, _P, _SZ, _P]),
    'comic_decode_beam': (_I, [_P, _P, _P, _P, _P, _I, _I, _F, _I, _P, _P, _P, _P, _P, _P, _P, _P, _SZ, _P]),
    'comic_beam_step': (_I, [_P, _P, _I, _I, _I, _I, _I, _F, _P, _P, _P, _P, _P, _P, _P]),
    'comic_gather_tree': (_I, [_P, _P, _P, _P, _I, _I, _I, _I, _P, _P]),
    'comic_gemm_f32': (_I, [_P, _P, _I, _P, _I, _P, _P, _I, _I, _I, _I, _P, _SZ, _P]),
    'comic_launch_count': (_I, [_P, C.POINTER(C.c_int64)]),
    'comic_set_precision': (_I, [_P, _I]),
    'comic_set_option': (_I, [_P, _I, _I]),
    'comic_preprocess_train': (_I, [_P, _P, _I, _I, _I, _I, _I, _P, _P, _P, _P]),
    'comic_decode_trace': (_I, [_P, _P, _I, _P, _P]),
    'comic_train_workspace_bytes': (_I, [_P, _I, _I, C.POINTER(_SZ)]),
    'comic_dropout_masks': (_I, [_P, _P, _SZ, _F, C.c_uint64, C.c_uint64, _P]),
    'comic_train_fwd_bwd': (_I, [_P, _P, _P, _I, _P, _P, _P, _P, _I, _I, C.POINTER(ComicTrainMasks), _F, _P, _P, _P,
                                 C.POINTER(ComicDecoderGrads), _P, _SZ, _P]),
    'comic_l2_regularise': (_I, [_P, _P, _P, _SZ, _F, _P, _P, _SZ, _P]),
    'comic_adam_step': (_I, [_P, _P, _P, _P, _P, _SZ, _F, _F, _F, _F, _I, _F, _P]),
    'comic_momentum_step': (_I, [_P, _P, _P, _P, _SZ, _F, _F, _F, _P]),
    'comic_clip_by_norm': (_I, [_P, _P, _P, _P, _I, _F, _P]),
    'comic_refresh_packed': (_I, [_P, _P, _SZ, _P]),
    'comic_refresh_packed_cnn': (_I, [_P, _P, _SZ, _P]),
    'comic_train_encoder_grads': (_I, [_P, _I, _I, _P, _P, _P, _SZ, _P]),
    'comic_legacy_head_bwd_bytes': (_I, [_P, _I, _P]),
    'comic_legacy_head_bwd': (_I, [_P, _P, _I, _P, _P, _P, _P, _P, _SZ, _P]),
    'comic_encode_train_bytes': (_I, [_P, _I, C.POINTER(_SZ), C.POINTER(_SZ)]),
    'comic_encode_train_fwd': (_I, [_P, _P, _I, _P, _P, _P, _SZ, _P, _SZ, _P]),
    'comic_encode_bwd': (_I, [_P, _P, _I, _P, _P, _P, _SZ, C.POINTER(ComicCnnGrads), _P, _SZ, _P]),
    'comic_profile_enable': (_I, [_P, C.c_uint32]),
    'comic_profile_read': (_I, [_P, _I, C.POINTER(C.c_double), C.POINTER(C.c_int64)]),
}

KERNEL_TAGS = ['conv', 'pool', 'project', 'init', 'gates', 'lstm', 'lq', 'scores', 'ctx', 'beam',
               'final', 'misc', 'persist']


def load_library(path=LIB_PATH):
    """dlopen the C-ABI library and type every exported symbol."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get('COMIC_B200_LIB', path)      # experiment builds (same ABI); still no fallback
    if not os.path.exists(path):
        raise ComicError('libcomic_b200.so not built (%s); run `python __graft_entry__.py build`' % path)
    lib = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)      # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def executed_steps(T):
    """Host read of a decode call's executed step count (the one device->host sync); -1 is the
    persistent loop kernel's watchdog verdict (a grid barrier never completed)."""
    t = int(T.item())
    if t < 0:
        raise ComicError('decode loop aborted: the persistent kernel gave up at a grid barrier')
    return t


def _ptr(t):
    if t is None:
        return None
    return C.c_void_p(t.data_ptr())


class Engine(object):
    """One handle = one model description on one GPU (one process per GPU)."""

    def __init__(self, config, device=None):
        import torch
        if not torch.cuda.is_available():
            raise ComicError('comic_b200 requires a CUDA device (B200, sm_100a); no CPU fallback exists')
        self.torch = torch
        self.lib = load_library()
        self.device = torch.device('cuda', torch.cuda.current_device() if device is None else device)
        torch.cuda.set_device(self.device)
        self.c = config
        d = self.dims = wts.Dims(config)
        if config.rnn_name not in CELL:
            raise ComicError('rnn_name=%s is not built (LSTM and GRU are)' % config.rnn_name)
        self.gru = config.rnn_name == 'GRU'
        if config.attn_alignment_method not in ALIGN:
            raise ValueError('Invalid alignment method.')             # src/model_base.py:133-138
        if config.attn_probability_fn not in PROB:
            raise ValueError('Invalid alignment method.')             # src/model_base.py:140-145
        if config.token_type == 'radix':
            go, eos = config.radix_base, config.radix_base + 1        # src/model_base.py:701-703
        else:
            go, eos = config.wtoi['<GO>'], config.wtoi['<EOS>']
        self.go, self.eos = int(go), int(eos)
        cfg = ComicCfg(
            rnn_size=d.R, word_size=d.W, num_heads=d.H, fm_channels=d.C, fm_positions=d.M,
            embed_size=d.E, vocab=d.V, fm_projection=FM_PROJ[config.cnn_fm_projection],
            context_layer=int(bool(config.attn_context_layer)), init_method=INIT[config.rnn_init_method],
            alignment=ALIGN[config.attn_alignment_method], prob_fn=PROB[config.attn_probability_fn],
            embed_lookup=int(config.token_type == 'word'), legacy=int(bool(config.legacy)),
            go_id=self.go, eos_id=self.eos)
        self._h = C.c_void_p()
        self._check(self.lib.comic_create(C.byref(cfg), C.byref(self._h)))
        self._check(self.lib.comic_set_rnn_cell(self._h, CELL[config.rnn_name]))
        self._dev_weights = {}
        self._packed = None
        self._ws = {}
        self.bound_cnn = False
        # experiment hook: COMIC_B200_OPTS="name=value,..." applies engine tunables (set_option) to every
        # engine of the process, e.g. to run the whole test suite on a non-default kernel variant
        for kv in filter(None, os.environ.get('COMIC_B200_OPTS', '').split(',')):
            name, value = kv.split('=')
            self.set_option(name.strip(), int(value))

    # -- plumbing -----------------------------------------------------------
    def _check(self, rc):
        if rc != 0:
            msg = self.lib.comic_last_error().decode()
            if rc == -4:
                raise NotImplementedError(msg)
            if rc in (-1, -2):
                raise ValueError(msg)
            raise ComicError('comic_b200 error %d: %s' % (rc, msg))

    def __del__(self):
        try:
            if self._h:
                self.lib.comic_destroy(self._h)
                self._h = C.c_void_p()
        except Exception:
            pass

    def stream(self):
        return C.c_void_p(self.torch.cuda.current_stream(self.device).cuda_stream)

    def _workspace(self, mode, B, k, T):
        n = C.c_size_t()
        self._check(self.lib.comic_workspace_bytes(self._h, mode, B, k, T, C.byref(n)))
        key = mode
        buf = self._ws.get(key)
        if buf is None or buf.numel() < n.value:
            buf = self.torch.empty(n.value, dtype=self.torch.uint8, device=self.device)
            self._ws[key] = buf
        return buf

    def f32(self, *shape):
        return self.torch.empty(shape, dtype=self.torch.float32, device=self.device)

    def to_dev(self, a, dtype=None):
        t = self.torch.as_tensor(a)
        if dtype is not None:
            t = t.to(dtype)
        return t.to(self.device).contiguous()

    # -- weights ------------------------------------------------------------
    def bind_weights(self, W, with_cnn=True):
        """W: dict TF-variable-name -> numpy/torch fp32 array (weights.py)."""
        torch = self.torch
        c = self.c
        dev = {}
        for k, v in W.items():
            dev[k] = torch.as_tensor(np.ascontiguousarray(v) if isinstance(v, np.ndarray) else v,
                                     dtype=torch.float32).to(self.device).contiguous()
        self._dev_weights = dev
        self._bind_generation = getattr(self, '_bind_generation', 0) + 1      # invalidates captured graphs (Engine.graphed)
        D, ENC, CNN = wts.DEC, wts.ENC, wts.CNN
        cs = wts.cell_scope(c)
        att = D + 'multi_add_attention/'

        def g(name):
            t = dev.get(name)
            return None if t is None else C.c_void_p(t.data_ptr())
        w = ComicWeights()
        if self.gru:     # gates/{kernel, bias} travel in the LSTM fields; the candidate is bound by pointer beside them
            w.lstm_kernel = g(cs + 'gates/kernel')
            w.lstm_bias = g(cs + 'gates/bias')
            self._check(self.lib.comic_bind_gru_candidate(self._h, g(cs + 'candidate/kernel'), g(cs + 'candidate/bias')))
        else:
            w.lstm_kernel = g(cs + 'kernel')
            w.lstm_bias = g(cs + 'bias')
        w.init_weight = g(D + ('rnn_init_input/projection/weight' if c.rnn_init_method == 'first_input'
                               else 'rnn_initial_state/weight'))
        w.memory_kernel = g(D + 'memory_layer/kernel')
        w.value_kernel = g(D + 'value_layer/kernel')
        w.query_kernel = g(att + 'query_layer/kernel')
        w.attention_v = g(att + 'attention_v')
        w.ln_gamma = g(att + 'LN_tanh/gamma')
        w.ln_beta = g(att + 'LN_tanh/beta')
        if (D + 'softmax_temperature') in dev:
            dev[D + 'softmax_temperature'] = dev[D + 'softmax_temperature'].reshape(1).contiguous()
        w.temperature = g(D + 'softmax_temperature')
        w.a_layer = g(D + 'a_layer/kernel')
        w.out_kernel = g(D + 'output_projection/kernel')
        w.out_bias = g(D + 'output_projection/bias')
        w.embedding_map = g(D + 'embedding_map')
        w.enc_ln_gamma = g(ENC + 'LN_tanh/gamma')
        w.enc_ln_beta = g(ENC + 'LN_tanh/beta')
        w.enc_embed_weight = g(ENC + 'im_embed/weight')
        have_cnn = with_cnn and (CNN + 'Conv2d_1a_7x7/weights') in dev
        if have_cnn:
            for i, (scope, _k, _s, _ci, _co) in enumerate(wts.cnn_conv_list()):
                w.conv_w[i] = g(CNN + scope + '/weights')
                w.bn_beta[i] = g(CNN + scope + '/BatchNorm/beta')
                w.bn_mean[i] = g(CNN + scope + '/BatchNorm/moving_mean')
                w.bn_var[i] = g(CNN + scope + '/BatchNorm/moving_variance')
        n = C.c_size_t()
        self._check(self.lib.comic_packed_bytes(self._h, C.byref(n)))
        self._packed = torch.empty(n.value, dtype=torch.uint8, device=self.device)
        self._check(self.lib.comic_bind_weights(self._h, C.byref(w), int(have_cnn), _ptr(self._packed),
                                                n.value, self.stream()))
        self.bound_cnn = bool(have_cnn)
        self._wstruct = w

    # -- E1/E2 ----------------------------------------------------------------
    def encode(self, images, want_mixed5c=False):
        """images [B,224,224,3] fp32 NHWC on device -> (im_embed [B,1024], fm [B,196,C])."""
        torch = self.torch
        images = images.contiguous()
        if images.dim() != 4 or tuple(images.shape[1:]) != (224, 224, 3):
            raise ValueError('images must be [B,224,224,3] NHWC, got %s' % (tuple(images.shape),))
        B = images.shape[0]
        fm = self.f32(B, self.dims.M, self.dims.C)
        emb = self.f32(B, self.dims.E)
        m5c = self.f32(B, 7, 7, 1024) if want_mixed5c else None
        ws = self._workspace(0, B, 1, 1)
        self._check(self.lib.comic_encode_fwd(self._h, _ptr(images), B, _ptr(fm), _ptr(emb), _ptr(m5c),
                                              _ptr(ws), ws.numel(), self.stream()))
        return (emb, fm, m5c) if want_mixed5c else (emb, fm)

    def preprocess_eval(self, images_u8, out_hw=(224, 224)):
        """inception_preprocessing_radix.preprocess_image(is_training=False): uint8 [B,H,W,3] on device ->
        fp32 [B,224,224,3] in [-1,1] (resize 256 bilinear, central crop, (x - 0.5) * 2)."""
        torch = self.torch
        images_u8 = images_u8.contiguous()
        if images_u8.dtype != torch.uint8 or images_u8.dim() != 4 or images_u8.shape[3] != 3:
            raise ValueError('images must be uint8 [B,H,W,3], got %s %s' % (images_u8.dtype, tuple(images_u8.shape)))
        B, H, W = (int(v) for v in images_u8.shape[:3])
        out = self.f32(B, int(out_hw[0]), int(out_hw[1]), 3)
        self._check(self.lib.comic_preprocess_eval(self._h, _ptr(images_u8), B, H, W, int(out_hw[0]), int(out_hw[1]),
                                                   _ptr(out), self.stream()))
        return out

    def preprocess_train(self, images_u8, crop_yx, flip=None, out_hw=(224, 224)):
        """inception_preprocessing_radix.preprocess_image(is_training=True): uint8 [B,H,W,3] on device -> resize 256
        bilinear -> left-right flip where flip[b] -> crop at crop_yx[b] = (y0, x0) -> (x - 0.5) * 2.  `crop_yx` int32
        [B,2] and `flip` uint8 [B] are the caller's random draws (see train.random_crop_flip)."""
        torch = self.torch
        images_u8 = images_u8.contiguous()
        if images_u8.dtype != torch.uint8 or images_u8.dim() != 4 or images_u8.shape[3] != 3:
            raise ValueError('images must be uint8 [B,H,W,3], got %s %s' % (images_u8.dtype, tuple(images_u8.shape)))
        B, H, W = (int(v) for v in images_u8.shape[:3])
        crop = torch.as_tensor(crop_yx).to(device=self.device, dtype=torch.int32).contiguous()
        if tuple(crop.shape) != (B, 2):
            raise ValueError('crop_yx must be [B, 2]')
        if int(crop.min()) < 0 or int(crop[:, 0].max()) > 256 - out_hw[0] or int(crop[:, 1].max()) > 256 - out_hw[1]:
            raise ValueError('crop offsets must lie in [0, 256 - out]')
        fl = None if flip is None else torch.as_tensor(flip).to(device=self.device, dtype=torch.uint8).contiguous()
        out = self.f32(B, int(out_hw[0]), int(out_hw[1]), 3)
        self._check(self.lib.comic_preprocess_train(self._h, _ptr(images_u8), B, H, W, int(out_hw[0]), int(out_hw[1]),
                                                    _ptr(crop), _ptr(fl), _ptr(out), self.stream()))
        return out

    # -- D0 -------------------------------------------------------------------
    def project_fm(self, fm):
        B = fm.shape[0]
        d = self.dims
        keys = self.f32(B, d.M, d.R)
        values = self.f32(B, d.M, d.R) if d.fm_projection == 'independent' else None
        self._check(self.lib.comic_project_fm(self._h, _ptr(fm.contiguous()), B, _ptr(keys), _ptr(values),
                                              self.stream()))
        if d.fm_projection is None:
            values = fm
        elif d.fm_projection == 'tied':
            values = keys
        return keys, values

    # -- D1 -------------------------------------------------------------------
    def rnn_init(self, im_embed, in_mask=None, in_keep=1.0):
        """-> (c0, h0) [B, R]; c0 is None for the GRU cell (its state is h only)."""
        B = im_embed.shape[0]
        c0, h0 = (None if self.gru else self.f32(B, self.dims.R)), self.f32(B, self.dims.R)
        ws = self._workspace(4, B, 1, 1)
        self._check(self.lib.comic_rnn_init(self._h, _ptr(im_embed.contiguous()), B, _ptr(c0), _ptr(h0),
                                            _ptr(in_mask), float(in_keep), _ptr(ws), ws.numel(), self.stream()))
        return c0, h0

    # -- D3-D7 (unit) ---------------------------------------------------------
    def decode_step(self, keys, values, B, k, tokens, c_in, h_in, ctx_in, in_mask=None, out_mask=None,
                    att_mask=None, keeps=(1.0, 1.0, 1.0)):
        d = self.dims
        N = B * k
        c_out, h_out = (None if self.gru else self.f32(N, d.R)), self.f32(N, d.R)
        ctx_out = self.f32(N, d.A)
        align = self.f32(N, d.H * d.M)
        logits = self.f32(N, d.V)
        ws = self._workspace(3, B, k, 1)
        vals = None if d.fm_projection == 'tied' else values
        self._check(self.lib.comic_decode_step(
            self._h, _ptr(keys), _ptr(vals), B, k, _ptr(tokens), _ptr(c_in), _ptr(h_in), _ptr(ctx_in),
            _ptr(c_out), _ptr(h_out), _ptr(ctx_out), _ptr(align), _ptr(logits),
            _ptr(in_mask), _ptr(out_mask), _ptr(att_mask), float(keeps[0]), float(keeps[1]), float(keeps[2]),
            _ptr(ws), ws.numel(), self.stream()))
        return dict(c=c_out, h=h_out, attention=ctx_out, alignments=align, logits=logits)

    # -- B2 -------------------------------------------------------------------
    def decode_greedy(self, keys, values, c0, h0, max_it, want_logits=True, want_attn=True):
        torch = self.torch
        d = self.dims
        B = h0.shape[0]
        ids = torch.empty((max(max_it, 1), B), dtype=torch.int32, device=self.device)
        logits = self.f32(max(max_it, 1), B, d.V) if want_logits else None
        attn = self.f32(B, d.H, max(max_it, 1), d.M) if want_attn else None
        T = torch.zeros(1, dtype=torch.int32, device=self.device)
        ws = self._workspace(1, B, 1, max(max_it, 1))
        vals = None if d.fm_projection == 'tied' else values
        self._check(self.lib.comic_decode_greedy(self._h, _ptr(keys), _ptr(vals), _ptr(c0), _ptr(h0), B, max_it,
                                                 _ptr(ids), _ptr(logits), _ptr(attn), _ptr(T), _ptr(ws),
                                                 ws.numel(), self.stream()))
        return dict(ids=ids, logits=logits, attn=attn, T=T)

    # -- B1/B3 ----------------------------------------------------------------
    def decode_beam(self, keys, values, c0, h0, beam, lpw, max_it, want_attn=True):
        torch = self.torch
        d = self.dims
        B = h0.shape[0]
        Tm = max(max_it, 1)
        i32 = dict(dtype=torch.int32, device=self.device)
        pred = torch.empty((Tm, B, beam), **i32)
        step_ids = torch.empty((Tm, B, beam), **i32)
        parents = torch.empty((Tm, B, beam), **i32)
        scores = self.f32(Tm, B, beam)
        lengths = torch.empty((B, beam), dtype=torch.int64, device=self.device)
        attn = self.f32(B, d.H, Tm, d.M) if want_attn else None
        T = torch.zeros(1, dtype=torch.int32, device=self.device)
        ws = self._workspace(2, B, beam, Tm)
        vals = None if d.fm_projection == 'tied' else values
        self._check(self.lib.comic_decode_beam(self._h, _ptr(keys), _ptr(vals), _ptr(c0), _ptr(h0), B, beam,
                                               float(lpw), max_it, _ptr(pred), _ptr(step_ids), _ptr(parents),
                                               _ptr(scores), _ptr(lengths), _ptr(attn), _ptr(T), _ptr(ws),
                                               ws.numel(), self.stream()))
        return dict(predicted_ids=pred, step_ids=step_ids, parent_ids=parents, scores=scores,
                    lengths=lengths, attn=attn, T=T)

    # -- K10 / K11 / GEMM (unit) ----------------------------------------------
    def beam_step(self, logits, log_probs, finished, lengths, eos, lpw):
        torch = self.torch
        B, k, V = logits.shape
        logits = logits.contiguous()
        scores = self.f32(B, k)
        word = torch.empty((B, k), dtype=torch.int32, device=self.device)
        parent = torch.empty((B, k), dtype=torch.int32, device=self.device)
        self._check(self.lib.comic_beam_step(self._h, _ptr(logits), V, B, k, V, int(eos), float(lpw),
                                             _ptr(log_probs), _ptr(finished), _ptr(lengths), _ptr(scores),
                                             _ptr(word), _ptr(parent), self.stream()))
        return scores, word, parent

    def gather_tree(self, step_ids, parent_ids, max_seq_len, end_token):
        T, B, k = step_ids.shape
        out = self.torch.empty_like(step_ids)
        self._check(self.lib.comic_gather_tree(self._h, _ptr(step_ids.contiguous()), _ptr(parent_ids.contiguous()),
                                               _ptr(max_seq_len.contiguous()), T, B, k, int(end_token), _ptr(out),
                                               self.stream()))
        return out

    def gemm(self, A, Bm, bias=None):
        M, K = A.shape
        N = Bm.shape[1]
        out = self.f32(M, N)
        ws = self._workspace(5, N, K, 1)
        self._check(self.lib.comic_gemm_f32(self._h, _ptr(A), A.stride(0), _ptr(Bm), Bm.stride(0), _ptr(bias),
                                            _ptr(out), N, M, N, K, _ptr(ws), ws.numel(), self.stream()))
        return out

    def set_precision(self, mode):
        """'f32' (FFMA everywhere) or 'tf32x3' (tcgen05, fp32-equivalent; default)."""
        self._check(self.lib.comic_set_precision(self._h, {'f32': 0, 'tf32x3': 1, 'split': 1, 'fast': 2}[mode]))

    def set_option(self, name, value):
        self._check(self.lib.comic_set_option(self._h, {'fused_attn_min_images': 0, 'enc_chunk_stem': 1, 'enc_chunk_28': 2, 'enc_chunk_14': 3, 'persistent_max_rows': 4, 'persistent_trace': 5, 'stem_s2d': 9, 'tc_min_rows': 11, 'attn2': 12, 'tma_a': 15, 'persistent_watchdog_ms': 18, 'tc_splitk': 19}[name], int(value)))

    def decode_trace(self, max_steps=256):
        """Per-phase clock stamps of the last persistent decode call: int64 array [steps, 2, 16]."""
        import numpy as np
        out = np.zeros((max_steps, 2, 16), np.int64)
        n = C.c_int()
        self._check(self.lib.comic_decode_trace(self._h, out.ctypes.data_as(C.c_void_p), max_steps, C.byref(n),
                                                self.stream()))
        return out[:n.value]

    def profile_enable(self, tags):
        mask = 0
        for t in tags:
            mask |= 1 << KERNEL_TAGS.index(t)
        self._profiling = mask != 0
        self._check(self.lib.comic_profile_enable(self._h, mask))

    # -- CUDA graphs -------------------------------------------------------------
    def graphed(self, key, fn, *inputs):
        """fn(*inputs) through a CUDA graph: the inference path is ~370 dependent launches per batch (60 decode steps x 5
        kernels), and a replayed graph launches each node ~2 us sooner than the stream does.  The first call of a
        signature runs eagerly (it sizes the workspaces and does the one-time kernel attribute calls), the second captures,
        later ones replay.  The signature is the inputs' addresses / shapes / dtypes, the weight binding and the workspace
        addresses; when any of them changes the graph is dropped and rebuilt.  The returned tensors are the graph's own
        output buffers: consume them before the next call with the same key.  COMIC_B200_INFER_GRAPH=0 disables it; so
        does an active kernel-class profile (its events cannot be captured)."""
        torch = self.torch
        if not getattr(self, 'infer_graph', True) or getattr(self, '_profiling', False):
            return fn(*inputs)
        if not hasattr(self, '_graphs'):
            self._graphs, self.replayed_launches = {}, 0
            self.infer_graph = os.environ.get('COMIC_B200_INFER_GRAPH', '1') != '0'
            if not self.infer_graph:
                return fn(*inputs)

        def signature():
            return (tuple((t.data_ptr(), tuple(t.shape), t.dtype) for t in inputs), getattr(self, '_bind_generation', 0),
                    tuple(sorted((k, v.data_ptr()) for k, v in self._ws.items() if hasattr(v, 'data_ptr'))))
        ent = self._graphs.get(key)
        if ent is not None and ent['sig'] != signature():
            ent = None
        if ent is None:
            out = fn(*inputs)
            self._graphs[key] = {'sig': signature(), 'graph': None}
            return out
        if ent['graph'] is None:
            torch.cuda.synchronize(self.device)
            g = torch.cuda.CUDAGraph()
            n0 = self.launch_count()
            try:
                with torch.cuda.graph(g):
                    ent['out'] = fn(*inputs)
            except Exception:
                self.infer_graph = False
                torch.cuda.synchronize(self.device)
                return fn(*inputs)
            ent['graph'], ent['launches'] = g, self.launch_count() - n0
            if ent['sig'] != signature():                  # the capture itself allocated a workspace: not replayable as keyed
                self._graphs.pop(key)
                return fn(*inputs)
        ent['graph'].replay()
        self.replayed_launches += ent['launches']
        return ent['out']

    def profile_read(self, tag):
        ms, n = C.c_double(), C.c_int64()
        self._check(self.lib.comic_profile_read(self._h, KERNEL_TAGS.index(tag), C.byref(ms), C.byref(n)))
        return ms.value, n.value

    # -- training (T1-T4) ------------------------------------------------------
    def variable_to_grad_field(self):
        """TF variable name -> field of comic_decoder_grads_t."""
        c = self.c
        D = wts.DEC
        att = D + 'multi_add_attention/'
        cs = wts.cell_scope(c)
        if self.gru:     # gates/{kernel, bias} travel in the LSTM fields, as at binding
            cell = {cs + 'gates/kernel': 'lstm_kernel', cs + 'gates/bias': 'lstm_bias',
                    cs + 'candidate/kernel': 'cand_kernel', cs + 'candidate/bias': 'cand_bias'}
        else:
            cell = {cs + 'kernel': 'lstm_kernel', cs + 'bias': 'lstm_bias'}
        m = {D + 'rnn_init_input/projection/weight': 'init_weight', D + 'rnn_initial_state/weight': 'init_weight',
             D + 'memory_layer/kernel': 'memory_kernel', D + 'value_layer/kernel': 'value_kernel',
             att + 'query_layer/kernel': 'query_kernel', att + 'attention_v': 'attention_v',
             att + 'LN_tanh/gamma': 'ln_gamma', att + 'LN_tanh/beta': 'ln_beta',
             D + 'softmax_temperature': 'temperature', D + 'output_projection/kernel': 'out_kernel',
             D + 'output_projection/bias': 'out_bias', D + 'embedding_map': 'embedding_map',
             D + 'a_layer/kernel': 'a_layer'}
        m.update(cell)
        return m

    def dropout_masks(self, shape, keep, seed, stream_id):
        out = self.f32(*shape)
        self._check(self.lib.comic_dropout_masks(self._h, _ptr(out), out.numel(), float(keep), int(seed),
                                                 int(stream_id), self.stream()))
        return out

    def train_fwd_bwd(self, fm, im_embed, inputs_tm, targets_tm, coef_tm, lens, T_run, grad_views, masks=None,
                      keeps=(1.0, 1.0, 1.0), map_loss_scale=1.0, want_logits=False, want_attn=False):
        """grad_views: dict grad-field -> device tensor view receiving that gradient."""
        torch = self.torch
        d = self.dims
        T, B = inputs_tm.shape
        loss = torch.zeros(4, dtype=torch.float32, device=self.device)
        logits = self.f32(B, T, d.V) if want_logits else None
        attn = self.f32(B, d.H, T_run, d.M) if want_attn else None
        g = None
        if grad_views is not None:                     # None: forward only (evaluation perplexity)
            g = ComicDecoderGrads()
            for f in GRAD_FIELDS:
                t = grad_views.get(f)
                setattr(g, f, None if t is None else C.c_void_p(t.data_ptr()))
        mk = None
        if masks is not None:
            mk = ComicTrainMasks()
            for f in ('init_in', 'inp', 'out', 'att'):
                t = masks.get(f)
                setattr(mk, f, None if t is None else C.c_void_p(t.data_ptr()))
            mk.in_keep, mk.out_keep, mk.att_keep = [float(x) for x in keeps]
        n = C.c_size_t()
        self._check(self.lib.comic_train_workspace_bytes(self._h, B, T_run, C.byref(n)))
        ws = self._ws.get('train')
        if ws is None or ws.numel() < n.value:
            ws = self._ws['train'] = torch.empty(n.value, dtype=torch.uint8, device=self.device)
        self._check(self.lib.comic_train_fwd_bwd(
            self._h, _ptr(fm), _ptr(im_embed), B, _ptr(inputs_tm), _ptr(targets_tm), _ptr(coef_tm), _ptr(lens), T,
            int(T_run), None if mk is None else C.byref(mk), float(map_loss_scale), _ptr(loss), _ptr(logits),
            _ptr(attn), None if g is None else C.byref(g), _ptr(ws), ws.numel(), self.stream()))
        return loss, logits, attn

    # -- cnn_finetune (encoder forward-with-tape + backward) ---------------------
    def encode_train(self, images):
        """Forward that keeps every activation: -> (im_embed [B,1024], fm [B,196,C]); the tape stays
        in this engine until `encode_bwd`."""
        torch = self.torch
        images = images.contiguous()
        if images.dim() != 4 or tuple(images.shape[1:]) != (224, 224, 3):
            raise ValueError('images must be [B,224,224,3] NHWC, got %s' % (tuple(images.shape),))
        B = images.shape[0]
        nt, nw = C.c_size_t(), C.c_size_t()
        self._check(self.lib.comic_encode_train_bytes(self._h, B, C.byref(nt), C.byref(nw)))
        for key, n in (('enc_tape', nt.value), ('enc_train_ws', nw.value)):
            if self._ws.get(key) is None or self._ws[key].numel() < n:
                self._ws[key] = torch.empty(n, dtype=torch.uint8, device=self.device)
        tape, ws = self._ws['enc_tape'], self._ws['enc_train_ws']
        fm = self.f32(B, self.dims.M, self.dims.C)
        emb = self.f32(B, self.dims.E)
        self._check(self.lib.comic_encode_train_fwd(self._h, _ptr(images), B, _ptr(fm), _ptr(emb), _ptr(tape),
                                                    tape.numel(), _ptr(ws), ws.numel(), self.stream()))
        return emb, fm

    def train_encoder_grads(self, B, T_run):
        """d loss / d (fm, im_embed) of the `train_fwd_bwd` call that just ran (same B, T_run)."""
        dfm = self.f32(B, self.dims.M, self.dims.C)
        demb = self.f32(B, self.dims.E)
        ws = self._ws['train']
        self._check(self.lib.comic_train_encoder_grads(self._h, B, int(T_run), _ptr(dfm), _ptr(demb), _ptr(ws),
                                                       ws.numel(), self.stream()))
        return dfm, demb

    def legacy_head_bwd(self, mixed5c, d_im_embed, d_gamma, d_beta, d_weight):
        """--legacy, train_mode=decoder: gradients of Model/encoder/LN_tanh/{gamma, beta} and Model/encoder/im_embed/weight
        from Mixed_5c [B,7,7,1024] and d loss / d im_embed [B,1024] (comic_legacy_head_bwd)."""
        B = mixed5c.shape[0]
        n = C.c_size_t()
        self._check(self.lib.comic_legacy_head_bwd_bytes(self._h, B, C.byref(n)))
        ws = self._ws.get('legacy_head')
        if ws is None or ws.numel() < n.value:
            ws = self._ws['legacy_head'] = self.torch.empty(n.value, dtype=self.torch.uint8, device=self.device)
        self._check(self.lib.comic_legacy_head_bwd(self._h, _ptr(mixed5c.contiguous()), B, _ptr(d_im_embed.contiguous()),
                                                   _ptr(d_gamma), _ptr(d_beta), _ptr(d_weight), _ptr(ws), ws.numel(),
                                                   self.stream()))

    def encode_bwd(self, images, dfm, dim_embed, conv_grads, beta_grads):
        """Backward of the last `encode_train`: conv_grads / beta_grads are lists of 57 device tensors
        (views into the flat gradient buffer) in comic_conv_table() order."""
        B = images.shape[0]
        g = ComicCnnGrads()
        for i in range(NUM_CONVS):
            g.conv_w[i] = C.c_void_p(conv_grads[i].data_ptr())
            g.bn_beta[i] = C.c_void_p(beta_grads[i].data_ptr())
        tape, ws = self._ws['enc_tape'], self._ws['enc_train_ws']
        self._check(self.lib.comic_encode_bwd(self._h, _ptr(images.contiguous()), B, _ptr(dfm.contiguous()),
                                              _ptr(dim_embed.contiguous()), _ptr(tape), tape.numel(), C.byref(g),
                                              _ptr(ws), ws.numel(), self.stream()))

    def refresh_packed_cnn(self):
        self._bind_generation = getattr(self, '_bind_generation', 0) + 1      # see refresh_packed
        self._check(self.lib.comic_refresh_packed_cnn(self._h, _ptr(self._packed), self._packed.numel(),
                                                      self.stream()))

    def l2_regularise(self, params, grads, decay, reg_out):
        ws = self._ws.get('l2')
        if ws is None:
            ws = self._ws['l2'] = self.torch.empty(8192, dtype=self.torch.uint8, device=self.device)
        self._check(self.lib.comic_l2_regularise(self._h, _ptr(params), _ptr(grads), params.numel(), float(decay),
                                                 _ptr(reg_out), _ptr(ws), ws.numel(), self.stream()))

    def adam_step(self, params, grads, m, v, lr, step, beta1=0.9, beta2=0.999, eps=1e-2, grad_scale=1.0):
        self._check(self.lib.comic_adam_step(self._h, _ptr(params), _ptr(grads), _ptr(m), _ptr(v), params.numel(),
                                             float(lr), float(beta1), float(beta2), float(eps), int(step),
                                             float(grad_scale), self.stream()))

    def momentum_step(self, params, grads, accum, lr, momentum=0.9, grad_scale=1.0):
        self._check(self.lib.comic_momentum_step(self._h, _ptr(params), _ptr(grads), _ptr(accum), params.numel(), float(lr),
                                                 float(momentum), float(grad_scale), self.stream()))

    def clip_by_norm(self, grads, offsets, sizes, max_norm):
        """offsets / sizes: int64 device tensors, one entry per variable of the flat gradient buffer."""
        self._check(self.lib.comic_clip_by_norm(self._h, _ptr(grads), _ptr(offsets), _ptr(sizes), int(offsets.numel()),
                                                float(max_norm), self.stream()))

    def refresh_packed(self):
        # the weights changed in place: captured inference graphs (Engine.graphed) are dropped, so that their next eager call
        # re-validates the streaming attention kernel's score bound on the host
        self._bind_generation = getattr(self, '_bind_generation', 0) + 1
        self._check(self.lib.comic_refresh_packed(self._h, _ptr(self._packed), self._packed.numel(), self.stream()))

    def launch_count(self):
        """Kernel launches so far: the library's host-side count plus the kernels executed through graph replays."""
        n = C.c_int64()
        self._check(self.lib.comic_launch_count(self._h, C.byref(n)))
        return n.value + getattr(self, 'replayed_launches', 0)

"""Training on the CUDA engine: `train_mode` = decoder | scst (frozen CNN) | cnn_finetune
(InceptionV1 conv kernels + BN betas train too; src/train.py:241-250).

Mirrors the pieces of the reference that surround one `sess.run(train_op)`:
  ModelBase._process_inputs        src/model_base.py:501-528  (inputs / targets / masks)
  ModelBase._train_caption_model   src/model_base.py:325-405  (loss terms, Adam, no clipping)
  ModelBase._create_cosine_lr      src/model_base.py:809-820
  train_fn / train_fn_scst loops   src/train_fn.py:26-147, 150-307 (one step each)
The arithmetic runs in libcomic_b200.so (csrc/train.cu); this module only prepares the
int32 / fp32 host arrays, owns the flat parameter / gradient / Adam buffers and calls
`torch.distributed.all_reduce` on the flat gradient buffer when a process group exists
(one process per GPU, NCCL over NVLink; the reference is single-GPU).
"""
from __future__ import annotations

import math

import os

import numpy as np

from . import weights as wts
from .engine import Engine, pack_images


def process_inputs(captions, token_type):
    """_process_inputs (src/model_base.py:501-528): captions [B,L] int32 (PAD = -1) ->
    (inputs [B,L-1], targets [B,L-1], masks [B,L-1] f32, lens [B] i32)."""
    cap = np.asarray(captions, np.int32)
    masks = np.sign((cap[:, 1:] + 1).astype(np.float32))
    lens = masks.sum(axis=1).astype(np.int32)
    clipped = np.maximum(cap, 0)
    inputs = clipped[:, :-1] if token_type == 'word' else cap[:, :-1]
    return inputs, clipped[:, 1:], masks, lens


def loss_coefficients(masks, rewards=None):
    """Per-token weight of the cross-entropy (src/model_base.py:337-347): XE mode
    mask / (sum(mask) + 1e-12); SCST mode reward_b / B * mask / (sum_t mask + 1e-12)."""
    m = masks.astype(np.float32)
    if rewards is None:
        return m / (m.sum(dtype=np.float32) + np.float32(1e-12))
    r = np.asarray(rewards, np.float32)[:, None]
    return (r / np.float32(m.shape[0])) * m / (m.sum(axis=1, keepdims=True) + np.float32(1e-12))


def cosine_lr(step, max_step, lr_start, lr_end):
    """_create_cosine_lr (src/model_base.py:809-820)."""
    s = min(1.0, float(step) / float(max_step))
    return (lr_start - lr_end) * (1.0 + math.cos(s * math.pi)) / 2.0 + lr_end


def legacy_lr_reduce(config, epoch, learning_rate):
    """_lr_reduce_check (src/train_fn.py:310-317): the legacy models halve the rate every
    `lr_reduce_every_n_epochs` epochs, floored at `lr_end`."""
    if learning_rate > config.lr_end and epoch % config.lr_reduce_every_n_epochs == 0:
        learning_rate /= 2
        if learning_rate < config.lr_end:
            learning_rate = config.lr_end
    return learning_rate


def random_crop_flip(batch, out_hw=(224, 224), rng=None, resized=256):
    """The two random draws of `preprocess_for_train` (inception_preprocessing_radix.py:182-185): a fair coin per image
    for tf.image.random_flip_left_right and a uniform top-left corner for tf.random_crop of the 256 x 256 image.
    Returns (crop_yx int32 [B,2], flip uint8 [B]) for Engine.preprocess_train."""
    rng = rng or np.random.default_rng()
    crop = np.stack([rng.integers(0, resized - out_hw[0] + 1, size=batch),
                     rng.integers(0, resized - out_hw[1] + 1, size=batch)], axis=1).astype(np.int32)
    flip = (rng.random(batch) < 0.5).astype(np.uint8)
    return crop, flip


class Trainer(object):
    """Flat fp32 parameter / gradient / Adam-slot buffers over the decoder variables, one
    engine handle, one optimiser step per `step()`."""

    def __init__(self, config, weights, engine=None, with_cnn=True):
        self.c = c = config
        if c.train_mode not in ('decoder', 'scst', 'cnn_finetune'):
            raise ValueError("train_mode must be decoder | cnn_finetune | scst, got '%s'" % c.train_mode)
        self.finetune_cnn = c.train_mode == 'cnn_finetune'
        if self.finetune_cnn and not with_cnn:
            raise ValueError('train_mode=cnn_finetune needs the CNN weights')
        # options the reference accepts but this path does not build: refuse instead of silently training differently
        if getattr(c, 'optimiser', 'adam') not in ('adam', 'sgd'):
            raise ValueError('Unknown optimiser.')                                 # src/model_base.py:881-882
        self.engine = eng = engine or Engine(c)
        torch = self.torch = eng.torch
        self.shapes = dict(wts.decoder_shapes(c))
        # --legacy: the image-embedding head (LN_tanh + im_embed, src/model_base.py:80-91) sits outside Model/encoder/cnn, so it
        # trains with the decoder; the reference only trains legacy models in train_mode=decoder (src/train.py:242, 253)
        self.legacy_head = bool(getattr(c, 'legacy', False))
        if self.legacy_head:
            if c.train_mode != 'decoder':
                raise NotImplementedError("--legacy models train in train_mode=decoder only (src/train.py:242, 253)")
            self.shapes.update(wts.encoder_head_shapes(c))
        self.n_decoder_vars = len(self.shapes)
        if self.finetune_cnn:
            # trainable CNN variables: conv kernels + BN betas (BN runs with is_training=False,
            # src/model_base.py:71-77, so the moving statistics are constants)
            for scope, k, _s, cin, cout in wts.cnn_conv_list():
                self.shapes[wts.CNN + scope + '/weights'] = (k, k, cin, cout)
                self.shapes[wts.CNN + scope + '/BatchNorm/beta'] = (cout,)
        self.offsets, off = {}, 0
        for name, shp in self.shapes.items():
            n = int(np.prod(shp)) if len(shp) else 1
            self.offsets[name] = (off, n, shp)
            off += (n + 3) // 4 * 4                     # 16-byte aligned views
            if len(self.offsets) == self.n_decoder_vars:
                self.n_decoder_flat = off
        self.n_flat = off
        self.params = torch.zeros(off, dtype=torch.float32, device=eng.device)
        self.grads = torch.zeros(off, dtype=torch.float32, device=eng.device)
        self.adam_m = torch.zeros(off, dtype=torch.float32, device=eng.device)
        self.adam_v = torch.zeros(off, dtype=torch.float32, device=eng.device)
        W = dict(weights)
        for name, (o, n, shp) in self.offsets.items():
            self.params[o:o + n].copy_(torch.as_tensor(np.asarray(W[name], np.float32).reshape(-1)))
            W[name] = self.params[o:o + n].view(shp if len(shp) else (1,))
        eng.bind_weights(W, with_cnn=with_cnn)
        self._bound, self._with_cnn = W, with_cnn
        # The teacher-forced forward + backward is ~1,100 small launches at batch 32 (25 per time step x 41 steps): replayed
        # as ONE CUDA graph per (batch, length) shape after two eager calls of that shape.  COMIC_B200_TRAIN_GRAPH=0 or
        # `trainer.cuda_graph = False` keeps every step eager.
        self.cuda_graph = os.environ.get('COMIC_B200_TRAIN_GRAPH', '1') != '0'
        self._graphs = {}
        self.replayed_launches = 0       # kernel launches executed through graph replays (the engine counts host launches)
        fields = eng.variable_to_grad_field()
        self.grad_views = {}
        for name, (o, n, shp) in self.offsets.items():
            if name in fields:
                self.grad_views[fields[name]] = self.grads[o:o + n]
        if self.finetune_cnn:
            convs = wts.cnn_conv_list()
            self.cnn_grad_w = [self.gradient(wts.CNN + sc + '/weights') for sc, *_ in convs]
            self.cnn_grad_b = [self.gradient(wts.CNN + sc + '/BatchNorm/beta') for sc, *_ in convs]
        self.global_step = 0
        # crop / flip draws of `cnn_input_augment` for raw-pixel batches when a step gives no seed
        self._augment_rng = np.random.default_rng(int(getattr(c, 'rand_seed', 48964896)))
        self.reg = torch.zeros(1, dtype=torch.float32, device=eng.device)
        # slim clip_gradient_norms: per-variable slices of the flat gradient buffer (device tables for comic_clip_by_norm)
        self.clip_norm = float(getattr(c, 'clip_gradient_norm', 0) or 0)
        self._var_off = torch.tensor([o for o, n, _ in self.offsets.values()], dtype=torch.int64, device=eng.device)
        self._var_len = torch.tensor([n for o, n, _ in self.offsets.values()], dtype=torch.int64, device=eng.device)

    # -- views ------------------------------------------------------------------
    def variable(self, name):
        o, n, shp = self.offsets[name]
        return self.params[o:o + n].view(shp if len(shp) else (1,))

    def gradient(self, name):
        o, n, shp = self.offsets[name]
        return self.grads[o:o + n].view(shp if len(shp) else (1,))

    def dropout_seed(self, seed=None):
        """Seed of this step's dropout masks: explicit, or derived from `config.rand_seed` and the global step so that
        the default training call is regularised like the reference's (DropoutWrapper keep 0.65 in / out,
        attention-map keep 0.9: src/model_base.py:636-648, common/ops_rnn.py:696-701)."""
        if seed is not None:
            return int(seed)
        return (int(getattr(self.c, 'rand_seed', 48964896)) * 1000003 + self.global_step) & 0x7fffffff

    def variables_numpy(self):
        """The trainable variables (views of the flat buffer) plus the bound constants, as host arrays."""
        W = {k: np.asarray(v) if not hasattr(v, 'cpu') else v.detach().cpu().numpy() for k, v in self._bound.items()}
        for name in self.offsets:
            W[name] = self.variable(name).detach().cpu().numpy().reshape(self.offsets[name][2])
        return W

    def load_variables(self, weights, extra=None):
        """Overwrite the flat parameter buffer (and, when resuming from a TF checkpoint, the Adam slots `<var>/Adam`,
        `<var>/Adam_1` and `global_step`) from a W-table; re-binds and re-packs the engine."""
        torch, eng = self.torch, self.engine
        W = dict(self._bound)
        W.update(weights)
        for name, (o, n, shp) in self.offsets.items():
            self.params[o:o + n].copy_(torch.as_tensor(np.asarray(W[name], np.float32).reshape(-1)))
            W[name] = self.params[o:o + n].view(shp if len(shp) else (1,))
            if extra:
                slots = ((('/Momentum', self.adam_m),) if getattr(self.c, 'optimiser', 'adam') == 'sgd'
                         else (('/Adam', self.adam_m), ('/Adam_1', self.adam_v)))
                for slot, buf in slots:
                    if name + slot in extra:
                        buf[o:o + n].copy_(torch.as_tensor(np.asarray(extra[name + slot], np.float32).reshape(-1)))
        if extra and 'global_step' in extra:
            self.global_step = int(np.asarray(extra['global_step']))
        self._bound = W
        eng.bind_weights(W, with_cnn=self._with_cnn)
        self._graphs.clear()                             # captured steps hold the previous binding's device pointers

    def make_masks(self, B, T_run, seed):
        """Seeded Philox dropout masks (DropoutWrapper in/out, attention-map dropout)."""
        c, d, eng = self.c, self.engine.dims, self.engine
        keeps = (1.0 - c.dropout_rnn_in, 1.0 - c.dropout_rnn_out, c.attn_keep_prob)
        XA = d.W + d.A
        if getattr(c, 'rnn_recurr_dropout', False):
            # DropoutWrapper(variational_recurrent=True) (src/model_base.py:641-647; TF r1.9 rnn_cell_impl.py builds its
            # noise with a leading dimension of 1: "the same dropout mask for all batch elements"): ONE input mask [1, W+A]
            # and ONE output mask [1, R] per step of the optimiser, shared by every row and every time step -- and by the
            # rnn-init call, which runs through the same wrapped cell.  state_keep_prob stays 1.
            mi = eng.dropout_masks((1, XA), keeps[0], seed, 1)
            mo = eng.dropout_masks((1, d.R), keeps[1], seed, 2)
            masks = dict(init_in=mi.expand(B, XA).contiguous(), inp=mi.expand(T_run, B, XA).contiguous(),
                         out=mo.expand(T_run, B, d.R).contiguous())
        else:
            masks = dict(init_in=eng.dropout_masks((B, XA), keeps[0], seed, 0),
                         inp=eng.dropout_masks((T_run, B, XA), keeps[0], seed, 1),
                         out=eng.dropout_masks((T_run, B, d.R), keeps[1], seed, 2))
        if keeps[2] < 1.0:
            masks['att'] = eng.dropout_masks((T_run, B, d.H * d.M), keeps[2], seed, 3)
        return masks, keeps

    # -- one fwd + bwd (+ optimiser) ---------------------------------------------
    def forward_backward(self, fm, im_embed, captions, rewards=None, masks=None, keeps=(1.0, 1.0, 1.0),
                         want_logits=False, want_attn=False, images=None, forward_only=False, mixed5c=None):
        """captions [B,L] int32 host array.  Returns dict(loss=[total, xe, map, reg] device tensor, ...);
        gradients land in self.grads.  forward_only: cross-entropy only (loss[1]); no backward, no L2 term, and
        self.grads is left untouched (the evaluation graph of train_fn._run_eval_loop)."""
        c, eng, torch = self.c, self.engine, self.torch
        inputs, targets, wmask, lens = process_inputs(captions, c.token_type)
        coef = loss_coefficients(wmask, rewards)
        T_run = int(lens.max())
        dev = eng.device
        to = lambda a, dt: torch.as_tensor(np.ascontiguousarray(a)).to(dt).to(dev)
        inputs_tm = to(inputs.T, torch.int32)
        targets_tm = to(targets.T, torch.int32)
        coef_tm = to(coef.T, torch.float32)
        lens_d = to(lens, torch.int32)
        if masks:
            # the kernels index the masks by executed step: a mask set drawn for fewer steps would be read out of bounds
            Bm = inputs.shape[0]
            for name in ('inp', 'out', 'att'):
                m_ = masks.get(name)
                if m_ is not None and (m_.shape[0] < T_run or m_.shape[1] != Bm):
                    raise ValueError("dropout mask '%s' has shape %s; this batch executes %d steps of %d rows"
                                     % (name, tuple(m_.shape), T_run, Bm))
            if masks.get('init_in') is not None and masks['init_in'].shape[0] != Bm:
                raise ValueError("dropout mask 'init_in' has %d rows; the batch has %d" % (masks['init_in'].shape[0], Bm))
        if forward_only:
            loss, logits, attn = eng.train_fwd_bwd(fm.contiguous(), im_embed.contiguous(), inputs_tm, targets_tm, coef_tm,
                                                   lens_d, T_run, None, masks, keeps, c.rnn_map_loss_scale,
                                                   want_logits, want_attn)
            loss[0:1] = loss[1:2]
            return dict(loss=loss, logits=logits, attn=attn, T_run=T_run)
        self.grads.zero_()
        if self.cuda_graph and not want_logits and not want_attn:
            loss, logits, attn = self._graphed_fwd_bwd(fm, im_embed, inputs_tm, targets_tm, coef_tm, lens_d, T_run, masks,
                                                       keeps), None, None
        else:
            loss, logits, attn = eng.train_fwd_bwd(fm.contiguous(), im_embed.contiguous(), inputs_tm, targets_tm,
                                                   coef_tm, lens_d, T_run, self.grad_views, masks, keeps,
                                                   c.rnn_map_loss_scale, want_logits, want_attn)
        mult = 1.0
        if self.legacy_head:
            if mixed5c is None:
                raise ValueError('--legacy: forward_backward needs Mixed_5c of the encoder forward (Engine.encode(images, '
                                 'want_mixed5c=True)) for the gradient of the image-embedding head')
            _dfm, demb = eng.train_encoder_grads(fm.shape[0], T_run)
            eng.legacy_head_bwd(mixed5c, demb, self.gradient(wts.ENC + 'LN_tanh/gamma'), self.gradient(wts.ENC + 'LN_tanh/beta'),
                                self.gradient(wts.ENC + 'im_embed/weight'))
        if self.finetune_cnn:
            if images is None:
                raise ValueError('cnn_finetune: forward_backward needs the images of the last encode_train')
            # chain rule into the encoder: d loss / d (fm, im_embed) -> conv kernel / beta gradients
            dfm, demb = eng.train_encoder_grads(fm.shape[0], T_run)
            eng.encode_bwd(images, dfm, demb, self.cnn_grad_w, self.cnn_grad_b)
            mult = float(getattr(c, 'cnn_grad_multiplier', 1.0))
        if c.l2_decay > 0:
            eng.l2_regularise(self.params, self.grads, c.l2_decay, loss[3:4])
        if mult != 1.0:
            # slim gradient_multipliers scale the gradient of the TOTAL loss, L2 term included, for the CNN
            # variables (src/model_base.py:380-401)
            self.grads[self.n_decoder_flat:].mul_(mult)
        loss[0:1] = loss[1:2] + loss[2:3] + loss[3:4]
        return dict(loss=loss, logits=logits, attn=attn, T_run=T_run)

    def _graphed_fwd_bwd(self, fm, im_embed, inputs_tm, targets_tm, coef_tm, lens_d, T_run, masks, keeps):
        """`Engine.train_fwd_bwd` through a CUDA graph: the launch sequence of `comic_train_fwd_bwd` depends only on the
        shapes (the per-row lengths are device data), so after two eager calls of a shape the third captures it over
        static input buffers and later calls copy their inputs in and replay.  Gradients land in self.grads either way."""
        torch, eng, c = self.torch, self.engine, self.c
        names = tuple(sorted(masks)) if masks else ()
        key = (tuple(fm.shape), tuple(inputs_tm.shape), int(T_run), names, tuple(float(k) for k in keeps))
        ent = self._graphs.get(key)
        if ent is None:
            ent = self._graphs[key] = {'calls': 0, 'graph': None}
        ent['calls'] += 1
        live = dict(fm=fm.contiguous(), im=im_embed.contiguous(), inp=inputs_tm, tgt=targets_tm, coef=coef_tm, lens=lens_d)
        for n in names:
            live['m_' + n] = masks[n]
        ws = eng._ws.get('train')
        if ent['graph'] is not None and (ws is None or ws.data_ptr() != ent['ws_ptr']):
            ent['graph'] = None                          # the engine's workspace moved (a longer batch came by): recapture
        if ent['graph'] is None and ent['calls'] <= 2:
            return eng.train_fwd_bwd(live['fm'], live['im'], inputs_tm, targets_tm, coef_tm, lens_d, T_run, self.grad_views,
                                     masks, keeps, c.rnn_map_loss_scale, False, False)[0]
        if ent['graph'] is None:
            ent['static'] = {k: v.clone() for k, v in live.items()}
            st = ent['static']
            smasks = {n: st['m_' + n] for n in names} if names else None
            torch.cuda.synchronize(eng.device)
            g = torch.cuda.CUDAGraph()
            n0 = eng.launch_count()
            try:
                with torch.cuda.graph(g):
                    ent['loss'] = eng.train_fwd_bwd(st['fm'], st['im'], st['inp'], st['tgt'], st['coef'], st['lens'], T_run,
                                                    self.grad_views, smasks, keeps, c.rnn_map_loss_scale, False, False)[0]
                ent['graph'] = g
                ent['launches'] = eng.launch_count() - n0
                ent['ws_ptr'] = eng._ws['train'].data_ptr()
            except Exception:                           # capture refused (e.g. profiling events active): stay eager
                self.cuda_graph = False
                torch.cuda.synchronize(eng.device)
                self.grads.zero_()
                return eng.train_fwd_bwd(live['fm'], live['im'], inputs_tm, targets_tm, coef_tm, lens_d, T_run,
                                         self.grad_views, masks, keeps, c.rnn_map_loss_scale, False, False)[0]
            self.grads.zero_()                           # (the capture itself does not execute the kernels)
        st = ent['static']
        for k, v in live.items():
            st[k].copy_(v)
        ent['graph'].replay()
        self.replayed_launches += ent['launches']
        return ent['loss'].clone()

    def apply_gradients(self, lr=None):
        """NCCL all-reduce (mean over ranks) + TF-form Adam + repack (model_base.py:387-401)."""
        c, eng = self.c, self.engine
        from .parallel import allreduce_sum_
        world = allreduce_sum_(self.grads)
        self.global_step += 1
        if lr is None:
            lr = cosine_lr(self.global_step - 1, c.max_step, c.lr_start, c.lr_end)
        if self.clip_norm > 0:
            # clip(g / world, c) = clip(g, c * world) / world: the 1 / world of the mean stays folded into the optimiser
            eng.clip_by_norm(self.grads, self._var_off, self._var_len, self.clip_norm * world)
        if getattr(c, 'optimiser', 'adam') == 'sgd':
            # tf.train.MomentumOptimizer(lr, 0.9, use_nesterov=False); its accumulator lives in the adam_m slot buffer
            eng.momentum_step(self.params, self.grads, self.adam_m, lr, 0.9, 1.0 / world)
        else:
            eng.adam_step(self.params, self.grads, self.adam_m, self.adam_v, lr, self.global_step, 0.9, 0.999,
                          c.adam_epsilon, 1.0 / world)
        if self.finetune_cnn:
            eng.refresh_packed_cnn()
        else:
            eng.refresh_packed()
        return lr

    def prepare_images(self, images, seed=None):
        """The images of one step as the encoder takes them.  fp32 [B,224,224,3] images are returned as given.  Raw
        decoded pixels -- a uint8 [B,H,W,3] tensor or array, or a list of uint8 [h,w,3] arrays of mixed sizes (packed
        and copied to the device in one copy) -- are pre-processed on the device: with `cnn_input_augment`,
        `preprocess_for_train` with a random flip and crop per image (train.random_crop_flip, drawn from a host
        generator seeded by `seed`, else by config.rand_seed), otherwise the evaluation pre-processing.  Returns
        (fp32 images, draws): draws = dict(crop_yx, flip) of the augmentation, else None."""
        torch, eng = self.torch, self.engine
        if isinstance(images, (list, tuple)):
            raw = pack_images(images).to(eng.device)
            B = len(raw)
        elif isinstance(images, (np.ndarray, torch.Tensor)) and images.dtype in (np.uint8, torch.uint8):
            raw = eng.to_dev(images)
            B = int(raw.shape[0])
        else:
            return images, None
        if getattr(self.c, 'cnn_input_augment', False):
            rng = np.random.default_rng(seed) if seed is not None else self._augment_rng
            crop, flip = random_crop_flip(B, rng=rng)
            return eng.preprocess_train(raw, crop, flip), dict(crop_yx=crop, flip=flip)
        return eng.preprocess_eval(raw), None

    def step(self, images, captions, rewards=None, seed=None, lr=None, dropout=True):
        """One `sess.run([train_op])`: encoder forward (frozen, or with tape when fine-tuning), decoder
        fwd+bwd (+ encoder backward), optimiser.  Dropout is ON as in the reference's train graph (masks seeded by
        `seed`, default derived from config.rand_seed and the global step); dropout=False runs without masks.
        `images` may be raw uint8 pixels (see prepare_images); the augmentation draws are then returned as
        out['crop_yx'] and out['flip']."""
        eng = self.engine
        images, draws = self.prepare_images(images, seed)
        m5c = None
        if self.finetune_cnn:
            images = eng.to_dev(images)
            im_embed, fm = eng.encode_train(images)
        elif self.legacy_head:
            im_embed, fm, m5c = eng.encode(images, want_mixed5c=True)
        else:
            im_embed, fm = eng.encode(images)
        B = im_embed.shape[0]
        masks, keeps = None, (1.0, 1.0, 1.0)
        if dropout:
            _, _, _, lens = process_inputs(captions, self.c.token_type)
            masks, keeps = self.make_masks(B, int(lens.max()), self.dropout_seed(seed))
        out = self.forward_backward(fm, im_embed, captions, rewards, masks, keeps,
                                    images=images if self.finetune_cnn else None, mixed5c=m5c)
        out['lr'] = self.apply_gradients(lr)
        if draws:
            out.update(draws)
        return out

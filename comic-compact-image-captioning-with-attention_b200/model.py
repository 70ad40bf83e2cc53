"""`CaptionModel` / `ModelBase` call surface of the reference
(src/model.py:21-73, src/model_base.py) over the CUDA engine.

The reference builds a TF graph once and the session loop runs
`sess.run(m.infer_output)` per batch (src/infer_fn.py:130).  Here the model
object owns an `Engine` with bound weights and `run()` executes one batch
eagerly on the current CUDA stream; `infer_output` evaluates the batch given as
`batch_ops` (the reference's attribute of the same name).
"""
from __future__ import annotations

import numpy as np

from . import rops
from . import weights as wts
from .engine import ComicError, Engine, RaggedImages, grown, pack_images


def number_to_base(n, base):
    """common/ops.py:25-40."""
    if base < 2:
        raise ValueError('Base cannot be less than 2.')
    if n < 0:
        sign = -1
        n *= sign
    elif n == 0:
        return [0]
    else:
        sign = 1
    digits = []
    while n:
        digits.append(sign * int(n % base))
        n //= base
    return digits[::-1]


class ModelBase(object):
    """src/model_base.py:32-46 + the helpers the inference path needs."""

    def __init__(self, config):
        self._config = c = config
        assert c.token_type in ['radix', 'word', 'char']
        if c.token_type == 'radix':
            self._softmax_size = c.radix_base + 2
        else:
            self._softmax_size = len(c.itow)

    def is_training(self):
        return self.mode == 'train'

    # -- encoder (src/model_base.py:56-104) ----------------------------------
    # True: decode calls keep the alignment history and return the top-beam attention maps (what the reference's
    # `sess.run(infer_output)` fetches, src/infer_fn.py:130); False: no history is written or copied -- the
    # production setting when `save_attention_maps` is off (src/infer_fn.py:169-171 only DUMPS the maps then)
    collect_attention_maps = True

    def _encoder(self, images):
        if isinstance(images, (list, tuple)):
            images = pack_images(images).to(self.engine.device)
        if isinstance(images, RaggedImages) or images.dtype == self.engine.torch.uint8:
            # raw decoded pixels (one size, or a packed batch of mixed sizes): the reference's evaluation
            # pre-processing on the device (inception_preprocessing_radix.py:229-235, 270-273)
            images = self.engine.preprocess_eval(images)
        self.im_embed, self.cnn_fmaps = self.engine.encode(images)
        return self.im_embed, self.cnn_fmaps

    # -- _rnn_dynamic_decoder ids / iterations (src/model_base.py:692-714) ---
    def _start_end_ids(self):
        c = self._config
        if c.token_type == 'radix':
            return int(c.radix_base), int(c.radix_base + 1)
        return int(c.wtoi['<GO>']), int(c.wtoi['<EOS>'])

    def _maximum_iterations(self):
        c = self._config
        m = c.infer_max_length
        if c.token_type == 'radix':
            m *= len(number_to_base(len(c.wtoi), c.radix_base))
        elif c.token_type == 'char':
            m *= 5
        return m

    # -- decoder (src/model_base.py:109-184) ---------------------------------
    def _decoder_rnn(self):
        c = self._config
        eng = self.engine
        align = c.attn_alignment_method
        if align == 'add_LN':
            att_mech = rops.MultiHeadAddLN
        elif align == 'dot':
            att_mech = rops.MultiHeadDot
        else:
            raise ValueError('Invalid alignment method.')
        if c.attn_probability_fn not in ('softmax', 'sigmoid'):
            raise ValueError('Invalid alignment method.')
        batch_size = self.im_embed.shape[0]
        is_inference = self.mode == 'infer'
        beam_search = is_inference and c.infer_beam_size > 1
        c0, h0 = eng.rnn_init(self.im_embed)                                   # _get_rnn_init :651-689
        rnn_init = h0 if c.rnn_name == 'GRU' else rops.LSTMStateTuple(c0, h0)   # GRUCell state: the h tensor
        cnn_attention = att_mech(c.rnn_size, self.cnn_fmaps, c.cnn_fm_projection, c.attn_num_heads,
                                 memory_sequence_length=None, probability_fn=c.attn_probability_fn,
                                 engine=eng)
        attention_cell = rops.MultiHeadAttentionWrapperV3(
            deep_output_layer=False, context_layer=c.attn_context_layer, alignments_keep_prob=1.0,
            cell=c.rnn_name, attention_mechanism=cnn_attention, attention_layer_size=None,
            alignment_history=self.collect_attention_maps, cell_input_fn=None, output_attention=False,
            initial_cell_state=rnn_init)
        attention_cell.im_embed = self.im_embed          # rops.rnn_decoder_training recomputes the initial state from it
        attention_cell._defer_T = bool(getattr(self, '_defer_T', False))
        start_id, end_id = self._start_end_ids()
        max_it = self._maximum_iterations()
        if beam_search:
            raw = rops.rnn_decoder_beam_search(attention_cell, None, None, batch_size, c.infer_beam_size,
                                               c.infer_length_penalty_weight, max_it, start_id, end_id)
        else:
            raw = rops.rnn_decoder_search(attention_cell, None, None, batch_size, max_it, start_id, end_id)
        logits, output_ids, attn_maps = self._decoder_post_process(raw, top_beam=True)
        self.dec_preds, self.dec_logits, self.dec_attn_maps = output_ids, logits, attn_maps
        self.dec_time = raw[2].time                      # executed steps: host int, or a device tensor with _defer_T
        return logits, output_ids, attn_maps

    # -- src/model_base.py:272-314 ---------------------------------------------
    def _decoder_post_process(self, rnn_raw_outputs, top_beam=True):
        beam_search = (self.mode == 'infer' and rnn_raw_outputs[0].dim() > 2)
        if beam_search:
            predicted_ids, scores, dec_states = rnn_raw_outputs          # (time, batch, beam)
            if top_beam:
                output_ids = predicted_ids[:, :, 0].transpose(0, 1)      # (batch, seq_len)
                logits = scores[:, :, 0].transpose(0, 1)
            else:
                output_ids = predicted_ids.permute(2, 1, 0)              # (beam, batch, time)
                logits = scores.permute(2, 1, 0)
        else:
            output_ids, logits, dec_states = rnn_raw_outputs
            logits = logits.transpose(0, 1)
            output_ids = output_ids.transpose(0, 1)
        # the engine already returns the (reordered, top-beam) map as [B, H, T, M]; () when no history was kept
        attn_map = dec_states.alignment_history
        if isinstance(attn_map, tuple):
            attn_map = None
        return logits, output_ids, attn_map


class CaptionModel(ModelBase):
    """src/model.py:21-73.  mode 'infer': `run()` / `infer_output`.  mode 'train' / 'eval':
    `train_step(images, captions)` = one `sess.run([dec_log_ppl, global_step])` of
    src/train_fn.py:120 (fwd + bwd + Adam), `eval_step` the teacher-forced perplexity of
    src/train_fn.py:320-338.  `reuse=True` shares the variables (engine / trainer) of `share`."""

    def __init__(self, config, mode, batch_ops=None, reuse=False, name=None, weights=None, engine=None,
                 share=None):
        assert mode in ['train', 'eval', 'infer']
        super(CaptionModel, self).__init__(config)
        self.mode = mode
        self.batch_ops = batch_ops
        self.reuse = reuse
        self.name = name
        self.trainer = None
        if share is not None:
            engine = share.engine
            self.trainer = share.trainer
        if mode in ('train', 'eval') and self.trainer is None:
            from .train import Trainer
            if weights is None:
                weights = wts.init_weights(config, seed=getattr(config, 'rand_seed', 48964896))
            self.trainer = Trainer(config, weights, engine=engine)
            engine = self.trainer.engine
        if engine is None:
            engine = Engine(config)
            if weights is None:
                weights = wts.init_weights(config, seed=getattr(config, 'rand_seed', 48964896))
            engine.bind_weights(weights)
        self.engine = engine
        self._weights = weights if weights is not None else getattr(share, '_weights', None)
        self._pinned = {}

    # -- ModelBase.get_global_step / update_lr (src/model_base.py:767-773) ----
    def get_global_step(self):
        return 0 if self.trainer is None else self.trainer.global_step

    def train_step(self, images, captions, seed=None, lr=None, dropout=True):
        """One optimiser step; returns (dec_log_ppl, global_step) like train_fn.py:120.  Dropout on by default
        (the reference's train graph); `seed` fixes the masks, dropout=False disables them."""
        assert self.mode == 'train'
        eng = self.engine
        if not isinstance(images, (list, tuple)):
            images = eng.torch.as_tensor(images).to(eng.device, non_blocking=True)
        out = self.trainer.step(images, np.asarray(captions), None, seed, lr, dropout)
        self.dec_log_ppl = out['loss'][1]
        return self.dec_log_ppl, self.trainer.global_step

    def eval_step(self, images, captions):
        """Teacher-forced log-perplexity without dropout or update (_run_eval_loop)."""
        eng = self.engine
        images = eng.torch.as_tensor(images).to(eng.device, non_blocking=True)
        im_embed, fm = eng.encode(images)
        # forward only: no gradient buffers are touched, and with train_mode=cnn_finetune no tape is needed
        out = self.trainer.forward_backward(fm, im_embed, np.asarray(captions), forward_only=True)
        return out['loss'][1]

    def restore_model(self, weights=None, checkpoint_path=None):
        """ModelBase.restore_model (src/model_base.py:422-490).  `weights`: a W-table to bind as is; otherwise the
        TF V2 checkpoint at `checkpoint_path` (default `config.checkpoint_path`; a directory resolves through its
        `checkpoint` state file) is read with the reference's rules -- resume / whole model minus
        `checkpoint_exclude_scopes` / CNN only (checkpoint.restore_weights) -- over the current variables.
        Returns the restore info dict (mode, restored names, optimiser tensors when resuming)."""
        from . import checkpoint as ckpt
        info = dict(mode='table', restored=sorted(weights) if weights is not None else [])
        if weights is None:
            cur = self.current_weights()
            weights, info = ckpt.restore_weights(self._config, cur, checkpoint_path=checkpoint_path)
        if self.trainer is not None:
            self.trainer.load_variables(weights, info.get('extra'))
        else:
            self.engine.bind_weights(weights)
        self._weights = weights
        return info

    def current_weights(self):
        """The model's variables as a W-table of numpy arrays (the trainer's flat buffer when training)."""
        if self.trainer is not None:
            return self.trainer.variables_numpy()
        W = getattr(self, '_weights', None)
        if W is None:
            raise ValueError('no W-table is attached to this model (pass weights= when constructing it)')
        return {k: np.asarray(v) for k, v in W.items()}

    def _to_host(self, t, key):
        """Device -> pinned host staging buffer (reused across calls)."""
        torch = self.engine.torch
        t = t.contiguous()
        buf = self._pinned.get(key)
        if buf is None or buf.shape != t.shape or buf.dtype != t.dtype:
            buf = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
            self._pinned[key] = buf
        buf.copy_(t, non_blocking=True)
        return buf

    def run(self, images=None):
        """One `sess.run(self.infer_output)` (src/infer_fn.py:130): images
        [B,224,224,3] NHWC fp32 (host numpy / torch -- pinned memory copies
        asynchronously -- or a device tensor), raw uint8 [B,H,W,3] pixels, or a
        list of uint8 [h,w,3] images of mixed sizes (packed, one copy, one
        pre-processing launch).  Returns [dec_preds (B,T) int32,
        attn_maps (B,H,T,M) fp32] as numpy views of pinned staging buffers that
        the next call overwrites."""
        eng = self.engine
        torch = eng.torch
        if images is None:
            images = self.batch_ops[0]
        if isinstance(images, (list, tuple)):
            dev_images = pack_images(images).to(eng.device)
        else:
            images = torch.as_tensor(images)
            if images.dtype not in (torch.float32, torch.uint8):
                images = images.float()
            dev_images = images.to(eng.device, non_blocking=True).contiguous()
        self._encoder(dev_images)
        self._decoder_rnn()
        preds = self._to_host(self.dec_preds, 'preds')
        attn = self._to_host(self.dec_attn_maps, 'attn') if self.dec_attn_maps is not None else None
        torch.cuda.current_stream(eng.device).synchronize()
        return [preds.numpy(), None if attn is None else attn.numpy()]

    def run_stream(self, batches, depth=2):
        """The inference loop of src/infer_fn.py:166-184 (`for each batch: sess.run(infer_output)`) as a
        software pipeline: yields [dec_preds, attn_maps] per batch, in order, like `run`.

        Three CUDA streams: the host->device copy of batch i+1 (pinned host memory copies at PCIe
        speed) and the device->host copy of batch i-1's results run while batch i computes, so in
        steady state a batch costs max(compute, H2D, D2H) instead of their sum.  `depth` device
        input buffers / pinned result buffers rotate: a yielded result stays valid until the
        following `next()`.  Device-resident batches skip the input copy.

        Batches may be uint8 [B,H,W,3] raw pixels: they cross PCIe as bytes (a quarter of the fp32 volume) and the
        reference's evaluation pre-processing runs on the device.  A batch may also be a list or tuple of uint8
        [h,w,3] images of mixed sizes: the host packs it (pack_images) into the slot's pinned staging buffer while the
        device computes the previous batch, one copy moves it into the slot's device buffer, and one launch
        pre-processes it.  Both buffers grow by at least 1.25x to the largest batch seen, so the slot's graph keeps
        replaying while the sizes change.  With `collect_attention_maps = False` the second
        element of every result is None and neither history nor maps are written or copied."""
        eng = self.engine
        torch = eng.torch
        dev = eng.device
        comp = torch.cuda.current_stream(dev)
        if not hasattr(self, '_pipe_streams'):
            self._pipe_streams = (torch.cuda.Stream(dev), torch.cuda.Stream(dev))
            self._pipe_slots = {}
        s_in, s_out = self._pipe_streams
        slots = self._pipe_slots.setdefault(depth, [dict() for _ in range(depth)])

        def stage_in(i, images):
            sl = slots[i % depth]
            if isinstance(images, (list, tuple)):
                if sl.get('ev_in') is not None:
                    sl['ev_in'].synchronize()               # the slot's previous copy has read its staging buffer
                packed = pack_images(images, sl.get('stage'))
                sl['stage'] = packed._buf
                buf = sl['dev_ragged'] = grown(sl.get('dev_ragged'), packed.nbytes, device=dev)
                with torch.cuda.stream(s_in):
                    if sl.get('ev_comp') is not None:
                        s_in.wait_event(sl['ev_comp'])
                    r = packed.to(dev, buf)
                    ev = torch.cuda.Event()
                    ev.record(s_in)
                sl['dev'], sl['ev_in'] = (r.data, r.offsets, r.hw), ev
                return
            images = torch.as_tensor(images)
            if images.dtype not in (torch.float32, torch.uint8):
                images = images.float()
            if images.is_cuda:
                sl['dev'], sl['ev_in'] = (images.contiguous(),), None
                return
            buf = sl.get('dev_in')
            if buf is None or buf.shape != images.shape or buf.dtype != images.dtype:
                buf = sl['dev_in'] = torch.empty(images.shape, dtype=images.dtype, device=dev)
            with torch.cuda.stream(s_in):
                if sl.get('ev_comp') is not None:
                    s_in.wait_event(sl['ev_comp'])          # the slot's previous batch has been consumed
                buf.copy_(images, non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(s_in)
            sl['dev'], sl['ev_in'] = (buf,), ev

        def pinned(sl, key, t):
            b = sl.get(key)
            if b is None or b.shape != t.shape or b.dtype != t.dtype:
                b = sl[key] = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
            return b

        def compute(i):
            sl = slots[i % depth]
            if sl['ev_in'] is not None:
                comp.wait_event(sl['ev_in'])
            def device_step(*images):
                # no host sync inside (rops: _defer_T): full-length results + the device step count, trimmed in finish()
                images = images[0] if len(images) == 1 else RaggedImages(*images)
                self._defer_T = True
                try:
                    self._encoder(images)
                    self._decoder_rnn()
                finally:
                    self._defer_T = False
                return (self.dec_preds.contiguous(),
                        self.dec_attn_maps.contiguous() if self.dec_attn_maps is not None else None,
                        self.dec_time.reshape(1))
            # one CUDA graph per input slot (Engine.graphed): replayed from the slot's third batch on
            preds, attn, t_dev = eng.graphed(('run_stream', i % depth, bool(self.collect_attention_maps)), device_step,
                                             *sl['dev'])
            ev = torch.cuda.Event()
            ev.record(comp)
            sl['ev_comp'] = ev
            hp = pinned(sl, 'h_preds', preds)
            ha = pinned(sl, 'h_attn', attn) if attn is not None else None
            ht = pinned(sl, 'h_time', t_dev)
            with torch.cuda.stream(s_out):
                s_out.wait_event(ev)
                hp.copy_(preds, non_blocking=True)
                ht.copy_(t_dev, non_blocking=True)
                preds.record_stream(s_out)
                if attn is not None:
                    ha.copy_(attn, non_blocking=True)
                    attn.record_stream(s_out)
                evo = torch.cuda.Event()
                evo.record(s_out)
            sl['ev_out'], sl['out'] = evo, (hp, ha, ht)

        def finish(i):
            sl = slots[i % depth]
            sl['ev_out'].synchronize()
            hp, ha, ht = sl['out']
            T = int(ht[0])
            if T < 0:
                raise ComicError('decode loop aborted: the persistent kernel gave up at a grid barrier')
            return [hp.numpy()[:, :T], None if ha is None else ha.numpy()[:, :, :T, :]]

        it = iter(batches)
        cur = next(it, None)
        if cur is None:
            return
        i, pending = 0, None
        stage_in(0, cur)
        while True:
            nxt = next(it, None)
            if nxt is not None:
                stage_in(i + 1, nxt)
            compute(i)
            if pending is not None:
                yield finish(pending)
            pending = i
            if nxt is None:
                break
            i += 1
        yield finish(pending)

    @property
    def infer_output(self):
        return self.run()


class CaptionModel_SCST(ModelBase):
    """src/model.py:76-141.  scst_mode 'sample': `sample(images)` -> (dec_preds_beam [k,B,T],
    dec_preds_greedy [B,T]) (greedy + beam-`scst_beam_size`, max length 20, no dropout);
    scst_mode 'train': `train_scst(images_or_features, captions, rewards)` = weighted-XE step."""

    def __init__(self, config, scst_mode, reuse=False, weights=None, share=None):
        assert scst_mode in ['train', 'sample']
        super(CaptionModel_SCST, self).__init__(config)
        self.mode = scst_mode if scst_mode == 'train' else 'infer'
        self.name = scst_mode
        self.reuse = reuse
        if share is not None:
            self.trainer = share.trainer
        else:
            from .train import Trainer
            if weights is None:
                weights = wts.init_weights(config, seed=getattr(config, 'rand_seed', 48964896))
            self.trainer = Trainer(config, weights)
        self.engine = self.trainer.engine

    def sample(self, images):
        from . import scst
        c = self._config
        eng = self.engine
        images = eng.torch.as_tensor(images).to(eng.device, non_blocking=True)
        cap_beam, cap_greedy, self.im_embed, self.cnn_fmaps = scst.sample_captions(eng, c, images, c.scst_beam_size)
        self.dec_preds_beam, self.dec_preds_greedy = cap_beam, cap_greedy
        return cap_beam, cap_greedy

    def train_scst(self, images, captions, rewards, seed=None, lr=None, dropout=True):
        """images: the k-times tiled batch of train_fn.py:251 (or None to reuse the features of the
        last `sample()` of the shared model, repeated k times)."""
        c, eng, tr = self._config, self.engine, self.trainer
        if images is not None:
            images = eng.torch.as_tensor(images).to(eng.device, non_blocking=True)
            im_embed, fm = eng.encode(images)
        else:
            raise ValueError('images required')
        captions = np.asarray(captions)
        masks, keeps = None, (1.0, 1.0, 1.0)
        if dropout:
            from .train import process_inputs
            lens = process_inputs(captions, c.token_type)[3]
            masks, keeps = tr.make_masks(fm.shape[0], int(lens.max()), tr.dropout_seed(seed))
        out = tr.forward_backward(fm, im_embed, captions, np.asarray(rewards, np.float32), masks, keeps)
        tr.apply_gradients(lr)
        return out['loss'][1]


def synthetic_images(batch, seed=0):
    """SURVEY.md §8d: uniform(-1,1) fp32 [B,224,224,3], seeded."""
    rng = np.random.default_rng(seed)
    return rng.uniform(-1.0, 1.0, size=(batch, 224, 224, 3)).astype(np.float32)

"""Host-side mirror of the reference's decoder ops library `common/ops_rnn.py`.

Same names, argument meaning and error behaviour as the reference; the TF graph
the reference builds is replaced by calls into libcomic_b200.so (engine.py).

  rnn_decoder_beam_search     common/ops_rnn.py:49-112
  rnn_decoder_search          common/ops_rnn.py:115-180
  rnn_decoder_training        common/ops_rnn.py:183-243   (forward; the fused fwd + bwd lives in train.py)
  MultiHeadAddLN / MultiHeadDot  common/ops_rnn.py:403-565, 603-632
  MultiHeadAttentionWrapperV3  common/ops_rnn.py:635-803
"""
from __future__ import annotations

import collections

from .engine import executed_steps

AttentionWrapperState = collections.namedtuple(
    'AttentionWrapperState',
    ('cell_state', 'attention', 'time', 'alignments', 'alignment_history', 'attention_state'))

LSTMStateTuple = collections.namedtuple('LSTMStateTuple', ('c', 'h'))


class MultiHeadAttV3(object):
    """Attention mechanism with its memory bound (common/ops_rnn.py:403-520).

    `feature_map` is the UNTILED [B, M, C] device tensor: keys (= fm . W_k) and
    values are computed once per image and shared by the image's beams, where
    the reference computes them after `tile_batch` (src/model_base.py:130-131).
    """
    _alignment = None

    def __init__(self, num_units, feature_map, fm_projection, num_heads=None, scale=True,
                 memory_sequence_length=None, probability_fn='softmax', name='MultiHeadAttV3',
                 engine=None):
        assert fm_projection in [None, 'independent', 'tied']           # ops_rnn.py:433
        if engine is None:
            raise ValueError('an Engine is required')
        if memory_sequence_length is not None:
            raise NotImplementedError('memory_sequence_length is always None in the reference model '
                                      '(src/model_base.py:155)')
        d = engine.dims
        if fm_projection in ('tied', 'independent'):
            assert num_units % num_heads == 0, \
                'For `tied` projection, attention size/depth must be divisible by the number of attention heads.'
        else:
            assert feature_map.shape[-1] % num_heads == 0, \
                'For `none` projection, feature map channel dim size must be divisible by the number of attention heads.'
        if (num_units, num_heads, fm_projection) != (d.R, d.H, d.fm_projection):
            raise ValueError('attention mechanism does not match the engine configuration')
        self._engine = engine
        self._num_units = num_units
        self._num_heads = num_heads
        self._fm_projection = fm_projection
        self._feature_map_shape = list(feature_map.shape)
        self._name = name
        self.batch_size = feature_map.shape[0]
        self.feature_map = feature_map
        self.keys, self.values = engine.project_fm(feature_map)          # ops_rnn.py:441-477


class MultiHeadAddLN(MultiHeadAttV3):
    """common/ops_rnn.py:523-565."""
    _alignment = 'add_LN'


class MultiHeadDot(MultiHeadAttV3):
    """common/ops_rnn.py:603-632."""
    _alignment = 'dot'


class MultiHeadAttentionWrapperV3(object):
    """common/ops_rnn.py:635-803.  `cell` is the (name of the) inner RNN cell;
    `initial_cell_state` an LSTMStateTuple of per-image [B, R] tensors (LSTM) or
    the [B, R] h tensor (GRU: TF's GRUCell state is a tensor, not a tuple)."""

    def __init__(self, deep_output_layer=False, context_layer=True, alignments_keep_prob=1.0,
                 cell='LSTM', attention_mechanism=None, attention_layer_size=None,
                 alignment_history=True, cell_input_fn=None, output_attention=False,
                 initial_cell_state=None, name=None):
        if attention_mechanism is None or isinstance(attention_mechanism, (list, tuple)):
            raise ValueError('Only a single attention mechanism can be used.')   # ops_rnn.py:656-657
        if cell not in ('LSTM', 'GRU'):
            raise NotImplementedError('Only `LSTM` and `GRU` are built on the CUDA path.')
        if attention_layer_size is not None or cell_input_fn is not None or output_attention:
            raise NotImplementedError('the reference always passes attention_layer_size=None, '
                                      'cell_input_fn=None, output_attention=False (src/model_base.py:157-167)')
        eng = attention_mechanism._engine
        if (cell == 'GRU') != eng.gru:
            raise ValueError('cell %s does not match the engine configuration' % cell)
        if bool(context_layer) != eng.dims.context_layer:
            raise ValueError('context_layer does not match the engine configuration')
        self._attention_mechanism = attention_mechanism
        self._alignment_history = bool(alignment_history)    # False: the decode loops keep no alignment history at all
        self._alignments_keep_prob = alignments_keep_prob
        self._initial_cell_state = initial_cell_state
        self._engine = eng
        self.name = name or 'multi_head_attention_wrapper_v3'

    @property
    def engine(self):
        return self._engine

    def zero_state(self, batch_size, dtype=None):
        """ops_rnn.py:776-803 (attention / alignments zeros, cell_state = initial_cell_state)."""
        eng, d = self._engine, self._engine.dims
        return AttentionWrapperState(
            cell_state=self._initial_cell_state,
            attention=eng.torch.zeros((batch_size, d.A), device=eng.device),
            time=0,
            alignments=eng.torch.zeros((batch_size, d.H * d.M), device=eng.device),
            alignment_history=(),
            attention_state=eng.torch.zeros((batch_size, d.H * d.M), device=eng.device))

    def __call__(self, inputs_ids, state, beam=1, masks=None, keeps=(1.0, 1.0, 1.0)):
        """One wrapper step (ops_rnn.py:660-755) on token ids [N]; returns
        (cell_output h', logits, new_state).  `state.cell_state` holds [N, R]
        tensors here (already tiled)."""
        eng = self._engine
        am = self._attention_mechanism
        N = inputs_ids.shape[0]
        B = N // beam
        m = masks or {}
        c_in, h_in = _split_cell_state(eng, state.cell_state)
        r = eng.decode_step(am.keys, am.values, B, beam, inputs_ids, c_in, h_in,
                            state.attention, m.get('inp'), m.get('out'), m.get('att'), keeps)
        new_state = AttentionWrapperState(
            cell_state=r['h'] if eng.gru else LSTMStateTuple(r['c'], r['h']), attention=r['attention'], time=state.time + 1,
            alignments=r['alignments'], alignment_history=(), attention_state=r['alignments'])
        return r['h'], r['logits'], new_state


def _split_cell_state(eng, cell_state):
    """(c, h) of a wrapper's cell state; c is None for the GRU cell, whose state is the h tensor itself."""
    if eng.gru:
        return None, cell_state
    return cell_state.c, cell_state.h


def _check_ids(cell, start_id, end_id):
    eng = cell.engine
    if int(start_id) != eng.go or int(end_id) != eng.eos:
        raise ValueError('start_id/end_id (%d, %d) do not match the bound model (%d, %d)'
                         % (int(start_id), int(end_id), eng.go, eng.eos))


def rnn_decoder_beam_search(cell, embedding_fn, output_layer, batch_size, beam_size,
                            length_penalty_weight, maximum_iterations, start_id, end_id,
                            swap_memory=True):
    """Beam search decode (common/ops_rnn.py:49-112).

    `embedding_fn` / `output_layer` are bound inside the engine (embedding_map,
    output_projection) and accepted for signature parity.  Returns
    (predicted_ids [T,B,k] int32, scores [T,B,k] fp32, cell_state) where
    cell_state.alignment_history is the reordered top-beam map [B,H,T,M] source
    (see model._decoder_post_process)."""
    del embedding_fn, output_layer, swap_memory
    _check_ids(cell, start_id, end_id)
    eng = cell.engine
    am = cell._attention_mechanism
    if am.batch_size != batch_size:
        raise ValueError('Non-matching batch sizes between the memory (encoder output) and the query '
                         '(decoder output).')                           # ops_rnn.py:679-690
    c0, h0 = _split_cell_state(eng, cell._initial_cell_state)
    want_attn = getattr(cell, '_alignment_history', True)
    r = eng.decode_beam(am.keys, am.values, c0, h0, int(beam_size), float(length_penalty_weight),
                        int(maximum_iterations), want_attn=want_attn)
    if getattr(cell, '_defer_T', False):
        # pipelined / graph-captured callers: no host sync here.  All maximum_iterations rows are returned (rows past the
        # executed count hold end_id / zero maps, as gather_tree and the map gather leave them) and `state.time` is the
        # DEVICE step count; the caller trims after its own copy to the host.
        T = int(maximum_iterations)
        state = AttentionWrapperState(cell_state=None, attention=None, time=r['T'], alignments=None,
                                      alignment_history=r['attn'] if want_attn else (), attention_state=None)
        rnn_decoder_beam_search.last_extra = dict(parent_ids=r['parent_ids'], step_ids=r['step_ids'], lengths=r['lengths'])
        return r['predicted_ids'], r['scores'], state
    T = executed_steps(r['T'])                       # the one device->host sync of a decode call
    r['T_host'] = T
    state = AttentionWrapperState(cell_state=None, attention=None, time=T, alignments=None,
                                  alignment_history=r['attn'][:, :, :T, :] if want_attn else (), attention_state=None)
    state_extra = dict(parent_ids=r['parent_ids'][:T], step_ids=r['step_ids'][:T], lengths=r['lengths'])
    rnn_decoder_beam_search.last_extra = state_extra
    return r['predicted_ids'][:T], r['scores'][:T], state


def rnn_decoder_search(cell, embedding_fn, output_layer, batch_size, maximum_iterations, start_id,
                       end_id, swap_memory=True, greedy_search=True):
    """Greedy decode (common/ops_rnn.py:115-180).  Returns (output_ids [T,B],
    rnn_out logits [T,B,V], state)."""
    del embedding_fn, output_layer, swap_memory
    if not greedy_search:
        raise NotImplementedError('sample search is commented out in the reference (src/model.py:127-129)')
    _check_ids(cell, start_id, end_id)
    eng = cell.engine
    am = cell._attention_mechanism
    if am.batch_size != batch_size:
        raise ValueError('Non-matching batch sizes between the memory (encoder output) and the query '
                         '(decoder output).')
    c0, h0 = _split_cell_state(eng, cell._initial_cell_state)
    want_attn = getattr(cell, '_alignment_history', True)
    r = eng.decode_greedy(am.keys, am.values, c0, h0, int(maximum_iterations), want_attn=want_attn)
    if getattr(cell, '_defer_T', False):             # see rnn_decoder_beam_search
        state = AttentionWrapperState(cell_state=None, attention=None, time=r['T'], alignments=None,
                                      alignment_history=r['attn'] if want_attn else (), attention_state=None)
        return r['ids'], r['logits'], state
    T = executed_steps(r['T'])
    state = AttentionWrapperState(cell_state=None, attention=None, time=T, alignments=None,
                                  alignment_history=r['attn'][:, :, :T, :] if want_attn else (), attention_state=None)
    return r['ids'][:T], r['logits'][:T], state


def rnn_decoder_training(cell, embeddings, output_layer, batch_size, sequence_length, swap_memory=True):
    """Teacher-forced decode (common/ops_rnn.py:183-243): TrainingHelper + BasicDecoder +
    dynamic_decode(impute_finished=True), time-major.

    `embeddings` are the decoder INPUT TOKEN IDS [time, batch] int32: the embedding map is bound inside the engine
    (as for `embedding_fn` of the search functions), so the lookup of src/model_base.py:587-593 happens on the device.
    `cell.im_embed` must hold the image embedding [batch, E] the initial state was built from (the engine's
    teacher-forced pass recomputes that state itself).  Returns (output_ids [T,B] int32 = arg-max samples, rnn_out
    logits [T,B,V] -- rows past their length are zero, steps past max(sequence_length) repeat the last executed step
    (:237-241) -- and a state whose alignment_history is [B,H,T_run,M])."""
    del output_layer, swap_memory
    eng = cell.engine
    torch = eng.torch
    am = cell._attention_mechanism
    if am.batch_size != batch_size:
        raise ValueError('Non-matching batch sizes between the memory (encoder output) and the query '
                         '(decoder output).')
    im_embed = getattr(cell, 'im_embed', None)
    if im_embed is None:
        raise ValueError('rnn_decoder_training: set cell.im_embed to the image embedding of the initial state')
    ids = torch.as_tensor(embeddings).to(device=eng.device, dtype=torch.int32).contiguous()
    if ids.dim() != 2 or ids.shape[1] != batch_size:
        raise ValueError('embeddings must be the [time, batch] input token ids, got %s' % (tuple(ids.shape),))
    lens = torch.as_tensor(sequence_length).to(device=eng.device, dtype=torch.int32).contiguous()
    T = int(ids.shape[0])
    T_run = int(lens.max().item())
    if T_run < 1 or T_run > T:
        raise ValueError('sequence_length must lie in [1, time]')
    zeros_i = torch.zeros_like(ids)
    zeros_f = torch.zeros(ids.shape, dtype=torch.float32, device=eng.device)
    _loss, logits, attn = eng.train_fwd_bwd(am.feature_map.contiguous(), im_embed.contiguous(), ids, zeros_i, zeros_f, lens,
                                            T_run, None, None, (1.0, 1.0, 1.0), 0.0, True, True)
    rnn_out = logits.transpose(0, 1).contiguous()                        # [T, B, V]
    if T_run < T:
        rnn_out[T_run:] = rnn_out[T_run - 1:T_run]
    valid = (torch.arange(T_run, device=eng.device)[:, None] < lens[None, :])
    output_ids = torch.zeros((T, batch_size), dtype=torch.int32, device=eng.device)
    output_ids[:T_run] = torch.where(valid, rnn_out[:T_run].argmax(dim=-1).to(torch.int32), torch.zeros_like(output_ids[:T_run]))
    if T_run < T:
        output_ids[T_run:] = output_ids[T_run - 1:T_run]
    state = AttentionWrapperState(cell_state=None, attention=None, time=T_run, alignments=None,
                                  alignment_history=attn, attention_state=None)
    return output_ids, rnn_out, state

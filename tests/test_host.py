"""Host-side logic (CPU): config.pkl contract, flag defaults against the
reference's argparse (recorded in tests/golden/reference_cli_flags.json), radix helpers."""
import json
import os
import pickle

import pytest

import comic_b200  # noqa: F401
from comic_b200 import configuration as conf

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')
PATH_FLAGS = ('infer_checkpoints_dir', 'dataset_dir')      # defaults are path expressions of the reference's checkout


def _reference_cli():
    """{'train.py' | 'infer.py': {flag: {'type', 'default', 'choices'}}} of the reference's two argparse parsers."""
    with open(os.path.join(GOLDEN, 'reference_cli_flags.json')) as f:
        return json.load(f)


def test_config_pickle_round_trip(tmp_path):
    c = conf.make_config(log_path=str(tmp_path))
    c.save_config_to_file()
    p = os.path.join(str(tmp_path), 'config.pkl')
    with open(p, 'rb') as f:
        raw = pickle.load(f)
    assert isinstance(raw, dict) and raw['rnn_size'] == 512 and raw['cnn_fm_projection'] == 'tied'
    c2 = conf.load_config(p)
    assert c2.__dict__ == c.__dict__
    # protocol 2, as common/configuration.py:34-35 writes it
    assert open(p, 'rb').read(2) == b'\x80\x02'


def test_python2_pickle_is_readable(tmp_path):
    """A py2 cPickle protocol-2 dict with a non-ASCII byte string loads via the latin1 retry."""
    blob = b'\x80\x02}q\x00(U\x04nameq\x01U\x04caf\xe9q\x02U\x08rnn_sizeq\x03M\x00\x02u.'
    p = tmp_path / 'config.pkl'
    p.write_bytes(blob)
    c = conf.load_config(str(p))
    assert c.rnn_size == 512


def test_north_star_fields_present():
    c = conf.make_config()
    for f in ('token_type', 'attn_num_heads', 'cnn_fm_projection', 'rnn_size', 'infer_beam_size', 'scst_beam_size',
              'legacy', 'radix_base', 'rnn_word_size', 'attn_keep_prob', 'dropout_rnn_in', 'dropout_rnn_out',
              'l2_decay', 'adam_epsilon', 'lr_start', 'lr_end', 'itow', 'wtoi', 'vocab_size', 'max_step'):
        assert hasattr(c, f), f
    assert c.cnn_input_size == [224, 224]


def test_none_string_becomes_none_and_mode_overrides():
    c = conf.make_config(cnn_fm_projection='none', token_type='word', attn_num_heads=1)
    assert c.cnn_fm_projection is None
    s = conf.make_config(train_mode='scst')
    assert s.batch_size_train == 10 and s.lr_start == 1e-3 and s.scst_weight_bleu == [0.0, 0.0, 0.0, 2.0]
    f = conf.make_config(train_mode='cnn_finetune')
    assert f.freeze_scopes == '' and f.lr_start == 1e-3 and f.max_epoch == 10
    leg = conf.make_config(legacy=True)
    assert leg.rnn_init_method == 'project_hidden' and leg.attn_keep_prob == 1.0 and leg.adam_epsilon == 1e-6


def test_flag_defaults_match_reference_cli():
    """Every flag of src/train.py:29-162 / src/infer.py:27-72 exists with the same default."""
    ref_cli = _reference_cli()
    for fname, table in (('train.py', conf.TRAIN_DEFAULTS), ('infer.py', conf.INFER_DEFAULTS)):
        ref = ref_cli[fname]
        assert len(ref) > 10
        for flag, spec in ref.items():
            if flag in ('gpu', 'per_process_gpu_memory_fraction') + PATH_FLAGS:
                continue
            assert flag in table, '%s: flag --%s missing' % (fname, flag)
            val = spec['default']
            ours = table[flag]
            if flag == 'cnn_input_size':
                val = [int(v) for v in val.split(',')]
            if val == 'none':
                val = None if ours is None else val
            if isinstance(val, str) and val == '' and ours in ('', None):
                continue
            assert ours == val, '%s --%s: %r != reference %r' % (fname, flag, ours, val)


def test_number_to_base_and_max_iterations():
    from comic_b200.model import number_to_base
    assert number_to_base(0, 256) == [0]
    assert number_to_base(255, 256) == [255]
    assert number_to_base(256, 256) == [1, 0]
    assert number_to_base(9999, 256) == [39, 15]
    with pytest.raises(ValueError):
        number_to_base(5, 1)


def test_synthetic_vocab_layout():
    """datasets/preprocessing/prepro_base.py:149-223: words 0.., <UNK>, <GO>, <EOS>; PAD = -1."""
    itow, wtoi = conf.synthetic_vocab(1000)
    assert wtoi['<EOS>'] == 999 and wtoi['<GO>'] == 998 and wtoi['<UNK>'] == 997 and wtoi['<PAD>'] == -1
    assert itow['0'] == 'w0' and len(itow) == 1000


# ---------------------------------------------------------------------------
# CLI mirror (src/train.py:25-164, src/infer.py:23-74)
# ---------------------------------------------------------------------------
def test_cli_parsers_mirror_reference_flags():
    from comic_b200 import cli
    tp, ip = cli.create_train_parser(), cli.create_infer_parser()
    ours_t = {a.dest: a for a in tp._actions if a.dest != 'help'}
    ours_i = {a.dest: a for a in ip._actions if a.dest != 'help'}
    # known answers (SURVEY.md §8b): every flag of the two reference parsers
    assert len(ours_t) == 39 and len(ours_i) == 14
    assert ours_t['attn_num_heads'].default == 8 and ours_t['scst_beam_size'].default == 7
    assert ours_t['cnn_input_size'].default == '224,224' and ours_t['adam_epsilon'].default == 1e-2
    assert ours_i['infer_beam_size'].default == 3 and ours_i['batch_size_infer'].default == 25
    ref_cli = _reference_cli()
    for ours, fname in ((ours_t, 'train.py'), (ours_i, 'infer.py')):
        ref = ref_cli[fname]
        assert set(ref) == set(ours), (set(ref) ^ set(ours))
        for name, spec in ref.items():
            a = ours[name]
            assert a.type.__name__ == spec['type'], name
            assert (list(a.choices) if a.choices else None) == spec['choices'], name
            if name in PATH_FLAGS:
                continue
            assert a.default == spec['default'], (name, a.default, spec['default'])


def test_cli_config_assembly():
    from comic_b200 import cli
    args = cli.create_train_parser().parse_args(['--train_mode', 'scst', '--cnn_fm_projection', 'none', '--run', '2'])
    c = cli.config_from_train_args(args, n_words=500)
    assert c.batch_size_train == 10 and c.lr_start == 1e-3 and c.max_epoch == 10        # src/train.py:252-262
    assert c.cnn_fm_projection is None and c.rand_seed == 88888888                      # :277-279, :202-207
    assert c.scst_weight_bleu == [0.0, 0.0, 0.0, 2.0] and c.cnn_input_size == [224, 224]


def test_legacy_lr_schedule():
    from comic_b200.train import legacy_lr_reduce
    c = conf.make_config(legacy=True)                   # lr 1e-3 -> 2e-4, halved every 4 epochs (train.py:178-200)
    lr, seen = c.lr_start, []
    for epoch in range(1, 13):
        lr = legacy_lr_reduce(c, epoch, lr)
        seen.append(lr)
    assert seen[2] == 1e-3 and seen[3] == 5e-4 and seen[7] == 2.5e-4 and seen[11] == 2e-4


# ---------------------------------------------------------------------------
# inference driver: result files of src/infer_fn.py:76-184
# ---------------------------------------------------------------------------
class _FakeInferModel(object):
    """Stands in for CaptionModel('infer'): fixed radix ids per batch, attention maps tagged with the batch index."""

    def __init__(self, ids):
        self.ids = ids

    def run_stream(self, batches):
        import numpy as np
        for i, b in enumerate(batches):
            yield [self.ids, np.full((self.ids.shape[0], 8, self.ids.shape[1], 196), float(i), np.float32)]


def test_run_inference_writes_the_reference_result_files(tmp_path):
    """infer_fn.py:107 (whole batches only), :139-156 (image ids, coco json), :165-183 (the three files)."""
    import json
    import numpy as np
    from comic_b200 import inference as inf
    c = conf.make_config(n_words=1000, batch_size_infer=2, infer_beam_size=3, save_attention_maps=True)
    c.infer_save_path = str(tmp_path)
    # radix-256 digits of words 5 and 300, then EOS (257) and padding ids the decoder emits after EOS
    ids = np.array([[0, 5, 1, 44, 257, 257], [1, 44, 0, 5, 257, 257]], np.int32)
    files = ['COCO_val2014_000000000042.jpg', 'COCO_val2014_000000000073.jpg', 'mine@a/b/cat.jpg', 'x_7.jpg',
             'COCO_val2014_000000000099.jpg']                      # 5 files, batch 2 -> 2 whole batches
    batches = [np.zeros((2, 224, 224, 3), np.float32)] * 3
    raw, coco, t = inf.run_inference(c, '/ckpt/model_compact-12345', _FakeInferModel(ids), files, batches)
    assert [e['image_id'] for e in coco] == [42, 73, 'cat', 7]
    assert coco[0]['caption'] == 'w5 w300' and coco[1]['caption'] == 'w300 w5'
    assert raw['checkpoint_number'] == '12345' and raw['beam_size'] == 3
    assert raw['attention']['x_7.jpg'].shape == (8, 6, 196) and raw['attention']['x_7.jpg'][0, 0, 0] == 1.0
    assert json.load(open(tmp_path / 'captions___12345.json')) == coco
    with open(tmp_path / 'outputs___12345.pkl', 'rb') as f:
        assert sorted(pickle.load(f)['captions']) == sorted(files[:4])
    speed = open(tmp_path / 'infer_speed.txt', newline='').read().split('\r\n')
    assert speed[:4] == ['Using GPU #: 0', 'Inference batch size: 2', 'Inference beam size: 3', '']
    assert float(speed[4]) > 0
    # a second checkpoint appends one line and does not repeat the header
    c.save_attention_maps = False
    inf.run_inference(c, '/ckpt/model_compact-20000', _FakeInferModel(ids), files, batches)
    assert len(open(tmp_path / 'infer_speed.txt', newline='').read().split('\r\n')) == 6
    assert not (tmp_path / 'outputs___20000.pkl').exists()
    assert inf.image_id_from_filename('COCO_test2014_000000000123.jpg') == 123
    with pytest.raises(ValueError):
        inf.image_id_from_filename('nodigits.jpg')


def test_unsupported_training_options_are_refused():
    """Options the reference accepts but this path does not build raise instead of silently training differently
    (ADVICE r1): unknown optimisers, the plain 'cider' reward.  (Recurrent dropout, per-variable gradient clipping and
    the momentum-SGD optimiser are built: tests/test_gpu_train.py.)"""
    from comic_b200.train import Trainer
    from comic_b200 import scst as S
    c = conf.make_config(train_mode='decoder', optimiser='rmsprop')
    with pytest.raises(ValueError):                                               # src/model_base.py:881-882
        Trainer(c, {})
    with pytest.raises(NotImplementedError):
        S.CaptionScorer({'document_frequency': {}, 'ref_len': 1}, dict(ciderD=1.0, cider=0.5))
    S.CaptionScorer({'document_frequency': {}, 'ref_len': 1}, dict(ciderD=1.0, cider=0.0, bleu=[0, 0, 0, 2]))


def test_default_dropout_seed_follows_rand_seed_and_step():
    from comic_b200.train import Trainer
    t = Trainer.__new__(Trainer)
    t.c = conf.make_config(train_mode='decoder')
    t.global_step = 0
    s0 = t.dropout_seed()
    t.global_step = 1
    s1 = t.dropout_seed()
    assert s0 != s1 and 0 <= s0 < 2 ** 31 and t.dropout_seed(7) == 7

"""Batches of decoded images of mixed sizes on the device: `comic_preprocess_ragged` against the oracle's
pre-processing run on each image alone (bit-exact), the uniform case against the stacked-tensor kernels, and the
captioning, inference-driver and training paths that take such batches."""
import json

import numpy as np
import pytest

import ragged_ref as R
from _common import comic_config, make_weights

pytestmark = pytest.mark.gpu

# upsampling, downsampling, odd sizes, 1 x 1, 1 x W and H x 1, and one 4000 x 3000 image (36 MB): offsets and the
# per-image pixel indices run far beyond the 224 scale
SIZES = [(100, 80), (640, 480), (480, 640), (333, 517), (1, 1), (1, 57), (45, 1), (4000, 3000), (224, 224)]


@pytest.fixture(scope='module')
def torch_mod():
    import torch
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    return torch


@pytest.fixture(scope='module')
def eng(torch_mod):
    from comic_b200.engine import Engine
    c = comic_config()
    e = Engine(c)
    e.bind_weights(make_weights(c, include_cnn=False), with_cnn=False)
    return e


@pytest.fixture(scope='module')
def mixed():
    return R.mixed_sizes(11, SIZES)


def _dev(eng, ims):
    from comic_b200.engine import pack_images
    return pack_images(ims).to(eng.device)


@pytest.mark.parametrize('out_hw', [(224, 224), (300, 200)])
def test_ragged_eval_bit_exact(eng, mixed, out_hw):
    got = eng.preprocess_eval(_dev(eng, mixed), out_hw).cpu().numpy()
    np.testing.assert_array_equal(got, R.preprocess_eval(mixed, out_hw))


def test_ragged_train_bit_exact(eng, mixed):
    from comic_b200.train import random_crop_flip
    B = len(mixed)
    crop, flip = random_crop_flip(B, rng=np.random.default_rng(5))
    crop[0], crop[1], flip[0], flip[1] = (0, 32), (32, 0), 1, 0      # the corners of the offset range
    got = eng.preprocess_train(_dev(eng, mixed), crop, flip).cpu().numpy()
    np.testing.assert_array_equal(got, R.preprocess_train(mixed, crop, flip))
    with pytest.raises(ValueError):
        eng.preprocess_train(_dev(eng, mixed), np.array([[0, 33]] * B), flip)


def test_uniform_list_equals_the_stacked_kernels(eng, torch_mod):
    from comic_b200.train import random_crop_flip
    torch = torch_mod
    x = np.random.default_rng(3).integers(0, 256, (3, 240, 320, 3), dtype=np.uint8)
    dx = torch.from_numpy(x).to(eng.device)
    for out_hw in ((224, 224), (300, 200)):
        assert torch.equal(eng.preprocess_eval(_dev(eng, list(x)), out_hw), eng.preprocess_eval(dx, out_hw))
    crop, flip = random_crop_flip(3, rng=np.random.default_rng(4))
    assert torch.equal(eng.preprocess_train(_dev(eng, list(x)), crop, flip), eng.preprocess_train(dx, crop, flip))


def test_engine_refuses_what_the_encoder_cannot_read(eng, torch_mod):
    """encode / encode_train read fp32 [B,224,224,3] on the engine's device: uint8 (4x fewer bytes) and host tensors
    are refused instead of being read as if they were; a ragged batch still in host memory is refused too."""
    from comic_b200.engine import pack_images
    torch = torch_mod
    for bad in (torch.zeros((2, 224, 224, 3), dtype=torch.uint8, device=eng.device), torch.zeros((2, 224, 224, 3)),
                np.zeros((2, 224, 224, 3), np.float32)):
        with pytest.raises(ValueError):
            eng.encode(bad)
        with pytest.raises(ValueError):
            eng.encode_train(bad)
    with pytest.raises(ValueError):
        eng.preprocess_eval(pack_images([np.zeros((4, 4, 3), np.uint8)]))


def _stream_batches():
    """9 batches of 8 images whose sizes change batch to batch.  Batches 0 and 1 fill each input slot's buffers;
    batch 2 is larger than 1.25x slot 0's buffer and forces its one growth; the rest fit."""
    rng = np.random.default_rng(21)
    out = []
    for i in range(9):
        sizes = [tuple(int(v) for v in rng.integers(20, 65, 2)) for _ in range(8)]
        if i in (0, 1):
            sizes[0] = (200, 200)
        if i == 2:
            sizes[3] = (300, 300)
        out.append(R.mixed_sizes(100 + i, sizes))
    return out


def test_run_stream_ragged_matches_the_fp32_path(torch_mod):
    from comic_b200.model import CaptionModel
    c = comic_config(infer_max_length=3)
    m = CaptionModel(c, 'infer', weights=make_weights(c))
    batches = _stream_batches()
    want = [tuple(a.copy() for a in m.run(R.preprocess_eval(b))) for b in batches]
    eng = m.engine
    replayed, n = [], 0
    for i, (p, a) in enumerate(m.run_stream(iter(batches))):
        np.testing.assert_array_equal(p, want[i][0], err_msg='batch %d ids' % i)
        np.testing.assert_array_equal(a, want[i][1], err_msg='batch %d attention maps' % i)
        replayed.append(getattr(eng, 'replayed_launches', 0))       # counted after compute(i + 1)
        n += 1
    assert n == len(batches)
    slot0 = m._pipe_slots[2][0]['dev_ragged']
    assert slot0.numel() >= 16 * 8 + 300 * 300 * 3             # grew once, for batch 2
    # slot 0: batch 2 eager (grown buffer), 4 captures, 6 and 8 replay
    assert replayed[5] > replayed[4] and replayed[7] > replayed[6], replayed
    # a list of same-size images takes the ragged path and gives what the stacked uint8 tensor gives
    same = R.mixed_sizes(7, [(240, 320)] * 4)
    p1, a1 = (x.copy() for x in m.run(same))
    p2, a2 = m.run(np.stack(same))
    np.testing.assert_array_equal(p1, p2)
    np.testing.assert_array_equal(a1, a2)


def test_run_inference_with_list_batches(torch_mod, tmp_path):
    from comic_b200 import inference as inf
    from comic_b200.model import CaptionModel
    c = comic_config(infer_max_length=3)
    c.batch_size_infer = 3
    c.save_attention_maps = False
    m = CaptionModel(c, 'infer', weights=make_weights(c))
    rng = np.random.default_rng(8)
    batches = [R.mixed_sizes(30 + s, [tuple(int(v) for v in rng.integers(30, 400, 2)) for _ in range(3)])
               for s in range(2)]
    files = ['COCO_val2014_%012d.jpg' % i for i in range(6)]
    out = {}
    for name, bs in (('lists', batches), ('fp32', [R.preprocess_eval(b) for b in batches])):
        c.infer_save_path = str(tmp_path / name)
        (tmp_path / name).mkdir()
        inf.run_inference(c, 'model_compact-77', m, files, iter(bs))
        out[name] = json.load(open(tmp_path / name / 'captions___77.json'))
    assert len(out['lists']) == 6 and out['lists'] == out['fp32']


def _train_pair(c, W):
    from comic_b200.train import Trainer
    return Trainer(c, W), Trainer(c, W)


def _captions(B, seed):
    rng = np.random.default_rng(seed)
    caps = np.full((B, 9), -1, np.int32)
    for b in range(B):
        n = int(rng.integers(3, 8))
        caps[b, 0], caps[b, 1:n], caps[b, n] = 256, rng.integers(0, 256, n - 1), 257
    return caps


@pytest.mark.parametrize('mode,augment', [('decoder', True), ('cnn_finetune', True), ('decoder', False)])
def test_train_step_on_ragged_pixels(torch_mod, mode, augment):
    """Trainer.step on a ragged uint8 batch = the same step fed the per-image pre-processed fp32 images."""
    torch = torch_mod
    c = comic_config(train_mode=mode, cnn_input_augment=augment, max_step=100)
    W = make_weights(c, seed=5)
    ims = R.mixed_sizes(9, [(120, 90), (333, 517), (480, 640), (64, 64)])
    caps = _captions(len(ims), 2)
    a, b = _train_pair(c, W)
    out = a.step(ims, caps, seed=17, lr=1e-3)
    if augment:
        ref_imgs = R.preprocess_train(ims, out['crop_yx'], out['flip'])
        c2 = np.random.default_rng(17)
        from comic_b200.train import random_crop_flip
        crop, flip = random_crop_flip(len(ims), rng=c2)          # the step's seed reproduces its draws
        np.testing.assert_array_equal(crop, out['crop_yx'])
        np.testing.assert_array_equal(flip, out['flip'])
    else:
        assert 'crop_yx' not in out
        ref_imgs = R.preprocess_eval(ims)
    ref = b.step(b.engine.to_dev(ref_imgs), caps, seed=17, lr=1e-3)
    assert torch.equal(out['loss'], ref['loss'])
    assert torch.equal(a.grads, b.grads) and torch.equal(a.params, b.params)
    if augment:                                           # no seed: the draws come from config.rand_seed's generator
        d1, d2 = a.step(ims, caps, lr=1e-3), a.step(ims, caps, lr=1e-3)
        assert not (np.array_equal(d1['crop_yx'], d2['crop_yx']) and np.array_equal(d1['flip'], d2['flip']))


def test_scst_step_on_ragged_pixels(torch_mod):
    from comic_b200 import scst as S
    torch = torch_mod
    c = comic_config(train_mode='scst', scst_beam_size=3, n_words=1000, max_step=50)
    W = make_weights(c)
    ims = R.mixed_sizes(12, [(200, 150), (37, 513)])
    rng = np.random.default_rng(0)
    refs = [[' '.join('w%d' % w for w in rng.integers(0, 997, size=10)) for _ in range(5)] for _ in ims]
    df = {'document_frequency': S.compute_doc_freq(refs), 'ref_len': len(ims)}
    scorer = S.CaptionScorer(df, dict(ciderD=c.scst_weight_ciderD, bleu=c.scst_weight_bleu))
    a, b = _train_pair(c, W)
    out = S.scst_step(a, scorer, ims, refs, seed=3, lr=1e-3)
    ref = S.scst_step(b, scorer, b.engine.to_dev(R.preprocess_train(ims, out['crop_yx'], out['flip'])), refs, seed=3,
                      lr=1e-3)
    np.testing.assert_array_equal(out['rewards'], ref['rewards'])
    assert torch.equal(out['loss'], ref['loss'])
    assert torch.equal(a.grads, b.grads)

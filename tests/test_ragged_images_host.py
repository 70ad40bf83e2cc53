"""Batches of decoded images of mixed sizes, host side: the packer's layout and its input checks, and the per-image
oracle composition that the GPU tests compare the device pre-processing against."""
import numpy as np
import pytest
import torch

import comic_b200  # noqa: F401  (import shim)
import inception_v1_oracle as I
import ragged_ref as R
from comic_b200.engine import RaggedImages, pack_images


def test_pack_tables_and_offsets():
    ims = R.mixed_sizes(0, [(2, 3), (1, 1), (5, 1), (4, 7)])
    ims[2] = torch.from_numpy(ims[2])                       # host tensors are accepted next to arrays
    r = pack_images(ims)
    assert isinstance(r, RaggedImages) and len(r) == 4
    sizes = [2 * 3 * 3, 3, 5 * 3, 4 * 7 * 3]
    np.testing.assert_array_equal(r.offsets.numpy(), np.r_[0, np.cumsum(sizes)[:-1]])
    np.testing.assert_array_equal(r.hw.numpy(), [[2, 3], [1, 1], [5, 1], [4, 7]])
    assert r.offsets.dtype == torch.int64 and r.hw.dtype == torch.int32
    assert r.nbytes == 16 * 4 + sum(sizes)
    want = np.concatenate([np.asarray(im).reshape(-1) for im in ims])
    np.testing.assert_array_equal(r.data.numpy()[:sum(sizes)], want)
    # one buffer holds the tables, then the pixels: one copy moves the batch
    buf = r._buf.numpy()
    np.testing.assert_array_equal(buf[:32].view(np.int64), r.offsets.numpy())
    np.testing.assert_array_equal(buf[32:64].view(np.int32).reshape(4, 2), r.hw.numpy())
    np.testing.assert_array_equal(buf[64:r.nbytes], want)


def test_pack_reuses_and_grows_the_staging_buffer():
    small = R.mixed_sizes(1, [(4, 4), (3, 5)])
    r = pack_images(small)
    stage = r._buf
    assert stage.numel() == r.nbytes
    r2 = pack_images(small[::-1], stage)
    assert r2._buf is stage
    np.testing.assert_array_equal(r2.hw.numpy(), [[3, 5], [4, 4]])
    r3 = pack_images(small + [np.zeros((1, 2, 3), np.uint8)], stage)       # 6 more bytes + one more table entry
    assert r3._buf.numel() >= (stage.numel() * 5) // 4 and r3._buf.numel() >= r3.nbytes


def test_pack_uniform_list_is_the_stacked_batch():
    x = np.random.default_rng(2).integers(0, 256, (3, 6, 5, 3), dtype=np.uint8)
    r = pack_images(list(x))
    np.testing.assert_array_equal(r.data.numpy()[:x.size], x.reshape(-1))
    np.testing.assert_array_equal(r.offsets.numpy(), [0, 90, 180])


@pytest.mark.parametrize('bad', [
    [np.zeros((4, 4, 3), np.float32)],                     # dtype
    [np.zeros((4, 4), np.uint8)],                          # rank 2
    [np.zeros((1, 4, 4, 3), np.uint8)],                    # rank 4
    [np.zeros((4, 4, 1), np.uint8)],                       # 1 channel
    [np.zeros((4, 4, 4), np.uint8)],                       # 4 channels
    [np.zeros((4, 4, 3), np.uint8), np.zeros((0, 4, 3), np.uint8)],     # empty image
    [np.zeros((4, 0, 3), np.uint8)],
    [[[[0, 0, 0]]]],                                       # not an array
    ['image.jpg'],
    [],                                                    # no images
], ids=['float32', 'rank2', 'rank4', 'c1', 'c4', 'h0', 'w0', 'nested_list', 'path', 'empty'])
def test_pack_rejects(bad):
    with pytest.raises(ValueError):
        pack_images(bad)


def test_pack_rejects_a_tensor_batch():
    with pytest.raises(ValueError):
        pack_images(np.zeros((2, 4, 4, 3), np.uint8))


def test_per_image_oracle_composition():
    """Same-size images: the per-image composition equals the oracle's batched pre-processing (eval and train);
    a 1 x 1 image is its own value everywhere in the crop, and padding is -1 after the standardisation."""
    ims = R.mixed_sizes(3, [(37, 53)] * 3)
    x = np.stack(ims)
    for out_hw in ((224, 224), (300, 200)):
        np.testing.assert_array_equal(R.preprocess_eval(ims, out_hw), I.preprocess_eval(x, out_hw))
    crop = np.array([[0, 32], [17, 5], [32, 0]], np.int32)
    flip = np.array([1, 0, 1], np.uint8)
    np.testing.assert_array_equal(R.preprocess_train(ims, crop, flip), I.preprocess_train(x, crop, flip))
    one = np.full((1, 1, 3), 51, np.uint8)
    got = R.preprocess_eval([one, ims[0]], (300, 200))
    assert got.shape == (2, 300, 200, 3)
    v = (np.float32(51) * np.float32(1 / 255.0) - np.float32(0.5)) * np.float32(2.0)
    np.testing.assert_array_equal(got[0, 22:278], v)
    np.testing.assert_array_equal(got[0, :22], -1.0)
    np.testing.assert_array_equal(got[1], I.preprocess_eval(ims[0][None], (300, 200))[0])


def test_pack_large_batch_over_threads():
    """A batch above the threaded-copy size packs the same bytes as one thread does."""
    from comic_b200 import engine
    ims = R.mixed_sizes(4, [(1000, 1500), (3, 2), (800, 600), (1024, 1024), (7, 9), (600, 800)] * 2)
    assert sum(im.size for im in ims) > engine.PACK_THREADED_BYTES
    r = pack_images(ims)
    np.testing.assert_array_equal(r.data.numpy()[:r.nbytes - 16 * len(ims)],
                                  np.concatenate([im.reshape(-1) for im in ims]))

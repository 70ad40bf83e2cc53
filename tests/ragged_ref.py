"""References for batches of decoded images of mixed sizes: the oracle's pre-processing run on each image alone, which
is what the reference does (it decodes and resizes every file on its own, inception_preprocessing_radix.py:229-235,
270-273), stacked in batch order."""
import numpy as np

import inception_v1_oracle as I


def preprocess_eval(images, out_hw=(224, 224)):
    return np.concatenate([I.preprocess_eval(im[None], out_hw) for im in images])


def preprocess_train(images, crop_yx, flip, out_hw=(224, 224)):
    return np.concatenate([I.preprocess_train(im[None], crop_yx[b:b + 1], flip[b:b + 1], out_hw)
                           for b, im in enumerate(images)])


def mixed_sizes(seed, sizes):
    """Seeded uint8 RGB images, one per (h, w)."""
    rng = np.random.default_rng(seed)
    return [rng.integers(0, 256, (h, w, 3), dtype=np.uint8) for h, w in sizes]

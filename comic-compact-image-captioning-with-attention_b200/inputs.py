"""Host-side input managers (SURVEY.md section 8f-4): the reference's caption side of
common/inputs/manager_image_caption.py -- vocabulary files, word / radix / char tokenisation, shuffling, bucketing by
caption length, padding with <PAD> -- as plain Python iterators of (image paths, int32 captions [B, L]).

What is NOT here: tf.data, JPEG decoding.  Images are produced by a caller-supplied `image_loader(paths)` returning
decoded pixels: a uint8 [B, h, w, 3] array when the images share one size, or a list of uint8 [h, w, 3] arrays of
mixed sizes (as the files of a real dataset are); the device side of the reference's preprocessing then is
`Engine.preprocess_eval` / `Engine.preprocess_train`, which `CaptionModel.run` / `run_stream`, `Trainer.step` and
`scst.scst_step` run themselves on such batches.  With no loader the managers yield paths and captions only.

Reference behaviour reproduced (file:line of common/inputs/manager_image_caption.py):
  * vocabulary: `captions/<pattern.format('itow')>.json`, `...('wtoi')>.json`; `vocab_size = len(itow)` (:98-108);
  * split files `captions/<pattern.format(split)>.txt`, one `filepath,w0 w1 ... wN` per line (:124-131);
  * `max_step = int(len(train) / batch_size_train * max_epoch / accum_grads_step)` (:134-141); the eval split must be a
    multiple of `batch_size_eval` (:144-145), the inference file list of `batch_size_infer` (:118);
  * buckets [11, 13, 15] (coco) / [7, 10, 13] (insta) in words (:83-86), x digits-per-word for radix (:241),
    [45, 55, 70] / [29, 42, 61] for char (:291-295); batches come from
    `bucket_by_sequence_length(boundaries, [batch] * (n + 1), pad_to_bucket_boundary=False)` (:177-183): an example
    goes to bucket #{boundaries <= len}, a bucket is emitted when it holds `batch` examples, padded with <PAD> to the
    longest caption IN THE BATCH;
  * word ids `wtoi.get(w, wtoi['<UNK>'])` (:218-221); radix digits `number_to_base(id, base)` left-padded to the digit
    count of `len(wtoi)`, <GO> = base, <EOS> = base + 1, <PAD> = -1 (:242-255, :271-274); char: the words between
    <GO> and <EOS> joined by spaces, one id per character over ' ' + digits + lowercase, ids from <PAD> upwards
    (:299-326, :347-350);
  * the training list is shuffled with `random.seed(rand_seed)` at start and again after every epoch (:59, :212-227).
The per-word validation perplexity of src/train_fn.py:320-338 is `run_eval_loop`.
"""
import json
import os
import random
import string

import numpy as np

pjoin = os.path.join


def number_to_base(n, base):
    """common/ops.py:25-40: digits of n in `base`, most significant first (0 -> [0])."""
    if base < 2:
        raise ValueError('Base cannot be less than 2.')
    if n == 0:
        return [0]
    sign = -1 if n < 0 else 1
    n = abs(int(n))
    digits = []
    while n:
        digits.append(sign * (n % base))
        n //= base
    return digits[::-1]


def bucket_batches(examples, boundaries, batch_size, pad_value, drop_remainder=True):
    """tf.contrib.data.bucket_by_sequence_length with equal bucket batch sizes and pad_to_bucket_boundary=False.
    `examples`: iterable of (key, int array).  Yields (keys, int32 [batch, longest])."""
    held = [[] for _ in range(len(boundaries) + 1)]
    for key, cap in examples:
        n = len(cap)
        b = sum(1 for x in boundaries if x <= n)
        held[b].append((key, cap))
        if len(held[b]) == batch_size:
            yield _pad_batch(held[b], pad_value)
            held[b] = []
    if not drop_remainder:
        for h in held:
            if h:
                yield _pad_batch(h, pad_value)


def _pad_batch(items, pad_value):
    longest = max(len(c) for _, c in items)
    out = np.full((len(items), longest), pad_value, np.int32)
    for i, (_, c) in enumerate(items):
        out[i, :len(c)] = c
    return [k for k, _ in items], out


class InputManager(object):
    """Word-token manager (manager_image_caption.py:27-228)."""

    def __init__(self, config, is_inference=False, image_loader=None):
        c = self.config = config
        self.is_inference = is_inference
        self.image_loader = image_loader
        s = getattr(c, 'cnn_input_size', None)
        if not (isinstance(s, list) and len(s) == 2 and 0 not in s):
            c.cnn_input_size = [224, 224]            # inception_v1.default_image_size
        c.split_sizes = {}
        self._rng = random.Random(c.rand_seed)
        self._get_vocab()
        pat = c.dataset_file_pattern
        if 'coco' in pat:
            self.buckets = [11, 13, 15]
        elif 'insta' in pat:
            self.buckets = [7, 10, 13]
        else:
            raise ValueError('`dataset_file_pattern` must name a coco or insta dataset (bucket boundaries).')
        if is_inference:
            self.filenames_infer = self._infer_filenames()
            assert len(self.filenames_infer) % c.batch_size_infer == 0
            c.split_sizes['infer'] = len(self.filenames_infer)
        else:
            self.data = {sp: self._read_split(sp) for sp in ('train', 'valid')}
            for sp in self.data:
                c.split_sizes[sp] = len(self.data[sp])
            gs = getattr(c, 'accum_grads_step', 1)
            c.max_step = int(len(self.data['train']) / c.batch_size_train * c.max_epoch / gs)
            assert len(self.data['valid']) % c.batch_size_eval == 0

    # ---- files ----
    def _get_vocab(self):
        c = self.config
        if '{}' not in c.dataset_file_pattern:
            raise ValueError('`dataset_file_pattern` must have `{}`.')
        with open(pjoin(c.dataset_dir, 'captions', c.dataset_file_pattern.format('itow') + '.json')) as f:
            c.itow = json.load(f)
        with open(pjoin(c.dataset_dir, 'captions', c.dataset_file_pattern.format('wtoi') + '.json')) as f:
            c.wtoi = json.load(f)
        c.vocab_size = len(c.itow)

    def _read_split(self, split):
        c = self.config
        with open(pjoin(c.dataset_dir, 'captions', c.dataset_file_pattern.format(split) + '.txt')) as f:
            rows = [l.strip().split(',') for l in f if l.strip()]
        return [[r[0], r[1].split(' ')] for r in rows]

    def _infer_filenames(self):
        c = self.config
        if 'coco' in c.infer_set:
            coco_set = 'test2014' if c.infer_set == 'coco_test' else 'val2014'
            if coco_set == 'val2014':
                c.batch_size_infer = 61
            return [pjoin(c.dataset_dir, coco_set, f) for f in sorted(os.listdir(pjoin(c.dataset_dir, coco_set)))]
        name = {'test': 'filenames_test.txt', 'valid': 'filenames_valid.txt'}[c.infer_set]
        with open(pjoin(c.dataset_dir, 'captions', name)) as f:
            return [l.strip() for l in f if l.strip()]

    # ---- tokenisation ----
    def encode(self, words):
        """One caption (list of words incl. <GO> / <EOS>) -> int32 ids."""
        w = self.config.wtoi
        return np.array([w.get(x, w['<UNK>']) for x in words], np.int32)

    # ---- iterators ----
    def examples(self, split, epochs=None):
        """(path, ids) in the reference's order: the training list shuffled before every epoch."""
        c = self.config
        data = self.data[split]
        train = split == 'train'
        e = 0
        while epochs is None or e < epochs:
            if train:
                self._rng.shuffle(data)
            for path, words in data:
                yield pjoin(c.dataset_dir, path), self.encode(words)
            e += 1

    def batches(self, split, epochs=None):
        """Bucketed batches: (images or paths, captions int32 [B, L])."""
        c = self.config
        bs = c.batch_size_train if split == 'train' else c.batch_size_eval
        for paths, caps in bucket_batches(self.examples(split, epochs), self.buckets, bs, c.wtoi['<PAD>']):
            yield (self.image_loader(paths) if self.image_loader else paths), caps

    def infer_batches(self):
        c = self.config
        fn = self.filenames_infer
        for i in range(0, len(fn), c.batch_size_infer):
            paths = fn[i:i + c.batch_size_infer]
            yield (self.image_loader(paths) if self.image_loader else paths), paths


class InputManager_Radix(InputManager):
    """Radix-token manager (manager_image_caption.py:231-281)."""

    def __init__(self, config, is_inference=False, image_loader=None):
        super(InputManager_Radix, self).__init__(config, is_inference, image_loader)
        c = self.config
        self.max_word_len = len(number_to_base(len(c.wtoi), c.radix_base))
        self.buckets = [b * self.max_word_len for b in self.buckets]
        assert c.wtoi['<PAD>'] == -1
        self.radix_wtoi = {}
        for k, v in c.wtoi.items():
            if k == '<GO>':
                idx = [c.radix_base]
            elif k == '<EOS>':
                idx = [c.radix_base + 1]
            elif k == '<PAD>':
                idx = [-1]
            else:
                d = number_to_base(v, c.radix_base)
                idx = [0] * (self.max_word_len - len(d)) + d
            self.radix_wtoi[k] = idx

    def encode(self, words):
        r = self.radix_wtoi
        return np.concatenate([r.get(x, r['<UNK>']) for x in words]).astype(np.int32)


class InputManager_Char(InputManager):
    """Character-token manager (manager_image_caption.py:284-357)."""

    def __init__(self, config, is_inference=False, image_loader=None):
        super(InputManager_Char, self).__init__(config, is_inference, image_loader)
        pat = self.config.dataset_file_pattern
        self.buckets = [45, 55, 70] if 'coco' in pat else [29, 42, 61]

    def _get_vocab(self):
        c = self.config
        if '{}' not in c.dataset_file_pattern:
            raise ValueError('`dataset_file_pattern` must have `{}`.')
        with open(pjoin(c.dataset_dir, 'captions', c.dataset_file_pattern.format('wtoi') + '.json')) as f:
            pad_value = json.load(f)['<PAD>']
        ctoi, itoc = {}, {}
        idx = pad_value
        for ch in ['<PAD>', ' '] + list(string.digits + string.ascii_lowercase):
            ctoi[ch] = idx
            itoc[idx] = ch
            idx += 1
        # the reference numbers <GO> / <EOS> by table SIZE (= last id + 2 with <PAD> = -1), not by the running index
        ctoi['<GO>'] = len(ctoi)
        ctoi['<EOS>'] = len(ctoi)
        itoc[len(itoc)] = '<GO>'
        itoc[len(itoc)] = '<EOS>'
        c.itow, c.wtoi, c.vocab_size = itoc, ctoi, len(itoc)

    def encode(self, words):
        w = self.config.wtoi
        body = [w[ch] for ch in ' '.join(words[1:-1])]
        return np.array([w['<GO>']] + body + [w['<EOS>']], np.int32)


def get_input_manager(config, is_inference=False, image_loader=None):
    """token_type -> manager class (src/train.py / src/infer.py pick the class the same way)."""
    cls = {'word': InputManager, 'radix': InputManager_Radix, 'char': InputManager_Char}[config.token_type]
    return cls(config, is_inference, image_loader)


def run_eval_loop(model, batches, num_batches=None):
    """src/train_fn.py:320-338: mean of the per-batch teacher-forced log-perplexities, exponentiated.
    `model`: CaptionModel in 'eval' (or 'train') mode; `batches`: iterable of (images, captions)."""
    ppl = []
    for i, (images, caps) in enumerate(batches):
        if num_batches is not None and i >= num_batches:
            break
        ppl.append(float(model.eval_step(images, caps)))
    if not ppl:
        raise ValueError('run_eval_loop: no batches')
    return float(np.exp(np.mean(ppl)))

"""The reference's inference driver (`src/infer_fn.py:76-184`, `run_inference`) on the CUDA engine.

Same result files, same keys, same text:

    <infer_save_path>/captions___<ckpt>.json   [{"image_id": ..., "caption": ...}, ...]     (infer_fn.py:173-174)
    <infer_save_path>/outputs___<ckpt>.pkl     raw_outputs incl. attention maps, only with
                                               `save_attention_maps`                         (infer_fn.py:169-171)
    <infer_save_path>/infer_speed.txt          header once, then one images/s line per run   (infer_fn.py:175-183)

The reference pulls batches out of its in-graph `InputManager`; the dataset readers are out of scope here
(DESIGN.md §7), so the caller hands over `filenames` and an iterable of image batches in file order: `[B, 224, 224, 3]`
fp32 (host or device), raw uint8 `[B, H, W, 3]` pixels, or a list of uint8 `[h, w, 3]` images of mixed sizes (pre-processed
on the device).  Batches go through `CaptionModel.run_stream`, i.e. the H2D copy of batch i+1 and the D2H copy
of batch i-1 overlap the compute of batch i, where the reference issues one blocking `sess.run` per batch
(infer_fn.py:129-130).  As in the reference only whole batches are decoded (`num_batches = int(n / batch_size)`,
infer_fn.py:107) and every file must end up with exactly one caption (infer_fn.py:160-163).
"""
from __future__ import annotations

import json
import os
import pickle
import re
import time

from .scst import id_to_caption

pjoin = os.path.join

P_COCO = re.compile(r'(?<=_)\d+')      # infer_fn.py:32
P_CKPT = re.compile(r'\d+')            # infer_fn.py:33


def image_id_from_filename(f):
    """infer_fn.py:139-148: '<name>@...' files keep their base name, COCO files give the integer after '_'."""
    image_id = f.replace('.jpg', '')
    if '@' in image_id:
        return os.path.basename(image_id)
    found = P_COCO.findall(image_id)
    if isinstance(found, list) and len(found) > 0:
        return int(found[0])
    raise ValueError('Expected `image_id` to be list or string, saw `{}`'.format(type(found)))


def write_result_files(c, ckpt_num, raw_outputs, coco_json, images_per_second):
    """The three artefacts `evaluate_model` and the COCO scorers read (src/infer_fn.py:165-184), in the reference's
    formats: `captions___<ckpt>.json` (list of {image_id, caption}), `outputs___<ckpt>.pkl` (only with
    `save_attention_maps`) and `infer_speed.txt` -- a three-line header written once per directory, then one
    images-per-second figure appended per run, all separated by CRLF."""
    out_dir = c.infer_save_path
    if c.save_attention_maps:
        with open(pjoin(out_dir, 'outputs___%s.pkl' % ckpt_num), 'wb') as f:
            pickle.dump(raw_outputs, f, pickle.HIGHEST_PROTOCOL)
    with open(pjoin(out_dir, 'captions___%s.json' % ckpt_num), 'w') as f:
        json.dump(coco_json, f)
    speed_file = pjoin(out_dir, 'infer_speed.txt')
    header = '' if os.path.isfile(speed_file) else '\r\n'.join(
        ['Using GPU #: %s' % c.gpu, 'Inference batch size: %s' % c.batch_size_infer,
         'Inference beam size: %s' % c.infer_beam_size, ''])
    with open(speed_file, 'a') as f:
        f.write('%s\r\n%s' % (header, images_per_second))


def run_inference(config, curr_ckpt_path, model, filenames, batches):
    """infer_fn.py:76-184 with the model and the input batches supplied by the caller.

    model      `CaptionModel(config, 'infer', ...)` (anything with `run_stream(batches)` yielding
               `[word_ids [B, T], attn_maps [B, H, T, M]]` per batch)
    filenames  image files in batch order (`InputManager.filenames_infer`)
    batches    iterable of image batches of `config.batch_size_infer` images (tensors / arrays, or lists of
               per-image uint8 [h, w, 3] arrays of mixed sizes)
    Returns (raw_outputs, coco_json, seconds)."""
    c = config
    ckpt_dir, ckpt_file = os.path.split(curr_ckpt_path)
    ckpt_num = P_CKPT.findall(ckpt_file)[0]
    batch_size = c.batch_size_infer
    filenames = list(filenames)
    num_batches = int(len(filenames) / batch_size)

    raw_outputs = dict(captions={}, attention={}, image_ids={}, beam_size=c.infer_beam_size,
                       max_caption_length=c.infer_max_length, checkpoint_path=curr_ckpt_path,
                       checkpoint_number=ckpt_num)
    coco_json = []
    captions = []

    def limited():
        for step, b in enumerate(batches):
            if step >= num_batches:
                return
            yield b

    # the maps are only ever DUMPED with `save_attention_maps` (infer_fn.py:169-171): without it the decode loop keeps no
    # alignment history and nothing but the word ids crosses PCIe
    model.collect_attention_maps = bool(c.save_attention_maps)
    start_time = time.time()
    step = -1
    for step, (word_ids, attn_maps) in enumerate(model.run_stream(limited())):
        captions = id_to_caption(word_ids, c)
        batch_filenames = filenames[step * batch_size:(step + 1) * batch_size]
        for i, f in enumerate(batch_filenames):
            image_id = image_id_from_filename(f)
            raw_outputs['captions'][f] = captions[i]
            # a yielded batch lives in a rotating pinned buffer: keep a copy (the reference gets fresh arrays).
            # The reference keeps every map in memory and only DUMPS them with `save_attention_maps`; here they are
            # not kept at all without it (0.4 MB per image at 60 steps).
            raw_outputs['attention'][f] = attn_maps[i].copy() if c.save_attention_maps else None
            raw_outputs['image_ids'][f] = image_id
            coco_json.append(dict(image_id=image_id, caption=str(captions[i])))
    print("\nExample captions:\n{}\n".format("\n".join(captions[:3])))
    t = time.time() - start_time

    if step + 1 == num_batches:
        filenames = filenames[:num_batches * batch_size]
    # every image exactly once in every result container (the reference's three asserts, infer_fn.py:160-163)
    n_images = len(filenames)
    if not (len(set(filenames)) == n_images == len(coco_json) == len(raw_outputs['image_ids'])):
        raise AssertionError('inference results do not cover the file list exactly once: %d files, %d captions, %d ids'
                             % (n_images, len(coco_json), len(raw_outputs['image_ids'])))
    write_result_files(c, ckpt_num, raw_outputs, coco_json, n_images / t)
    print("\nINFO: Inference completed. Time taken: {:4.2f} mins\n".format(t / 60))
    return raw_outputs, coco_json, t

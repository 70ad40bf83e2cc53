"""Captioning throughput from decoded images of one size and of mixed sizes, through CaptionModel.run_stream.

    python scripts/bench_ragged_images.py [--reps 3] [--steps 10] [--out profiles/ragged_images_bench.json]

COMIC-256 (radix, beam 3, tied projection), 512 images a batch, seeded random weights, no attention maps returned
(the production setting without `save_attention_maps`).  Batches start in host memory, as an image decoder hands them
over.  Arms:
  uniform_224     uint8 [512, 224, 224, 3] pinned tensors: the end-to-end arm of bench.py
  uniform_640x480 uint8 [512, 480, 640, 3] pinned tensors: one common camera size, 6x the bytes of 224 x 224
  coco_mix        lists of 512 [h, w, 3] arrays of seeded COCO-like sizes (640 x 480, 480 x 640, 640 x 427, 500 x 375,
                  612 x 612, 427 x 640 and a few odd sizes): packed on the host, one copy, one pre-processing launch
  uniform_224_list  the uniform_224 images as lists: the ragged path on the same bytes as the first arm
Each arm reports captions/s (host clock around `steps` batches that ends in a device synchronise, after a warm-up that
takes every input slot through its eager call, CUDA-graph capture and first replay), the pre-processing kernel time
(CUDA events around 20 launches on the device-resident batch), the host pack time per batch (lists only: pack_images
into a reused pinned buffer) and the bytes one batch copies host -> device.  Two batches of each arm alternate, and
the arms are timed alternately, `reps` times each.  The card's name and power limit are read in the same call.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import comic_b200  # noqa: E402,F401  (import shim)
from comic_b200 import configuration as conf  # noqa: E402
from comic_b200 import weights as wts  # noqa: E402
from comic_b200 import engine  # noqa: E402
from comic_b200.engine import Engine, pack_images  # noqa: E402
from comic_b200.model import CaptionModel  # noqa: E402

B = 512
COCO_SIZES = [(480, 640), (640, 480), (427, 640), (375, 500), (612, 612), (640, 427)]
ODD_SIZES = [(333, 517), (100, 80), (1024, 768), (256, 341)]


def card():
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:                                      # noqa: BLE001
        out = 'unknown (%s)' % e
    return out


def coco_mix(rng):
    """Mostly the common COCO sizes, one image in 32 of an odd size."""
    out = []
    for _ in range(B):
        pool = ODD_SIZES if rng.random() < 1 / 32 else COCO_SIZES
        h, w = pool[int(rng.integers(len(pool)))]
        out.append(rng.integers(0, 256, (h, w, 3), dtype=np.uint8))
    return out


def main():
    p = argparse.ArgumentParser()
    p.add_argument('--reps', type=int, default=3)
    p.add_argument('--steps', type=int, default=10)
    p.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'ragged_images_bench.json'))
    a = p.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit('bench_ragged_images.py needs a CUDA device')
    c = conf.make_config()
    c.infer_beam_size, c.batch_size_infer = 3, B
    W = wts.init_weights(c, seed=c.rand_seed, cnn_init='he')
    rng = np.random.default_rng(2026)
    arms = {
        'uniform_224': [torch.from_numpy(rng.integers(0, 256, (B, 224, 224, 3), dtype=np.uint8)).pin_memory()
                        for _ in range(2)],
        'uniform_640x480': [torch.from_numpy(rng.integers(0, 256, (B, 480, 640, 3), dtype=np.uint8)).pin_memory()
                            for _ in range(2)],
        'coco_mix': [coco_mix(rng) for _ in range(2)],
    }
    arms['uniform_224_list'] = [list(t.numpy()) for t in arms['uniform_224']]
    res = dict(card=card(), torch=torch.__version__, host_cpus=os.cpu_count(), pack_threads=engine.PACK_THREADS,
               images=B, beam=3,
               config='COMIC-256 (radix, R=512, tied, add_LN, 8 heads), no attention maps returned',
               timing='CaptionModel.run_stream from host memory; host clock around `steps` batches ending in a '
                      'device synchronise', arms={})

    models = {}

    def run(name, n):
        model, batches = models[name], arms[name]
        got = 0
        for out in model.run_stream(batches[j % 2] for j in range(n)):
            got += int(out[0].shape[0])
        assert got == n * B

    for name, batches in arms.items():
        # one engine per arm: each keeps its own input slots and CUDA graphs while the arms alternate
        eng = Engine(c)
        eng.bind_weights(W)
        model = models[name] = CaptionModel(c, 'infer', engine=eng)
        model.collect_attention_maps = False
        r = res['arms'][name] = dict(runs=[])
        if isinstance(batches[0], list):
            r['sizes'] = sorted({'%dx%d' % im.shape[:2] for b in batches for im in b})
            threads, stage = engine.PACK_THREADS, None
            for key, engine.PACK_THREADS in (('host_pack_ms_1_thread', 1), ('host_pack_ms', threads)):
                ms = []
                for _ in range(5):
                    t0 = time.perf_counter()
                    packed = pack_images(batches[0], stage)
                    ms.append((time.perf_counter() - t0) * 1e3)
                    stage = packed._buf
                r[key] = round(float(np.median(ms)), 3)
            r['h2d_bytes'] = packed.nbytes
            dev = packed.to(eng.device)
        else:
            r['sizes'] = ['%dx%d' % tuple(batches[0].shape[1:3])]
            r['host_pack_ms'] = 0.0
            r['h2d_bytes'] = batches[0].numel()
            dev = batches[0].to(eng.device)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        eng.preprocess_eval(dev)
        ev0.record()
        for _ in range(20):
            eng.preprocess_eval(dev)
        ev1.record()
        torch.cuda.synchronize()
        r['preprocess_kernel_ms'] = round(ev0.elapsed_time(ev1) / 20, 4)
        del dev
        run(name, 6)                                          # per slot: eager, capture, first replay
        torch.cuda.synchronize()
        print(name, {k: v for k, v in r.items() if k != 'sizes'}, flush=True)
    for rep in range(a.reps):
        for name in arms:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            run(name, a.steps)
            torch.cuda.synchronize()
            dt = (time.perf_counter() - t0) / a.steps
            x = dict(captions_per_s=round(B / dt, 1), ms_per_batch=round(dt * 1e3, 3))
            res['arms'][name]['runs'].append(x)
            print(rep, name, x, flush=True)
    for r in res['arms'].values():
        r['captions_per_s_median'] = float(np.median([x['captions_per_s'] for x in r['runs']]))
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, 'w') as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == '__main__':
    main()

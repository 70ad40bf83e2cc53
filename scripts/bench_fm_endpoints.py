"""Decode and training throughput at three attention end points (`--cnn_fm_attention`) on one GPU.

    python scripts/bench_fm_endpoints.py [--reps 3] [--steps 10] [--out profiles/fm_endpoints_bench.json]

Mixed_4f (the default: 14 x 14 x 832), Mixed_4c (14 x 14 x 512) and Mixed_5b (7 x 7 x 832).  Inference: COMIC-256
(radix, beam 3, tied projection) with seeded random weights at 512 and 25 images: the decoder part of a batch
(project_fm + rnn_init + decode_beam) on feature maps resident on the device, replayed as one CUDA graph
(Engine.graphed), timed with a host clock around `steps` replays that end in a device synchronise.  The encoder runs the
same InceptionV1 layers whatever the end point, so it is left out.  Random weights end beams at different steps for
different end points, so the executed step count and the time per step are reported too.  Training: train_mode=decoder
and train_mode=cnn_finetune at batch 32 as scripts/bench_train.py runs them (T = 41 radix steps with every row full
length, seeded dropout, Adam), device-timed with CUDA events.  The end points are timed alternately, `reps` times each,
to show the spread.  The card's name and power limit are read in the same call.
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
from comic_b200.engine import Engine, executed_steps  # noqa: E402
from comic_b200.model import number_to_base  # noqa: E402

BEAM = 3
ENDPOINTS = ('Mixed_4f', 'Mixed_4c', 'Mixed_5b')


def card():
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:                                      # noqa: BLE001
        out = 'unknown (%s)' % e
    return out


class Arm(object):
    def __init__(self, torch, endpoint, B, seed=0):
        c = conf.make_config(cnn_fm_attention=endpoint)
        self.eng = eng = Engine(c)
        eng.bind_weights(wts.init_weights(c, seed=1234, include_cnn=False), with_cnn=False)
        self.T = c.infer_max_length * len(number_to_base(len(c.wtoi), c.radix_base))   # src/model_base.py:709-714
        g = torch.Generator().manual_seed(seed)
        d = eng.dims
        self.fm = torch.rand((B, d.M, d.C), generator=g).to(eng.device)
        self.emb = torch.rand((B, d.E), generator=g).to(eng.device)
        self.B = B

    def step(self):
        eng = self.eng

        def run(fm, emb):
            keys, values = eng.project_fm(fm)
            c0, h0 = eng.rnn_init(emb)
            return eng.decode_beam(keys, values, c0, h0, BEAM, 0.0, self.T, want_attn=False)
        return eng.graphed('bench_fm', run, self.fm, self.emb)

    def time(self, torch, steps):
        r = self.step()
        torch.cuda.synchronize()
        T = executed_steps(r['T'])
        t0 = time.perf_counter()
        for _ in range(steps):
            self.step()
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / steps
        return dict(captions_per_s=round(self.B / dt, 1), ms_per_batch=round(dt * 1e3, 3), steps=T,
                    ms_per_step=round(dt * 1e3 / max(T, 1), 4))


class TrainArm(object):
    def __init__(self, torch, endpoint, mode, B=32):
        from comic_b200.train import Trainer
        c = conf.make_config(cnn_fm_attention=endpoint, train_mode=mode, batch_size_train=B, max_step=100000)
        self.tr = Trainer(c, wts.init_weights(c, seed=c.rand_seed, cnn_init='he'))
        g = torch.Generator().manual_seed(100)
        self.images = torch.empty((B, 224, 224, 3)).uniform_(-1, 1, generator=g).to(self.tr.engine.device)
        rng = np.random.default_rng(0)
        self.caps = np.concatenate([np.full((B, 1), 256), rng.integers(0, 256, size=(B, 40)), np.full((B, 1), 257)],
                                   axis=1).astype(np.int32)       # L = 42 -> T = 41, mask all ones
        self.i = 0

    def step(self):
        self.i += 1
        return self.tr.step(self.images, self.caps, None, seed=1000 + self.i)

    def time(self, torch, steps):
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        ev0.record()
        for _ in range(steps):
            out = self.step()
        ev1.record()
        torch.cuda.synchronize()
        ms = ev0.elapsed_time(ev1) / steps
        return dict(steps_per_s=round(1e3 / ms, 2), ms_per_step=round(ms, 3), xe=round(float(out['loss'][1]), 5))


def main():
    p = argparse.ArgumentParser()
    p.add_argument('--reps', type=int, default=3)
    p.add_argument('--steps', type=int, default=10)
    p.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'fm_endpoints_bench.json'))
    a = p.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit('bench_fm_endpoints.py needs a CUDA device')
    res = dict(card=card(), torch=torch.__version__, beam=BEAM, config='COMIC-256 (radix, R=512, tied, add_LN, 8 heads)',
               timing='decoder of one batch (project_fm + rnn_init + decode_beam) as a replayed CUDA graph',
               training='batch 32, T = 41, Adam, seeded dropout', arms={}, train={})
    arms = {}
    for B in (512, 25):
        for ep in ENDPOINTS:
            arm = arms[(ep, B)] = Arm(torch, ep, B)
            for _ in range(3):                                  # eager, capture, replay
                arm.step()
            res['arms']['%s_b%d' % (ep, B)] = dict(runs=[])
    for rep in range(a.reps):
        for B in (512, 25):
            for ep in ENDPOINTS:
                r = arms[(ep, B)].time(torch, a.steps)
                res['arms']['%s_b%d' % (ep, B)]['runs'].append(r)
                print(rep, ep, B, r, flush=True)
    del arms
    for mode in ('decoder', 'cnn_finetune'):
        trains = {}
        for ep in ENDPOINTS:
            arm = trains[ep] = TrainArm(torch, ep, mode)
            for _ in range(3):                                  # eager, capture, replay
                arm.step()
            res['train']['%s_%s' % (mode, ep)] = dict(runs=[])
        for rep in range(a.reps):
            for ep in ENDPOINTS:
                r = trains[ep].time(torch, a.steps)
                res['train']['%s_%s' % (mode, ep)]['runs'].append(r)
                print(rep, mode, ep, r, flush=True)
        del trains
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, 'w') as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == '__main__':
    main()

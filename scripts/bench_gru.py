"""Decode throughput of the GRU cell against the LSTM cell on one GPU.

    python scripts/bench_gru.py [--reps 3] [--steps 10] [--out profiles/gru_bench.json]

COMIC-256 (radix, beam 3) decoder with seeded random weights at 512 and 25 images: the decoder part of a batch
(project_fm + rnn_init + decode_beam) on feature maps resident on the device, replayed as one CUDA graph
(Engine.graphed), timed with a host clock around `steps` replays that end in a device synchronise.  The two cells
are timed alternately, `reps` times each, to show the spread.  The per-class kernel time of one eager batch
(profile_read, outside the timed region) goes beside each number.  Random weights end beams at different steps for
the two cells, so the executed step count and the time per step are reported too.  Training: train_mode=decoder at batch
32 as scripts/bench_train.py runs it (frozen-CNN encoder forward, teacher-forced forward + backward over T = 41 radix
steps with every row full length, seeded dropout, Adam; the step replayed as a CUDA graph), device-timed with CUDA
events, the two cells alternately.  The card's name and power limit are read in the same call.
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
from comic_b200.engine import Engine, KERNEL_TAGS, executed_steps  # noqa: E402
from comic_b200.model import number_to_base  # noqa: E402

BEAM = 3


def card():
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:                                      # noqa: BLE001
        out = 'unknown (%s)' % e
    return out


class Arm(object):
    def __init__(self, torch, cell, B, seed=0):
        c = conf.make_config(rnn_name=cell)
        self.eng = eng = Engine(c)
        eng.bind_weights(wts.init_weights(c, seed=1234, include_cnn=False), with_cnn=False)
        self.T = c.infer_max_length * len(number_to_base(len(c.wtoi), c.radix_base))   # src/model_base.py:709-714
        g = torch.Generator().manual_seed(seed)
        d = eng.dims
        self.fm = torch.rand((B, d.M, d.C), generator=g).to(eng.device)
        self.emb = torch.rand((B, d.E), generator=g).to(eng.device)
        self.B, self.cell = B, cell

    def step(self):
        eng = self.eng

        def run(fm, emb):
            keys, values = eng.project_fm(fm)
            c0, h0 = eng.rnn_init(emb)
            return eng.decode_beam(keys, values, c0, h0, BEAM, 0.0, self.T, want_attn=False)
        return eng.graphed('bench_gru', run, self.fm, self.emb)

    def breakdown(self, torch):
        eng = self.eng
        eng.profile_enable(KERNEL_TAGS)
        r = self.step()
        torch.cuda.synchronize()
        table = {t: round(eng.profile_read(t)[0], 4) for t in KERNEL_TAGS}
        eng.profile_enable([])
        table = {t: v for t, v in table.items() if v > 0}
        return table, executed_steps(r['T'])

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
    def __init__(self, torch, cell, B=32):
        from comic_b200.train import Trainer
        c = conf.make_config(rnn_name=cell, train_mode='decoder', batch_size_train=B, max_step=100000)
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
            self.step()
        ev1.record()
        torch.cuda.synchronize()
        ms = ev0.elapsed_time(ev1) / steps
        return dict(steps_per_s=round(1e3 / ms, 2), ms_per_step=round(ms, 3))


def main():
    p = argparse.ArgumentParser()
    p.add_argument('--reps', type=int, default=3)
    p.add_argument('--steps', type=int, default=10)
    p.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'gru_bench.json'))
    a = p.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit('bench_gru.py needs a CUDA device')
    res = dict(card=card(), torch=torch.__version__, beam=BEAM, config='COMIC-256 (radix, R=512, tied, add_LN, 8 heads)',
               timing='decoder of one batch (project_fm + rnn_init + decode_beam) as a replayed CUDA graph',
               training='train_mode=decoder, batch 32, T = 41, Adam, CUDA-graph replay', arms={}, train={})
    arms = {}
    for B in (512, 25):
        for cell in ('LSTM', 'GRU'):
            arm = arms[(cell, B)] = Arm(torch, cell, B)
            for _ in range(3):                                  # eager, capture, replay
                arm.step()
            torch.cuda.synchronize()
            table, T = arm.breakdown(torch)
            res['arms']['%s_b%d' % (cell, B)] = dict(kernel_ms_one_batch=table, steps=T, runs=[])
    for rep in range(a.reps):
        for B in (512, 25):
            for cell in ('LSTM', 'GRU'):
                r = arms[(cell, B)].time(torch, a.steps)
                res['arms']['%s_b%d' % (cell, B)]['runs'].append(r)
                print(rep, cell, B, r, flush=True)
    trains = {}
    for cell in ('LSTM', 'GRU'):
        arm = trains[cell] = TrainArm(torch, cell)
        for _ in range(3):                                      # eager, capture, replay
            arm.step()
        res['train'][cell] = dict(runs=[])
    for rep in range(a.reps):
        for cell in ('LSTM', 'GRU'):
            r = trains[cell].time(torch, a.steps)
            res['train'][cell]['runs'].append(r)
            print(rep, 'train', cell, r, flush=True)
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, 'w') as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == '__main__':
    main()

#!/usr/bin/env python
"""bench.py -- captions/sec of the COMIC caption-decoding hot path on B200.

    python bench.py --gpus N --steps K --warmup W            # our CUDA path
    python bench.py --impl reference --gpus N --steps K ...   # the reference's CPU path (NumPy oracle)
    python bench.py ... --dump-outputs DIR                    # + the last timed step's outputs as DIR/<name>.npy

A "step" = one pass of the hot path over one batch of synthetic images on every
rank: InceptionV1 encode -> key projection -> rnn init -> 60-step beam-3 decode
(COMIC-256, radix tokens, max_it = infer_max_length 30 x 2 digits) -> gather_tree
+ top-beam attention maps.  Images are sharded across ranks with no collective
(weak scaling: --batch images per GPU).  `value` times the K steps with inputs
resident in HBM; `e2e` times the same K steps through the public API
(`CaptionModel.run_stream`, the pipelined inference loop) from pinned HOST images,
host<->device copies of every batch included.
Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, 'oracle')):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402

METRIC = 'captions/sec COMIC-256 beam-3'          # --workload word reports METRIC_WORD instead
METRIC_WORD = 'captions/sec baseline word model (V=10,000, no fm projection, 1 head) beam-3'
UNIT = 'captions/s'


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--batch', type=int, default=512, help='images per GPU per step')
    ap.add_argument('--beam', type=int, default=3)
    ap.add_argument('--workload', default='comic256', choices=['comic256', 'word'])
    ap.add_argument('--ref-batch', type=int, default=32, help='images per step of the CPU reference arm')
    ap.add_argument('--cpu-sample', type=int, default=96, help='images of the cpu_baseline sample')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-train', action='store_true', help='skip the train block (BASELINE.json configs 3-5)')
    ap.add_argument('--train-steps', type=int, default=10)
    ap.add_argument('--precision', default='split', choices=['f32', 'split', 'fast'],
                    help='engine arithmetic mode (include/comic_b200.h comic_set_precision)')
    ap.add_argument('--opt', action='append', default=[], help='engine tunable name=value (Engine.set_option)')
    ap.add_argument('--breakdown', action='store_true', help='also print a per-kernel-class time table to stderr')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write the decode outputs of the last timed step to DIR/<name>.npy (rank 0; see beam_outputs)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'ours':
        ap.error('--dump-outputs writes what the CUDA path computed (--impl ours)')
    return args


def make_config(workload):
    import comic_b200  # noqa: F401
    from comic_b200 import configuration as conf
    if workload == 'comic256':
        return conf.make_config()                       # COMIC-256 defaults, V=258, 60 radix steps
    return conf.make_config(token_type='word', cnn_fm_projection='none', attn_num_heads=1, n_words=10000)


def workload_name(workload, batch, beam, c):
    steps = c.infer_max_length * (2 if c.token_type == 'radix' else 1)
    if workload == 'comic256':
        return ('COMIC-256 (radix-256, 8-head add_LN softmax attention, tied projection) beam-%d, %d synthetic '
                '224x224 images/GPU/step, encoder + %d decode steps' % (beam, batch, steps))
    return ('baseline word model (V=10000, fm_projection none, 1 head) beam-%d, %d synthetic 224x224 images/GPU/step, '
            'encoder + %d decode steps' % (beam, batch, steps))


# ---------------------------------------------------------------------------
# clocks sampler (NVML)
# ---------------------------------------------------------------------------
class ClockSampler(object):
    REASONS = {0x1: 'gpu_idle', 0x2: 'applications_clocks_setting', 0x4: 'sw_power_cap', 0x8: 'hw_slowdown',
               0x10: 'sync_boost', 0x20: 'sw_thermal_slowdown', 0x40: 'hw_thermal_slowdown',
               0x80: 'hw_power_brake_slowdown', 0x100: 'display_clock_setting'}

    def __init__(self, index):
        self.samples, self.reasons = [], set()
        self.max_mhz = None
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in self.REASONS.items():
                    if r & bit and name != 'gpu_idle':
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.02)

    def start(self):
        if self.nv is not None:
            self._stop.clear()
            self._thr = threading.Thread(target=self._run, daemon=True)
            self._thr.start()

    def stop(self):
        if self._thr is not None:
            self._stop.set()
            self._thr.join()
            self._thr = None

    def summary(self):
        if not self.samples:
            return {'sm_mhz': None, 'sm_max_mhz': self.max_mhz, 'reasons': sorted(self.reasons)}
        return {'sm_mhz': float(np.median(self.samples)), 'sm_max_mhz': self.max_mhz,
                'reasons': sorted(self.reasons), 'samples': len(self.samples)}


# ---------------------------------------------------------------------------
# CPU side: the reference's algorithm on host cores (NumPy oracle)
# ---------------------------------------------------------------------------
def cpu_reference_step(c, W, images, beam, keep=None):
    import comic_oracle as O
    import inception_v1_oracle as I
    emb, fm, _ = I.encoder(images, W, c)
    res = O.beam_search_decode(O.Decoder(W, c), emb, fm, beam, c.infer_length_penalty_weight, return_trace=keep is not None)
    _, ids, am = O.post_process_beam(res, c.attn_num_heads, beam)
    if keep is not None:
        keep.update(res=res, ids=ids, attn=am, images=images)
    return res['T']


def time_cpu_single_thread(c, W, n_images, beam):
    """The same NumPy restatement limited to ONE BLAS / OpenMP thread (BASELINE.md section 4), bounded sample."""
    try:
        from threadpoolctl import threadpool_limits
    except Exception:
        return None
    rng = np.random.default_rng(124)
    img = rng.uniform(-1, 1, (n_images, 224, 224, 3)).astype(np.float32)
    with threadpool_limits(limits=1):
        t0 = time.perf_counter()
        cpu_reference_step(c, W, img, beam)
        dt = time.perf_counter() - t0
    return n_images / dt


def time_cpu(c, W, n_images, beam, steps, warmup, keep=None):
    rng = np.random.default_rng(123)
    img = rng.uniform(-1, 1, (n_images, 224, 224, 3)).astype(np.float32)
    for _ in range(warmup):
        cpu_reference_step(c, W, img, beam)
    t0 = time.perf_counter()
    for i in range(steps):
        cpu_reference_step(c, W, img, beam, keep if i == steps - 1 else None)
    dt = time.perf_counter() - t0
    return n_images * steps / dt, dt / steps


def parity_block(model, kept, beam):
    """The CUDA path against the oracle's outputs on the cpu_baseline sample (outside every timed region): per image,
    the first step where ids / parents leave the oracle is accepted only at an oracle near-tie (top-(k+1) candidates
    within 1e-6 relative), as in tests/test_gpu_parity_large.py."""
    res, images = kept['res'], kept['images']
    eng = model.engine
    emb, fm = eng.encode(eng.to_dev(images))
    keys, values = eng.project_fm(fm)
    c0, h0 = eng.rnn_init(emb)
    r = eng.decode_beam(keys, values, c0, h0, beam, 0.0, res['T'])
    T = res['T']
    ids, par = r['step_ids'][:T].cpu().numpy(), r['parent_ids'][:T].cpu().numpy()
    same = (ids == res['step_ids']) & (par == res['parent_ids'])
    n_img = images.shape[0]
    near, bad = 0, 0
    keep_rows = []
    for b in range(n_img):
        ok = same[:, b, :].all(axis=1)
        if ok.all():
            keep_rows.append(b)
            continue
        t = int(np.argmin(ok))
        tot = res['trace'][t]['total'][b].reshape(-1).astype(np.float64)
        top = np.sort(tot)[::-1][:beam + 1]
        gap = float(np.min((top[:-1] - top[1:]) / np.maximum(np.abs(top[:-1]), 1e-30)))
        if gap < 1e-6:
            near += 1
        else:
            bad += 1
    am = kept['attn'][keep_rows]
    got = r['attn'][:, :, :T].cpu().numpy()[keep_rows]
    err = float(np.abs(got - am).max() / (np.abs(am).max() + 1e-30)) if keep_rows else None
    return {'images': n_img, 'steps': int(T), 'token_identical_images': len(keep_rows), 'near_tie_divergences': near,
            'other_divergences': bad, 'attention_map_rel_err': err, 'tolerance': 'ids / parents bit-exact except at oracle '
            'near-ties (< 1e-6 relative); attention maps 1e-3 relative'}


def cpu_train_step_baseline(batch=32, T=41):
    """BASELINE.json config 3 on the host cores: frozen InceptionV1 forward + teacher-forced decoder forward + backward
    (torch CPU autograd of the restatement in tests/torch_ref.py, the checker of the CUDA gradients; fp32, all cores) +
    the Adam update, ONE step of the same shapes as the GPU line (batch x T radix steps, every row full length)."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, 'tests'))
    import torch_ref as TR
    import comic_b200  # noqa: F401
    from comic_b200 import configuration as conf, weights as wts
    c = conf.make_config(train_mode='decoder', batch_size_train=batch)
    W = wts.init_weights(c, seed=c.rand_seed, cnn_init='he')
    rng = np.random.default_rng(0)
    images = rng.uniform(-1, 1, (batch, 224, 224, 3)).astype(np.float32)
    caps = np.concatenate([np.full((batch, 1), 256), rng.integers(0, 256, size=(batch, T - 1)), np.full((batch, 1), 257)],
                          axis=1).astype(np.int32)
    P = TR.to_params(W, dtype=torch.float32)
    PC = TR.cnn_params(W, dtype=torch.float32)
    m = {k: torch.zeros_like(v) for k, v in P.items()}
    v2 = {k: torch.zeros_like(v) for k, v in P.items()}
    t0 = time.perf_counter()
    with torch.no_grad():
        emb, fm = TR.encoder_forward(PC, images)
    tot = TR.training_loss(P, c, emb.double().numpy(), fm.double().numpy(), caps, dtype=torch.float32)[0]
    tot.backward()
    with torch.no_grad():
        for k, p_ in P.items():                       # tf.train.AdamOptimizer, step 1
            g = p_.grad
            m[k] += (g - m[k]) * 0.1
            v2[k] += (g * g - v2[k]) * 0.001
            p_ -= 1e-2 * m[k] / (v2[k].sqrt() + c.adam_epsilon)
    sec = time.perf_counter() - t0
    return {'value': 1.0 / sec, 'unit': 'steps/s', 'cores': torch.get_num_threads(), 'kind': 'port',
            'sample': '1 step, batch %d x %d steps: torch-CPU fp32 restatement (tests/torch_ref.py: InceptionV1 forward, '
                      'decoder forward + autograd backward, Adam)' % (batch, T)}


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return 0
    import comic_b200  # noqa: F401
    from comic_b200 import weights as wts
    c = make_config(args.workload)
    W = wts.init_weights(c, seed=c.rand_seed, cnn_init='he')
    cores = os.cpu_count()
    val, sec = time_cpu(c, W, args.ref_batch, args.beam, args.steps, max(args.warmup, 1))
    line = {
        'impl': 'reference', 'metric': METRIC if args.workload == 'comic256' else METRIC_WORD, 'value': val, 'unit': UNIT,
        'n_gpus': args.gpus,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': sec * 1e3, 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': workload_name(args.workload, args.batch, args.beam, c),
                   'note': 'reference arm: NumPy restatement of the TF1.9 graph (TF 1.9 / py2.7 not installable '
                           'offline), %d images per step on the host cores' % args.ref_batch},
        'cpu_baseline': {'value': val, 'unit': UNIT, 'cores': cores, 'kind': 'port',
                         'sample': '%d images x %d steps, encoder + beam-%d decode, NumPy/OpenBLAS all cores'
                                   % (args.ref_batch, args.steps, args.beam)},
        'e2e': {'value': val, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }
    print(json.dumps(line))
    return 0


# ---------------------------------------------------------------------------
# roofline accounting (DESIGN.md "Kernels")
# ---------------------------------------------------------------------------
def algorithmic_work(tag, eng, B, beam, T):
    """(amount per STEP, kind) for one kernel class; kind 'flop' or 'byte'."""
    d = eng.dims
    N = B * beam
    if tag == 'conv':
        from comic_b200 import weights as wts
        macs = 0
        hw = {'Conv2d_1a_7x7': 112, 'Conv2d_2b_1x1': 56, 'Conv2d_2c_3x3': 56}
        for scope, k, s, cin, cout in wts.cnn_conv_list():
            name = scope.split('/')[0]
            if name in hw:
                side = hw[name]
            elif name.startswith('Mixed_3'):
                side = 28
            elif name.startswith('Mixed_4'):
                side = 14
            else:
                side = 7
            macs += side * side * k * k * cin * cout
        return 2.0 * macs * B, 'flop'
    if tag == 'gates':
        return 2.0 * N * (d.W + d.A + d.R) * 4 * d.R * T, 'flop'
    if tag == 'lq':
        return 2.0 * N * d.R * (d.V + d.R) * T, 'flop'
    if tag == 'project':
        return 2.0 * B * d.M * d.C * d.R * (2 if d.fm_projection == 'independent' else 1), 'flop'
    if tag == 'scores':
        return (B * d.M * d.R * 4.0 + N * d.R * 4.0 + N * d.H * d.M * 4.0) * T, 'byte'
    if tag == 'ctx':
        return (B * d.M * d.VAL * 4.0 + 2.0 * N * d.H * d.M * 4.0 + N * d.A * 4.0) * T, 'byte'
    if tag == 'beam':
        return (N * d.V * 4.0 + N * 32.0) * T, 'byte'
    if tag == 'persist':
        # SURVEY.md 8(d): per decode step the weights once, the keys (and values) once per IMAGE, the
        # recurrent state read + written, the alignment history and the selection outputs
        KX = d.W + d.A + d.R
        wts_elems = KX * 4 * d.R + 4 * d.R + d.R * d.R + 3 * d.R + 1 + d.R * d.V + d.V
        per_step = (wts_elems * 4.0 + B * d.M * d.R * 4.0 + (0.0 if d.fm_projection == 'tied' else B * d.M * d.VAL * 4.0)
                    + 2.0 * N * (2 * d.R + d.A + d.W) * 4.0 + N * d.H * d.M * 4.0 + N * 12.0)
        return per_step * T, 'byte'
    if tag == 'lstm':
        return (N * 4 * d.R * 4.0 + 3.0 * N * d.R * 4.0) * T, 'byte'
    return 0.0, 'byte'


def load_peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        with open(p) as f:
            j = json.load(f)
        return {'hbm': j['hbm_gbs'], 'tensor': j.get('bf16_tflops_sustained', j['bf16_tflops']), 'which': 'measured'}
    return {'hbm': 6650.0, 'tensor': 1590.0, 'which': 'fallback'}


def load_traffic(tag):
    p = os.path.join(ROOT, 'profiles', 'traffic.json')
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f).get(tag)
    return None


DUMP_BYTES = 60 << 20         # --dump-outputs stays under 64 MB, npy headers included


def beam_outputs(r, T):
    """Host copies of what Engine.decode_beam returned (r), for --dump-outputs: the T executed steps only (the rows
    after them are never written), ids and lengths as float64 (exact), scores and attention maps as float32.  When all
    of it exceeds DUMP_BYTES (the attention maps of one 512-image step alone are 192 MB), every array is cut to the same
    fixed, seeded sample of images, listed in `images`; the sample depends on the batch shape only."""
    import torch
    B = r['lengths'].shape[0]
    itemsize = dict(predicted_ids=8, step_ids=8, parent_ids=8, scores=4, lengths=8, attn=4)     # as written
    per_image = sum(r[k].numel() * s for k, s in itemsize.items()) // B + 8                    # + its `images` entry
    n = min(B, DUMP_BYTES // per_image)
    idx = np.sort(np.random.default_rng(0).choice(B, n, replace=False))
    sel = torch.from_numpy(idx).to(r['lengths'].device)
    out = {k: r[k][:T].index_select(1, sel).cpu().numpy().astype(np.float64)
           for k in ('predicted_ids', 'step_ids', 'parent_ids')}
    out['scores'] = r['scores'][:T].index_select(1, sel).cpu().numpy().astype(np.float32)
    out['lengths'] = r['lengths'].index_select(0, sel).cpu().numpy().astype(np.float64)
    out['attn'] = r['attn'].index_select(0, sel)[:, :, :T].cpu().numpy().astype(np.float32)
    out['images'] = idx.astype(np.float64)
    return out


def dump_outputs(out_dir, arrays):
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + '.npy'), a)


# ---------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    import comic_b200  # noqa: F401
    from comic_b200 import weights as wts
    from comic_b200.engine import Engine, KERNEL_TAGS
    from comic_b200.model import CaptionModel
    from comic_b200 import parallel as par

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise SystemExit('bench.py: no CUDA device; the hot path has no CPU fallback')
    torch.cuda.set_device(local)
    # N > 1: every rank streams 0.5 GB per batch through pinned host memory; keep each rank (and the pinned buffers it
    # is about to allocate) on the CPUs next to its GPU.  N = 1 keeps all host cores (cpu_baseline uses them).
    numa_cpus = set()
    if world > 1 and os.environ.get('COMIC_B200_NUMA_BIND', '1') != '0':
        numa_cpus = par.bind_to_gpu_numa(local)
    if world > 1:
        # NCCL prints its version banner to stdout at NCCL_DEBUG=VERSION / WARN: keep stdout to the one JSON line
        if os.environ.get('NCCL_DEBUG', '').upper() in ('VERSION', 'WARN'):
            os.environ.pop('NCCL_DEBUG')
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    c = make_config(args.workload)
    c.infer_beam_size = args.beam
    c.batch_size_infer = args.batch
    W = wts.init_weights(c, seed=c.rand_seed, cnn_init='he')
    eng = Engine(c)
    eng.bind_weights(W)
    eng.set_precision(args.precision)
    for kv in args.opt:
        name, value = kv.split('=')
        eng.set_option(name, int(value))
    model = CaptionModel(c, 'infer', batch_ops=None, engine=eng)
    B, beam = args.batch, args.beam
    T = model._maximum_iterations()

    # synthetic inputs: pinned host copy (e2e) + device-resident copy (value); 308 MB/step > 126 MB L2
    g = torch.Generator().manual_seed(1000 + rank)
    host_images = torch.empty((B, 224, 224, 3), dtype=torch.float32).pin_memory()
    host_images.uniform_(-1.0, 1.0, generator=g)
    dev_images = host_images.to(eng.device, non_blocking=False)

    def step_eager(images):
        emb, fm = eng.encode(images)
        keys, values = eng.project_fm(fm)
        c0, h0 = eng.rnn_init(emb)
        return eng.decode_beam(keys, values, c0, h0, beam, c.infer_length_penalty_weight, T)

    def step_device():
        # the whole device step as one CUDA graph from the third call on (Engine.graphed); eager while a kernel-class
        # profile is active
        return eng.graphed('bench_step', step_eager, dev_images)

    host_images2 = torch.empty((B, 224, 224, 3), dtype=torch.float32).pin_memory()
    host_images2.copy_(host_images.flip(0))

    # raw-pixel variant of the same batches: uint8, what an image decoder hands over (77 MB instead of 308 MB per step)
    host_u8 = [((h + 1.0) * 127.5).clamp_(0, 255).to(torch.uint8).pin_memory() for h in (host_images, host_images2)]

    def e2e_loop(n, raw_pixels=True, maps=False):
        """n batches through the public pipelined inference loop (CaptionModel.run_stream), host buffers in, host
        buffers out.  raw_pixels: uint8 pixels cross PCIe and the reference's evaluation pre-processing runs on the
        device; maps: the top-beam attention maps come back too (only needed with `save_attention_maps`,
        src/infer_fn.py:169-171).  (False, True) is round 1's variant: fp32 images in, fp32 maps out."""
        src = host_u8 if raw_pixels else (host_images, host_images2)
        model.collect_attention_maps = maps
        got, out = 0, None
        for out in model.run_stream(src[j % 2] for j in range(n)):
            got += int(out[0].shape[0])
        assert got == n * B
        model.collect_attention_maps = True
        return out

    # ---- kernel-class breakdown (outside the timed region) -> dominant kernel
    for _ in range(max(args.warmup, 3)):
        r = step_device()
    torch.cuda.synchronize()
    eng.profile_enable(KERNEL_TAGS)
    step_device()
    torch.cuda.synchronize()
    table = {t: eng.profile_read(t) for t in KERNEL_TAGS}
    eng.profile_enable([])
    ranked = sorted(table, key=lambda t: -table[t][0])
    dominant, runner_up = ranked[0], ranked[1]
    if args.breakdown and rank == 0:
        tot = sum(v[0] for v in table.values())
        for t in KERNEL_TAGS:
            ms, n = table[t]
            sys.stderr.write('%-8s %9.3f ms %6d launches %5.1f%%\n' % (t, ms, n, 100 * ms / max(tot, 1e-9)))

    # ---- timed region 1: device-resident inputs (value)
    for _ in range(3):
        r = step_device()            # eager, capture, first replay
    torch.cuda.synchronize()
    sampler = ClockSampler(local)
    launches0 = eng.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    sampler.start()
    ev0.record()
    for _ in range(args.steps):
        r = step_device()
    ev1.record()
    barrier()
    sampler.stop()
    ms_total = ev0.elapsed_time(ev1)
    launches = eng.launch_count() - launches0
    from comic_b200.engine import executed_steps
    # r lives in the graph's output buffers, which the next step overwrites: copy the last timed step's outputs now
    dumped = beam_outputs(r, executed_steps(r['T'])) if args.dump_outputs and rank == 0 else None
    # ---- timed region 1b: the same K steps launched one by one with CUDA events around every launch of the two largest
    # kernel classes (events cannot be captured into the graph): the roofline block's launch durations and shares
    eng.profile_enable([dominant, runner_up])
    barrier()
    ev0.record()
    for _ in range(args.steps):
        r = step_device()
    ev1.record()
    barrier()
    ms_prof = ev0.elapsed_time(ev1)
    dom_ms, dom_n = eng.profile_read(dominant)
    run_ms, run_n = eng.profile_read(runner_up)
    eng.profile_enable([])
    T_exec = executed_steps(r['T'])

    # ---- timed region 2: end to end through CaptionModel.run_stream from pinned host memory
    out = e2e_loop(6)                # 3 batches per input slot: eager, CUDA-graph capture, first replay (Engine.graphed)
    barrier()
    t0 = time.perf_counter()
    out = e2e_loop(args.steps)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    barrier()
    # round 1's variant for continuity: fp32 images in, fp32 attention maps out
    out_f = e2e_loop(6, raw_pixels=False, maps=True)
    barrier()
    t0 = time.perf_counter()
    out_f = e2e_loop(args.steps, raw_pixels=False, maps=True)
    torch.cuda.synchronize()
    e2e_f_s = time.perf_counter() - t0
    barrier()
    # the same K batches one blocking CaptionModel.run call at a time (no copy/compute overlap)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        model.run(host_images)
    torch.cuda.synchronize()
    e2e_serial_s = time.perf_counter() - t0
    barrier()
    h2d = host_u8[0].numel()
    d2h = int(out[0].nbytes)
    h2d_f = host_images.numel() * 4
    d2h_f = int(out_f[0].nbytes + out_f[1].nbytes)

    t_dev = torch.tensor([ms_total, e2e_s * 1e3, e2e_f_s * 1e3], dtype=torch.float64, device=eng.device)
    if world > 1:
        dist.all_reduce(t_dev, op=dist.ReduceOp.MAX)
    ms_total, e2e_ms, e2e_f_ms = [float(x) for x in t_dev.tolist()]

    # ---- train block: BASELINE.json configs 3-5 on the same ranks (one NCCL sum all-reduce of the flat gradient per step)
    train = None
    if not args.no_train and args.workload == 'comic256':
        sys.path.insert(0, os.path.join(ROOT, 'scripts'))
        import bench_train
        train = {}
        # cnn_finetune runs in the arithmetic mode its gradient parity test verifies (tests/test_gpu_train_cnn.py: the
        # tape forward and the backward GEMMs in f32); the bf16x3 number is reported beside it, unverified
        for key, mode, batch, prec in (('decoder', 'decoder', 32, args.precision), ('cnn_finetune', 'cnn_finetune', 32, 'f32'),
                                       ('cnn_finetune_bf16x3_unverified', 'cnn_finetune', 32, args.precision),
                                       ('scst', 'scst', 10, args.precision)):
            r = bench_train.run_mode(mode, batch, args.train_steps, 3, prec)
            # algorithmic bytes of one teacher-forced fwd + bwd step (SURVEY.md section 8d: ~3x the forward): per time step the
            # decoder weights (12.08 MB) and the batch's keys (B x 401,408 B) stream once forward and twice backward
            if mode != 'scst':
                steps_t = 41
                alg = 3 * steps_t * (12.08e6 + batch * 401408)
                r['roofline'] = {'bound': 'hbm', 'achieved': alg / (r['ms_per_step'] * 1e-3) / 1e9, 'peak': load_peaks()['hbm'],
                                 'unit': 'GB/s', 'frac': alg / (r['ms_per_step'] * 1e-3) / 1e9 / load_peaks()['hbm'],
                                 'traffic': None, 'note': 'decoder part only; launch-bound (%d launches per step)' % r['gpu_launches_per_step']}
            r['cpu_baseline'] = None       # the NumPy oracle restates the forward and the losses only
            if key == 'decoder' and world == 1 and not args.no_cpu_baseline:
                try:
                    r['cpu_baseline'] = cpu_train_step_baseline(batch)
                except Exception as e:     # a reported baseline, never a reason to lose the line
                    r['cpu_baseline'] = {'unavailable': repr(e)[:200]}
            train[key] = r

    if rank == 0:
        peaks = load_peaks()

        def roofline_of(tag, tag_ms, tag_n):
            """Roofline block of one kernel class, from the CUDA-event time of its launches inside the timed region."""
            work, kind = algorithmic_work(tag, eng, B, beam, T_exec)
            per_launch = work * args.steps / max(tag_n, 1)
            avg_s = tag_ms * 1e-3 / max(tag_n, 1)
            if kind == 'flop':
                achieved = per_launch / avg_s / 1e12
                rf = {'bound': 'tensor', 'achieved': achieved, 'peak': peaks['tensor'], 'unit': 'TFLOP/s',
                      'frac': achieved / peaks['tensor']}
            else:
                achieved = per_launch / avg_s / 1e9
                rf = {'bound': 'hbm', 'achieved': achieved, 'peak': peaks['hbm'], 'unit': 'GB/s',
                      'frac': achieved / peaks['hbm']}
            rf.update({'traffic': load_traffic(tag), 'kernel': tag, 'launches': tag_n,
                       'avg_launch_us': avg_s * 1e6, 'share_of_step': tag_ms / ms_prof,
                       'timed': '%d steps launched eagerly with events around this class (%.3f ms per step; the value '
                                'region replays the step as a CUDA graph)' % (args.steps, ms_prof / args.steps),
                       'peak_source': peaks['which'] + (' sustained' if kind == 'flop' else ''),
                       'arithmetic': {'f32': 'fp32 FFMA', 'split': 'tcgen05 bf16x3 operand split, fp32 accumulate (fp32-equivalent)',
                                      'fast': 'tcgen05 bf16x3 + tanh.approx'}[args.precision] if kind == 'flop' else 'fp32'})
            return rf

        roof = roofline_of(dominant, dom_ms, dom_n)
        try:
            roof['runner_up'] = roofline_of(runner_up, run_ms, run_n)    # the second kernel class of the step, same method
        except Exception as e:      # a class without a work model
            roof['runner_up'] = {'kernel': runner_up, 'error': str(e)}
        caps = B * world * args.steps
        line = {
            'metric': METRIC if args.workload == 'comic256' else METRIC_WORD, 'value': caps / (ms_total * 1e-3), 'unit': UNIT,
            'n_gpus': world,
            'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms_total / args.steps,
            'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': {'f32': 'f32', 'split': 'f32 storage and accumulation; GEMM / conv operands split into 3 bf16 terms on tcgen05 (bf16x3)',
                      'fast': 'f32 storage and accumulation; bf16x3 GEMMs + tanh.approx.f32'}[args.precision],
            'data': 'synthetic',
            'config': {'workload': workload_name(args.workload, B, beam, c), 'images_per_gpu': B,
                       'global_batch': B * world, 'beam': beam, 'decode_steps': T_exec,
                       'parallelism': 'image-sharded x%d, no collective' % world,
                       'l2_policy': 'inputs larger than L2 (308 MB images + 206 MB keys per step)'},
            'decoder_step_us': None,
            'roofline': roof,
            'e2e': {'value': caps / (e2e_ms * 1e-3), 'unit': UNIT, 'h2d_bytes_per_step': h2d,
                    'd2h_bytes_per_step': d2h, 'ms_per_step': e2e_ms / args.steps,
                    'api': 'CaptionModel.run_stream (H2D / compute / D2H pipelined over 3 streams): uint8 pixels in, '
                           'evaluation pre-processing on the device, word ids out (attention maps only with '
                           'save_attention_maps, as inference.run_inference does)',
                    'fp32_images_and_attention_maps': {'value': caps / (e2e_f_ms * 1e-3), 'unit': UNIT,
                                                       'h2d_bytes_per_step': h2d_f, 'd2h_bytes_per_step': d2h_f,
                                                       'ms_per_step': e2e_f_ms / args.steps},
                    'serial_run_ms_per_step': e2e_serial_s * 1e3 / args.steps,
                    'host_cpus_bound': len(numa_cpus) or None},
            'gpu_launches': int(launches),
            'clocks': sampler.summary(),
            'kernel_ms_per_step': {t: round(table[t][0], 3) for t in KERNEL_TAGS if table[t][1]},
        }
        dec_ms = sum(table[t][0] for t in ('gates', 'lstm', 'lq', 'scores', 'ctx', 'beam', 'persist'))
        line['decoder_step_us'] = dec_ms * 1e3 / max(T_exec, 1)
        if world == 1 and not args.no_cpu_baseline:
            cores = os.cpu_count()
            kept = {}
            val, _sec = time_cpu(c, W, args.cpu_sample, beam, 1, 1, kept)
            line['parity'] = parity_block(model, kept, beam)
            st = time_cpu_single_thread(c, W, 4, beam)
            line['cpu_baseline'] = {'value': val, 'unit': UNIT, 'cores': cores, 'kind': 'port', 'single_thread_value': st,
                                    'single_thread_sample': '4 images, same path, BLAS / OpenMP threads limited to 1',
                                    'sample': '%d images, encoder + %d-step beam-%d decode, NumPy oracle on all host cores'
                                              % (args.cpu_sample, T, beam)}
        if train is not None:
            line['train'] = train
        if dumped is not None:
            dump_outputs(args.dump_outputs, dumped)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    args = parse_args()
    if args.impl == 'reference':
        return run_reference(args)
    return run_ours(args)


if __name__ == '__main__':
    sys.exit(main())

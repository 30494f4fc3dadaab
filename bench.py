#!/usr/bin/env python
"""bench.py -- X-UNet DDPM training throughput (BASELINE.json metric: train images/sec) on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload small64|small128|full128|full64]
                    [--batch B] [--dtype bf16|fp32] [--no-full128] [--sampler-steps 256] [--dump-outputs DIR]

One "step" = one optimisation step (pinned H2D staging -> forward -> backward -> [bucketed NCCL all-reduce, overlapped
with the backward] -> Adam) on a synthetic SRN-shaped batch of B (source,target) pairs PER GPU (weak scaling).
Headline workload = BASELINE.json configs[1]: small X-UNet (ch=32, ch_mult=(1,2), emb_ch=32, nrb=2, attn_res=(8,16,32),
heads=4), 64x64, bf16, B=8.

Printed JSON (rank 0, one line):
  value    : images/s with the inputs already resident in HBM (device tensors), CUDA-graph replayed step
  e2e      : images/s through the public API (TrainStep.__call__) with HOST numpy inputs: pinned staging + H2D copies and a
             D2H read of the loss inside the timed region, every step
  roofline : the dominant kernel of the step, timed alone with CUDA events on its launching stream
  cpu_baseline : the CPU oracle (restatement of the JAX reference; JAX is not installable here) on the host cores: thread
             sweep, best thread count, train step (config B) and the single eps-forward of BASELINE configs[0]
  full128  : BASELINE configs[2]/[3] in the SAME line at every N: full 3DiM X-UNet (439 M parameters) at 128x128, per-GPU
             batch 4: ms/step, images/s, step TFLOP/s and fraction of the sustained tensor peak, and at N>1 the measured
             all-reduce time of the 1.755 GB gradient bucket and how much of it the backward hides; at N=1 also the
             256-step CFG sampler of the full model at 128x128 (views/s at 1 view and at 4 views in flight)
--impl reference times the CPU oracle alone with the same metric/unit/config (rank 0 only).
--dump-outputs DIR writes what the last timed device-resident step handed its caller, as float32 .npy files (rank 0): loss,
the updated params / adam_mu / adam_nu and that step's grads (flat, in the library's parameter order), and e2e_losses (the
loss of every timed end-to-end step).  The inputs are seeded, so two builds run with the same arguments can be compared
output for output.  Flat buffers longer than DUMP_MAX_ELEMS (the full model's) are reduced to a fixed, seeded sample of
DUMP_MAX_ELEMS indices, the same for all four.  The outputs are not bit-reproducible: fp32 atomic reductions differ in the last
bits from run to run, and bf16 training amplifies that step by step (two runs of one build with the default arguments, 35
steps, B200 at 1000 W: loss 3e-4, params 1e-2, grads 2e-2 relative L2 apart), so judge a difference between builds against
the spread of two runs of the same build.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    #            model preset, side, default per-GPU batch, fwd FLOPs/sample (SURVEY 8(d))
    'small64': ('small', 64, 8, 13_997_445_120),
    'small128': ('small', 128, 8, 27_804_045_312),
    'full128': ('full', 128, 4, 3_155_647_528_960),
    'full64': ('full', 64, 4, 881_256_824_832),
}
METRIC, UNIT = 'xunet_train_images_per_sec', 'images/s'
DUMP_MAX_ELEMS = 3_000_000      # per flat buffer: 4 buffers x 12 MB stay under 64 MB (the small model's 1.05 M fit whole)


_T0 = time.perf_counter()


def progress(msg):
    """phase log on stderr (stdout carries exactly one JSON line)"""
    if int(os.environ.get('RANK', '0')) == 0:
        print(f'[bench +{time.perf_counter() - _T0:6.1f}s] {msg}', file=sys.stderr, flush=True)


def load_peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(hbm=p['hbm_gbs'], tf_burst=p['bf16_tflops'], tf_sustained=p.get('bf16_tflops_sustained', p['bf16_tflops']),
                    source='measured')
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sustained=1400.0, source='fallback')


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = 'clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
        'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, index=0):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--id={self.index}', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits',
                                          '-lms', '100'], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(',')])

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
                for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), r[3:7]):
                    if v.lower().startswith('active'):
                        reasons.add(name)
            except Exception:
                pass
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': mx, 'reasons': sorted(reasons), 'samples': len(sm)}


# ------------------------------------------------------------------------------------------------------------------
def make_host_batches(n, B, S, seed):
    """n synthetic SRN-shaped batches as the data loader would hand them over (data_loader.py:102-113: x float32; z, noise
    float64; logsnr float64)."""
    from novel_view_synthesis_3d_b200.synthetic import synthetic_batch
    return [synthetic_batch(B, S, seed=seed + i) for i in range(n)]


# ------------------------------------------------------------------------------------------------------------------
# CPU arm: the oracle (restatement of the JAX reference) on the host cores
# ------------------------------------------------------------------------------------------------------------------
class CpuOracle:
    """One training step (fwd + bwd by autograd + Adam on all leaves, train.py:49-76) or one eps-forward of the fp32 torch-CPU
    oracle at a given thread count."""

    def __init__(self, preset, S, B):
        import torch
        from oracle import xunet_ref as R
        self.torch, self.R, self.B, self.S = torch, R, B, S
        self.cfg = R.SMALL if preset == 'small' else R.FULL
        params = R.init_params(self.cfg, S, seed=0, zero_init=False, dtype=torch.float32)
        self.flat = R.flatten(params)
        self.m = {k: torch.zeros_like(v) for k, v in self.flat.items()}
        self.v = {k: torch.zeros_like(v) for k, v in self.flat.items()}
        self.batch, self.noise = R.synthetic_batch(B, S, seed=1234, dtype=torch.float32)
        self.cond = torch.ones(B)
        rng = np.random.RandomState(0)
        self.mask_fn = lambda idx, shape: torch.from_numpy(rng.random_sample(shape) >= self.cfg.dropout)
        self.it = 0

    def train_step(self):
        R = self.R
        self.it += 1
        loss, grads, _ = R.loss_and_grads(R.nest(self.flat), self.batch, self.noise, self.cond, self.cfg, train=True,
                                          drop_mask_fn=self.mask_fn)
        for k in self.flat:
            self.flat[k], self.m[k], self.v[k] = R.adam_update(self.flat[k], grads[k], self.m[k], self.v[k], self.it)
        return float(loss)

    def forward(self):
        with self.torch.no_grad():
            return self.R.xunet_forward(self.R.nest(self.flat), self.batch, self.cond, self.cfg, train=False)


def _timed(fn, n, budget_s):
    ts, t_begin = [], time.perf_counter()
    for i in range(n):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
        if time.perf_counter() - t_begin > budget_s and i >= 0:
            break
    return ts


def cpu_thread_sweep(preset, S, budget_s=14.0):
    """images/s of a batch-2 train step at {8,16,32,64,128,...} threads (one warm-up + up to two timed steps each, bounded;
    the likeliest winners first so that a cut-short sweep still holds them)."""
    import torch
    avail = len(os.sched_getaffinity(0))
    cands = sorted({t for t in (8, 16, 32, 64, 128) if t <= avail}, key=lambda t: (abs(math.log2(t / 32.0)), -t))
    orc = CpuOracle(preset, S, 2 if preset == 'small' else 1)
    out, t_begin, best_t = {}, time.perf_counter(), None
    for th in cands:
        if out and time.perf_counter() - t_begin > budget_s:
            break
        torch.set_num_threads(th)
        t0 = time.perf_counter()
        orc.train_step()
        warm = time.perf_counter() - t0
        if (best_t is not None and warm > 4.0 * best_t) or time.perf_counter() - t_begin > 2.0 * budget_s:
            out[th] = orc.B / warm       # far off (oversubscription) or out of time: record the single step and move on
            continue
        ts = _timed(orc.train_step, 2, budget_s / len(cands))
        out[th] = orc.B / float(np.median(ts))
        best_t = float(np.median(ts)) if best_t is None else min(best_t, float(np.median(ts)))
    best = max(out, key=out.get)
    return dict(sorted(out.items())), best, avail


def cpu_baseline(preset, S, B_sample, budget_s=30.0, threads=None):
    """Bounded CPU sample: thread sweep -> best thread count -> timed train steps, plus the single eps-forward of
    BASELINE.json configs[0] (small model only)."""
    import torch
    orc = CpuOracle(preset, S, B_sample)
    if threads is None and preset == 'small':
        sweep, best, avail = cpu_thread_sweep(preset, S, budget_s=budget_s * 0.45)
    elif threads is None:
        sweep, best, avail = {}, min(64, len(os.sched_getaffinity(0))), len(os.sched_getaffinity(0))
    else:
        sweep, best, avail = {}, threads, len(os.sched_getaffinity(0))
    torch.set_num_threads(best)
    orc.train_step()
    ts = _timed(orc.train_step, 8, budget_s * (0.35 if threads is None else 0.6))
    med = float(np.median(ts))
    cb = dict(value=B_sample / med, unit=UNIT, cores=best, cores_available=avail, kind='port',
              thread_sweep_images_per_sec={str(k): round(v, 4) for k, v in sweep.items()},
              sample=f'{len(ts)} timed train steps (fwd+bwd+Adam, fp32 torch-CPU oracle) of batch {B_sample} at {S}x{S}, '
                     f'median {med * 1e3:.0f} ms/step at the best of the swept thread counts; JAX itself is not installable offline')
    if preset == 'small':
        o0 = CpuOracle('small', 64, 2)           # BASELINE.json configs[0]: single eps-forward, batch 2, 64x64
        o0.forward()
        t0 = _timed(o0.forward, 6, budget_s * 0.15)
        cb['config0_single_eps_forward'] = {'batch': 2, 'side': 64, 'ms': float(np.median(t0)) * 1e3,
                                            'images_per_sec': 2 / float(np.median(t0)), 'cores': best}
    return cb


def _cpu_child(args, limit_s):
    """One bounded oracle measurement in a child process (a busy host or an oversubscribing thread count can make a single torch-CPU
    step take minutes; the child is killed at limit_s and the GPU line survives)."""
    cmd = [sys.executable, os.path.abspath(__file__), '--cpu-baseline-child'] + [str(a) for a in args]
    try:
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=limit_s)
        for line in reversed(r.stdout.strip().splitlines()):
            if line.startswith('{'):
                return json.loads(line)
        return {'error': 'no result: ' + r.stderr[-200:]}
    except subprocess.TimeoutExpired:
        return {'error': f'killed after {limit_s:.0f} s'}


def cpu_baseline_guarded(preset, S, B_sample, budget_s, hard_limit_s=150.0):
    """Thread sweep with ONE child process per thread count (each with its own time limit), then the best count's record."""
    avail = len(os.sched_getaffinity(0))
    cands = [t for t in (16, 32, 8, 64) if t <= avail] or [avail]
    t_begin, sweep, recs = time.perf_counter(), {}, {}
    for th in cands:
        left = hard_limit_s - (time.perf_counter() - t_begin)
        if left < 20 or (recs and time.perf_counter() - t_begin > budget_s * 1.5):
            break
        rec = _cpu_child([preset, S, B_sample, budget_s / 3.0, th], min(left, 45.0))
        sweep[str(th)] = round(rec['value'], 4) if 'value' in rec else rec.get('error')
        if 'value' in rec:
            recs[th] = rec
    if not recs:
        return {'error': 'every thread count failed or timed out', 'thread_sweep_images_per_sec': sweep, 'kind': 'port', 'cores_available': avail}
    best = max(recs, key=lambda t: recs[t]['value'])
    cb = recs[best]
    cb['thread_sweep_images_per_sec'] = sweep
    cb['cores_available'] = avail
    return cb


def run_reference(args, preset, S, B):
    """Reference arm: the CPU oracle on the arm's own config (same model, side and per-GPU batch), --warmup / --steps
    honoured up to a wall-clock budget (the actual counts are reported)."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    import torch
    budget = float(args.ref_budget_s)
    t_begin = time.perf_counter()
    Bs = B if preset == 'small' else 1
    orc = CpuOracle(preset, S, Bs)
    avail = len(os.sched_getaffinity(0))
    sweep, best = {}, min(16, avail)
    if preset == 'small':
        # thread sweep in child processes (batch-2 steps, each bounded): torch-CPU regresses beyond ~16 threads on this model
        best_v = -1.0
        for th in [t for t in (16, 32, 8, 64) if t <= avail] or [avail]:
            if time.perf_counter() - t_begin > budget * 0.25:
                break
            rec = _cpu_child([preset, S, 2, 6.0, th], 30.0)
            sweep[th] = rec.get('value', 0.0)
            if rec.get('value', 0.0) > best_v:
                best_v, best = rec['value'], th
    torch.set_num_threads(best)
    warm = _timed(orc.train_step, max(1, args.warmup), budget * 0.15)
    ts = _timed(orc.train_step, max(1, args.steps), budget - (time.perf_counter() - t_begin))
    mean = float(np.mean(ts))
    value = Bs / mean
    cb = dict(value=value, unit=UNIT, cores=best, cores_available=avail, kind='port',
              thread_sweep_images_per_sec={str(k): round(v, 4) for k, v in sweep.items()},
              sample=f'{len(ts)} timed train steps (fwd+bwd+Adam, fp32 torch-CPU oracle) of batch {Bs} at {S}x{S} after '
                     f'{len(warm)} warm-up steps; mean {mean * 1e3:.0f} ms/step')
    line = {'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': len(ts),
            'warmup': len(warm), 'steps_requested': args.steps, 'warmup_requested': args.warmup,
            'ms_per_step': 1e3 * mean, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': args.workload, 'model': preset, 'side': S, 'per_gpu_batch': Bs, 'global_batch': Bs,
                       'arm_per_gpu_batch': B, 'optimizer': 'adam lr1e-4', 'loss': 'frobenius (train.py:67)',
                       'note': 'CPU oracle = torch-CPU restatement of the JAX reference (JAX not installable offline); '
                               'one host process on rank 0, all host threads it scales to'},
            'cpu_baseline': cb,
            'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------------------------
def time_kernel(fn, iters=30, warm=5):
    import torch
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters * 1e-3


def dominant_kernel_roofline(P, model, B, S, peaks):
    """Times the step's heaviest kernels ALONE (CUDA events on the launching stream, >=3 warm-ups) through the operator-level
    C-ABI at the exact shapes and with the exact implementations (tcgen05) the step uses, and returns the roofline of the
    one with the largest share of the step.  Algorithmic FLOPs per launch are SURVEY 8(d)'s (2*MAC; backward := 2 x forward)."""
    import torch
    from novel_view_synthesis_3d_b200 import _lib
    lib = _lib.load()
    os.environ['XUNET_OP_CACHE_SHADOW'] = '1'     # time the conv kernel alone (the step converts weights once per forward)
    os.environ.pop('XUNET_OP_ATTN_FOLD', None)    # attention backward as the engine runs it: prep + fused dK/dV/dQ + store (hd <= 32)
    cfg = model.config
    tc = cfg.dtype == 'bf16'
    dt = _lib.DTYPE_BF16 if tc else _lib.DTYPE_F32
    impl = 1 if tc else 0
    tdt = torch.bfloat16 if tc else torch.float32
    st = torch.cuda.current_stream().cuda_stream
    N, dev, out = 2 * B, 'cuda', []
    nrb, L = cfg.num_res_blocks, len(cfg.ch_mult)

    def conv_case(H, Ci, Co, count):
        x = torch.randn(N, H, H, Ci, device=dev).to(tdt)
        w = torch.randn(9 * Ci * Co, device=dev) * 0.05
        b = torch.zeros(Co, device=dev)
        y = torch.empty(N, H, H, Co, device=dev, dtype=tdt)
        dw = torch.zeros(9 * Ci * Co, device=dev)
        flops = 2.0 * N * H * H * 9 * Ci * Co
        fn = lambda: lib.xunet_op_conv(dt, impl, x.data_ptr(), w.data_ptr(), b.data_ptr(), None, y.data_ptr(), N, H, H, Ci, Co, 3, 1, 1, 1.0, st)
        assert fn() == 0, lib.xunet_last_error()
        out.append(dict(kernel=f'conv3x3 fwd {Ci}->{Co} @{H} ({"tcgen05" if tc else "simt"})', seconds=time_kernel(fn), flops=flops, count=count))
        fw = lambda: lib.xunet_op_conv_wgrad(dt, impl, x.data_ptr(), y.data_ptr(), dw.data_ptr(), b.data_ptr(), N, H, H, Ci, Co, 3, 1, 1, 1.0, st)
        assert fw() == 0, lib.xunet_last_error()
        out.append(dict(kernel=f'conv3x3 wgrad {Ci}->{Co} @{H} ({"tcgen05" if tc else "simt"})', seconds=time_kernel(fw), flops=flops, count=count))

    def attn_case(Lq, C, heads, count):
        qkv = torch.randn(N, Lq, 3 * C, device=dev).to(tdt)
        res = torch.randn(N, Lq, C, device=dev).to(tdt)
        o = torch.empty(N, Lq, C, device=dev, dtype=tdt)
        lse = torch.empty(N, heads, Lq, device=dev)
        dscr = torch.zeros(N * Lq * (heads + C), device=dev)
        dqkv = torch.empty_like(qkv)
        flops = 4.0 * N * heads * Lq * Lq * (C // heads)
        fn = lambda: lib.xunet_op_attention(dt, impl, qkv.data_ptr(), res.data_ptr(), o.data_ptr(), lse.data_ptr(), N, Lq, C, heads, 0, st)
        assert fn() == 0, lib.xunet_last_error()
        out.append(dict(kernel=f'attention fwd L={Lq} hd={C // heads}', seconds=time_kernel(fn), flops=flops, count=count))
        fb = lambda: lib.xunet_op_attention_bwd(dt, impl, qkv.data_ptr(), res.data_ptr(), o.data_ptr(), res.data_ptr(), lse.data_ptr(),
                                                dscr.data_ptr(), dqkv.data_ptr(), N, Lq, C, heads, 0, st)
        assert fb() == 0, lib.xunet_last_error()
        # algorithmic backward work = 5 GEMMs (S, dP, dV, dK, dQ) = 2.5x the forward's two
        bname = 'attention bwd (prep + fused dK/dV/dQ + store)' if C // heads <= 32 else 'attention bwd (dQ + dK/dV)'
        out.append(dict(kernel=f'{bname} L={Lq} hd={C // heads}', seconds=time_kernel(fb), flops=2.5 * flops, count=count))

    feat = [cfg.ch * m for m in cfg.ch_mult]
    conv_case(S, feat[0], feat[0], 2 * nrb + 2)
    if L > 1:
        conv_case(S // 2, feat[1], feat[1], 2 * nrb + 4)
        if (S // 2) in cfg.attn_resolutions:
            attn_case((S // 2) ** 2, feat[1], cfg.attn_heads, 2 * (2 * nrb + 2))
    top = max(out, key=lambda r: r['seconds'] * r['count'])
    peak = peaks['tf_burst']
    achieved = top['flops'] / top['seconds'] / 1e12
    traffic = None
    tpath = os.path.join(ROOT, 'profiles', 'roofline_traffic.json')   # dram bytes/launch from the committed ncu --set full capture
    if os.path.exists(tpath):
        traffic = json.load(open(tpath)).get(top['kernel'])
    return {'bound': 'tensor', 'kernel': top['kernel'], 'achieved': achieved, 'peak': peak, 'unit': 'TFLOP/s',
            'frac': achieved / peak, 'traffic': traffic, 'peak_source': peaks['source'] + ' (burst, kernel timed alone)',
            'per_launch_us': top['seconds'] * 1e6, 'algorithmic_flops_per_launch': top['flops'],
            'candidates': [{'kernel': r['kernel'], 'us': r['seconds'] * 1e6, 'tflops': r['flops'] / r['seconds'] / 1e12,
                            'launches_per_step': r['count']} for r in out]}


# ------------------------------------------------------------------------------------------------------------------
class TrainBench:
    """One workload on this rank's GPU: build the model / state / fused step, time device-resident and end-to-end steps."""

    def __init__(self, P, xdist, preset, S, B, dtype, dev, use_graph=True, init_on_device=False, n_host=4):
        import torch
        self.P, self.xdist, self.torch, self.dev, self.B, self.S = P, xdist, torch, dev, B, S
        rank = xdist.rank()
        cfgk = dict(dtype=dtype)
        self.model = P.XUNet(**cfgk) if preset == 'small' else P.XUNet.from_config(P.XUNetConfig(**{**P.FULL_3DIM.__dict__, **cfgk}))
        self.state = P.create_train_state(0, 1, 1e-4, B, S, model=self.model, init_on_device=init_on_device)   # Flax-style init, rank-0 params broadcast
        self.step = P.TrainStep(self.state, use_graph=use_graph)
        self.eng = self.step.eng
        self.n_host = n_host
        self.host = make_host_batches(n_host, B, S, seed=1234 + 100 * rank)
        self.devb = [({k: torch.as_tensor(v, dtype=torch.float32).to(dev) for k, v in nb.items()},
                      torch.as_tensor(nz, dtype=torch.float32).to(dev)) for nb, nz in self.host]
        rng = np.random.RandomState(rank)
        self.masks = [np.where(rng.random_sample(B) > 0.1, 1, 0).astype(np.float32) for _ in range(n_host)]
        self.dmasks = [torch.as_tensor(m).to(dev) for m in self.masks]

    def sync_all(self):
        self.xdist.barrier()
        self.torch.cuda.synchronize(self.dev)

    def timed(self, run_one, K):
        torch = self.torch
        self.sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(K):
            run_one(i)
        e1.record()
        self.sync_all()
        return self.xdist.max_over_ranks(e0.elapsed_time(e1) * 1e-3)

    def dev_step(self, i, step=None):
        b, nz = self.devb[i % self.n_host]
        (step or self.step)(b, nz, cond_mask=self.dmasks[i % self.n_host])

    def run_device(self, warmup, K, step=None):
        for i in range(warmup):
            self.dev_step(i, step)
        return self.timed(lambda i: self.dev_step(i, step), K)

    def outputs(self):
        """Host copies of what the last step handed its caller (see --dump-outputs); call it before the next step."""
        torch = self.torch
        torch.cuda.synchronize(self.dev)
        s = self.state
        flat = {'params': s.params.flat, 'grads': self.eng.grads, 'adam_mu': s.opt_state.mu, 'adam_nu': s.opt_state.nu}
        n = s.params.flat.numel()
        idx = None
        if n > DUMP_MAX_ELEMS:
            # one seeded index from each of DUMP_MAX_ELEMS equal strides: the same sample at every run, spread over all leaves
            stride = n // DUMP_MAX_ELEMS
            pick = np.arange(DUMP_MAX_ELEMS) * stride + np.random.RandomState(0).randint(0, stride, DUMP_MAX_ELEMS)
            idx = torch.from_numpy(pick).to(self.dev)
        out = {'loss': self.eng.loss[0].float().cpu().numpy()}
        for k, v in flat.items():
            out[k] = (v if idx is None else v.index_select(0, idx)).float().cpu().numpy()
        return out

    def run_e2e(self, K):
        """host numpy inputs through the public API; the loss of every step is read back device->host inside the timed
        region, asynchronously into pinned memory (a real loop logs step i-1 while step i runs); the final synchronize of
        the timed region covers the last copy"""
        torch = self.torch
        ring = torch.zeros(K + 8, dtype=torch.float32).pin_memory()

        def host_step(i):
            nb, nz = self.host[i % self.n_host]
            loss = self.step(nb, nz, cond_mask=self.masks[i % self.n_host])
            ring[i % ring.numel()].copy_(loss, non_blocking=True)

        for i in range(3):
            host_step(i)
        h2d = self.step.h2d_bytes
        t = self.timed(host_step, K)
        return t, h2d, [float(v) for v in ring[:K]]


def bench_sampler(P, model, params, host_batch, S, views, steps, dev):
    """BASELINE.json's second metric: views/sec of the `steps`-step ancestral sampler with classifier-free guidance
    (sampling.py:119-151; cond + uncond evaluated as ONE forward of a 2B batch, CUDA-graph replayed per step)."""
    import torch
    runs = []
    for Bs in views:
        smp = P.Sampler(model, params, Bs, S, steps=steps, w=3.0, use_graph=True)
        sb = {k: np.concatenate([v] * ((Bs + len(v) - 1) // len(v)))[:Bs] for k, v in host_batch.items()}
        smp.capture(sb)                                 # static conditioning + graph capture (3 steps), not a full run
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        smp.sample(sb, seed=1)
        e1.record()
        torch.cuda.synchronize(dev)
        ts = e0.elapsed_time(e1) * 1e-3
        runs.append({'views_in_flight': Bs, 'views_per_sec': Bs / ts, 'ms_per_sampler_step': ts / len(smp.sched) * 1e3,
                     'seconds_per_run': ts})
        del smp
    return runs


def bench_full128(P, xdist, args, dev, peaks, rank, world):
    """BASELINE configs[2] (full 3DiM, 128x128, data parallel) and, at N=1, configs[3] (256-step sampler of the same model)."""
    import torch
    preset, S, B, fwd_flops = WORKLOADS['full128']
    B = args.full_batch or B
    K, W = max(1, min(args.steps, args.full_steps)), 3
    t0 = time.perf_counter()
    progress(f'full128: building the 439 M-parameter model, per-GPU batch {B}')
    tb = TrainBench(P, xdist, preset, S, B, 'bf16', dev, init_on_device=True, n_host=2)
    t_build = time.perf_counter() - t0
    progress(f'full128: built in {t_build:.1f} s (workspace {tb.eng.ws_bytes / 1e9:.1f} GB); timing {W}+{K} device steps')
    t_dev = tb.run_device(W, K)
    progress(f'full128: {t_dev / K * 1e3:.1f} ms/step; timing the end-to-end steps')
    t_e2e, h2d, losses = tb.run_e2e(K)
    progress('full128: train steps done')
    nparams = int(tb.state.params.flat.numel())
    train_flops = 3.0 * fwd_flops * B
    ms = t_dev / K * 1e3
    rec = {'workload': 'full128', 'model': 'full 3DiM X-UNet ch=256 ch_mult=(1,2,2,4) nrb=3 heads=8 emb_ch=1024', 'side': S,
           'params': nparams, 'per_gpu_batch': B, 'global_batch': B * world, 'n_gpus': world, 'steps': K, 'warmup': W,
           'ms_per_step': ms, 'images_per_sec': B * world * K / t_dev, 'e2e_images_per_sec': B * world * K / t_e2e,
           'h2d_bytes_per_step': int(h2d), 'step_tflops_per_gpu': train_flops / (ms * 1e-3) / 1e12,
           'step_tensor_frac_of_sustained': train_flops / (ms * 1e-3) / 1e12 / peaks['tf_sustained'],
           'mode': tb.step.mode, 'workspace_gb': tb.eng.ws_bytes / 1e9, 'build_seconds': t_build,
           'final_loss': losses[-1] if losses else None}
    if world > 1:
        # how much of the all-reduce the backward hides: the same step with the collectives switched off, and the bucketed
        # all-reduce of the same 1.755 GB buffer timed alone (CUDA events, max over ranks)
        step_noar = P.TrainStep(tb.state, allreduce=False)
        t_noar = tb.run_device(W, K, step_noar)
        bucket = tb.step.bucket_bytes // 4
        for _ in range(2):
            xdist.allreduce_sum_(tb.eng.grads, bucket_elems=bucket)
        t_ar = tb.timed(lambda i: xdist.allreduce_sum_(tb.eng.grads, bucket_elems=bucket), 5) / 5
        exposed = max(0.0, (t_dev - t_noar) / K)
        gb = nparams * 4 / 1e9
        rec['allreduce'] = {'bucket_bytes': nparams * 4, 'buckets': len(tb.step.reducer.ranges), 'bucket_mb': tb.step.bucket_bytes / 2 ** 20,
                            'alone_ms': t_ar * 1e3, 'bus_gbs': 2 * (world - 1) / world * gb / t_ar,
                            'step_ms_without_allreduce': t_noar / K * 1e3, 'exposed_ms': exposed * 1e3,
                            'overlap_fraction': max(0.0, 1.0 - exposed / t_ar) if t_ar > 0 else None}
        del step_noar
    if world == 1 and args.sampler_steps > 0:
        params = tb.state.params
        hb = tb.host[0][0]
        progress(f'full128: {args.sampler_steps}-step CFG sampler at 1 and 4 views in flight')
        rec['sampler'] = {'steps': args.sampler_steps, 'guidance_w': 3.0, 'side': S,
                          'runs': bench_sampler(P, tb.model, params, hb, S, (1, 4), args.sampler_steps, dev)}
    del tb
    torch.cuda.empty_cache()
    return rec


def main():
    if len(sys.argv) > 1 and sys.argv[1] == '--cpu-baseline-child':
        preset, S, Bs, budget = sys.argv[2], int(sys.argv[3]), int(sys.argv[4]), float(sys.argv[5])
        threads = int(sys.argv[6]) if len(sys.argv) > 6 else None
        print(json.dumps(cpu_baseline(preset, S, Bs, budget_s=budget, threads=threads)))
        return
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=30)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--workload', default='small64', choices=sorted(WORKLOADS))
    ap.add_argument('--batch', type=int, default=0, help='per-GPU batch (default: workload preset)')
    ap.add_argument('--dtype', default='bf16', choices=['bf16', 'fp32'])
    ap.add_argument('--no-graph', action='store_true')
    ap.add_argument('--skip-cpu-baseline', action='store_true')
    ap.add_argument('--sampler-steps', type=int, default=256, help='extra: DDPM sampler views/s at N=1 (0 = skip)')
    ap.add_argument('--no-full128', action='store_true', help='skip the full-3DiM 128x128 sub-record')
    ap.add_argument('--full-batch', type=int, default=0, help='per-GPU batch of the full128 sub-record (default 4)')
    ap.add_argument('--full-steps', type=int, default=8, help='timed steps of the full128 sub-record (<= --steps)')
    ap.add_argument('--ref-budget-s', type=float, default=200.0, help='wall-clock budget of --impl reference')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write the outputs of the last timed step to DIR/<name>.npy')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'b200':
        ap.error('--dump-outputs writes the outputs of the b200 path only')
    preset, S, B0, fwd_flops = WORKLOADS[args.workload]
    B = args.batch or B0
    if args.impl == 'reference':
        run_reference(args, preset, S, B)
        return

    import torch
    import novel_view_synthesis_3d_b200 as P
    from novel_view_synthesis_3d_b200 import dist as xdist
    if args.warmup < 3:
        args.warmup = 3
    local = xdist.init_from_env('nccl')
    world, rank = xdist.world_size(), xdist.rank()
    assert world == args.gpus or world == 1, f'--gpus {args.gpus} but WORLD_SIZE={world} (launch with torch.distributed.run)'
    dev = torch.device('cuda', local)
    torch.cuda.set_device(dev)
    peaks = load_peaks()

    progress(f'{args.workload}: building model / train state / step (world {world})')
    tb = TrainBench(P, xdist, preset, S, B, args.dtype, dev, use_graph=not args.no_graph, init_on_device=preset == 'full')
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    # ---- value: inputs resident in HBM; e2e: host numpy inputs through the public API, loss read back every step -------
    t_dev = tb.run_device(args.warmup, args.steps)
    dumped = tb.outputs() if args.dump_outputs and rank == 0 else None
    progress(f'{args.workload}: {t_dev / args.steps * 1e3:.3f} ms/step device-resident; timing end-to-end')
    t_e2e, h2d, losses = tb.run_e2e(args.steps)
    if dumped is not None:
        dumped['e2e_losses'] = np.asarray(losses, dtype=np.float32)
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, arr in dumped.items():
            np.save(os.path.join(args.dump_outputs, name + '.npy'), arr)
        progress(f'outputs of the last timed step written to {args.dump_outputs}: {sorted(dumped)}')
    clk = clocks.stop() if rank == 0 else None
    progress(f'{args.workload}: e2e {t_e2e / args.steps * 1e3:.3f} ms/step; kernel counts + roofline candidates')

    eng, state, model = tb.eng, tb.state, tb.model
    nf, nb_ = eng.count_kernels(state.params.flat)
    launches = (nf + nb_ + 1) * args.steps
    roof = dominant_kernel_roofline(P, model, B, S, peaks) if rank == 0 else None
    sampler = None
    if rank == 0 and world == 1 and args.sampler_steps > 0 and preset == 'small':
        progress(f'{args.sampler_steps}-step sampler (small model)')
        sampler = {'steps': args.sampler_steps, 'guidance_w': 3.0, 'model': preset, 'side': S,
                   'runs': bench_sampler(P, model, state.params, tb.host[0][0], S, (1, B), args.sampler_steps, dev)}
    mode = tb.step.mode
    ws_gb = eng.ws_bytes / 1e9
    full = None
    if args.workload == 'small64' and not args.no_full128 and args.dtype == 'bf16':
        del tb, eng, state, model
        torch.cuda.empty_cache()
        try:
            full = bench_full128(P, xdist, args, dev, peaks, rank, world)
        except Exception as ex:            # the headline must survive a failure of the extra record; say what happened
            full = {'workload': 'full128', 'error': f'{type(ex).__name__}: {ex}'[:400]}
    cb = None
    if rank == 0 and world == 1 and not args.skip_cpu_baseline:
        progress('cpu baseline (oracle on the host cores, in a child process with a hard wall-clock limit)')
        cb = cpu_baseline_guarded(preset, S, 2 if preset == 'small' else 1, budget_s=30.0 if preset == 'small' else 60.0)
    progress('done')
    if rank == 0:
        imgs = B * world * args.steps
        value = imgs / t_dev
        train_flops = 3.0 * fwd_flops * B
        line = {
            'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
            'ms_per_step': t_dev / args.steps * 1e3, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'bf16' if args.dtype == 'bf16' else 'f32', 'data': 'synthetic',
            'config': {'workload': args.workload, 'model': preset, 'side': S, 'per_gpu_batch': B, 'global_batch': B * world,
                       'parallelism': f'dp{world}', 'optimizer': 'adam lr1e-4', 'loss': 'frobenius (train.py:67)',
                       'cuda_graph': not args.no_graph, 'step_mode': mode,
                       'l2': 'no explicit flush: one step touches ~%.1f GB of activations+grads (>> 126 MB L2) and rotates over %d '
                             'different input batches' % (ws_gb, 4)},
            'e2e': {'value': imgs / t_e2e, 'unit': UNIT, 'h2d_bytes_per_step': int(h2d), 'd2h_bytes_per_step': 4,
                    'ms_per_step': t_e2e / args.steps * 1e3},
            'gpu_launches': int(launches), 'kernels_per_step': {'forward': nf, 'backward': nb_, 'adam': 1},
            'step_tflops': train_flops / (t_dev / args.steps) / 1e12,
            'step_tensor_frac_of_sustained': train_flops / (t_dev / args.steps) / 1e12 / peaks['tf_sustained'],
            'roofline': roof, 'sampler': sampler, 'full128': full, 'cpu_baseline': cb, 'clocks': clk,
            'final_loss': losses[-1] if losses else None,
        }
        print(json.dumps(line))
    if xdist.is_dist():
        # captured step graphs hold NCCL kernels of this process group: release them before tearing it down
        import gc
        tb = None
        gc.collect()
        torch.cuda.synchronize(dev)
        torch.distributed.destroy_process_group()


if __name__ == '__main__':
    main()

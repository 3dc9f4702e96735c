#!/usr/bin/env python
"""bench.py - train tokens/sec (text+latent) at d=512 L=8 seq=1024 (BASELINE.json `metric`, configs[1]).

    python bench.py --gpus N --steps K --warmup W            # B200 arm (one process per GPU under torchrun for N > 1)
    python bench.py --impl reference --gpus N --steps K ...  # reference arm: the reference's CPU algorithm on the host cores

A "step" = forward + backward + gradient all-reduce (N > 1) + fused Adam (+ bf16 weight repack) over one synthetic batch of
`--batch` sequences x 1024 packed tokens per GPU (weak scaling).  Prints ONE JSON line on rank 0.

  value  : whole-job tokens/s with the packed batch already resident in HBM (device-timed, CUDA events, max over ranks); the step is a
           CUDA-graph replay (`DataParallelTrainer.step_packed`), `--no-graph` launches the same kernels eagerly
  e2e    : same metric through the public API - `DataParallelTrainer.step(list_of_samples)`: Python pack/route, H2D of the token metadata
           and of the latents from pinned host memory every step (copy stream), the step graph, and a D2H read of every step's loss
           (fetched one step late through a side stream so the host packs the next batch meanwhile)
  roofline: dominant kernel family of the step (by measured device time of an eager profiling pass), algorithmic FLOPs / measured time
           against the sustained measured bf16 peak; `roofline.kernels` lists the five largest kernel instances with their ncu DRAM traffic
  cpu_baseline: the oracle port of the reference algorithm (oracle/torch_reference.py, fp32, per-token conditioning, dense masks - the
           reference's cost structure) timed on this box's host cores on a bounded sample
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CTOR = dict(num_text_tokens = 256, dim_latent = 384, modality_default_shape = (256,), transformer = dict(dim = 512, depth = 8))
CTOR4 = dict(num_text_tokens = 256, dim_latent = (384, 192), modality_default_shape = ((4,), (2,)), transformer = dict(dim = 512, depth = 8))
SEQ = 1024
WORKLOADS = {
    'train': 'configs[1]: single-modality text+latent d=512 depth=8 dim_latent=384 seq=1024',
    'config4': 'configs[3]: two modalities dim_latent=(384,192), ~15 short interleaved spans per 1024-token sample (span-mask attention stress)',
    'sample_many': 'configs[4]: sample_many, 32 mixed prompts, kv cache, cfg_scale=3.0, forced 256x384 modality (16 midpoint steps), greedy text to max_length 512',
}
ALGO_TRAIN_FLOP_PER_TOKEN = 195.4e6            # SURVEY.md section 8(d): 65.1 MFLOP/token forward x 3
METRIC = 'train tokens/sec (text+latent) at d=512 L=8 seq=1024'


def peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.isfile(path):
        p = json.load(open(path))
        return dict(hbm = p['hbm_gbs'], tf_burst = p['bf16_tflops'], tf_sustained = p.get('bf16_tflops_sustained', p['bf16_tflops']), src = 'measured')
    return dict(hbm = 6650., tf_burst = 1590., tf_sustained = 1400., src = 'fallback')


class ClockSampler:
    """samples SM clocks / throttle reasons DURING the timed region - from a separate PROCESS (in-process NVML, nvidia-smi as the fallback).
    A sampler THREAD in this process doubled the wall time of the launch-bound sample_many loop (25 k ctypes calls per sample_many: every one of them
    drops and re-takes the GIL, which is only free of charge while the interpreter has a single thread); spawning nvidia-smi five times a second
    holds driver locks for tens of ms each."""
    Q = 'clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'
    POLLER = r"""
import os, subprocess, sys, time
uuid, index, Q, period = sys.argv[1], int(sys.argv[2]), sys.argv[3], float(sys.argv[4])
parent, t_end = os.getppid(), time.time() + 3600.0       # never outlive the benchmark process
try:
    import pynvml
    pynvml.nvmlInit()
    try: h = pynvml.nvmlDeviceGetHandleByUUID(uuid)
    except Exception: h = pynvml.nvmlDeviceGetHandleByIndex(index)
    get = getattr(pynvml, 'nvmlDeviceGetCurrentClocksEventReasons', None) or pynvml.nvmlDeviceGetCurrentClocksThrottleReasons
except Exception:
    h = None
while os.getppid() == parent and time.time() < t_end:
    try:
        if h is not None:
            mask = int(get(h)); act = lambda bit: 'Active' if mask & bit else 'Not Active'
            row = [str(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)), str(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)),
                   str(pynvml.nvmlDeviceGetPowerUsage(h) / 1e3), act(0x8), act(0x40), act(0x20), act(0x4)]
        else:
            out = subprocess.run(['nvidia-smi', '--query-gpu=' + Q, '--format=csv,noheader,nounits', '-i', str(index)], capture_output = True, text = True, timeout = 5).stdout
            row = [c.strip() for c in out.strip().split(',')]
        print(','.join([repr(time.time())] + row), flush = True)
    except Exception:
        pass
    time.sleep(period)
"""

    def __init__(self, index, period = 0.2):
        """launches the poller at once (interpreter + NVML start-up take a few hundred ms - longer than a 10-step timed region); only the rows stamped
        between start() and stop() are kept"""
        self.index, self.rows, self.proc, self.t0 = index, [], None, None
        try:
            import torch
            uuid = 'GPU-' + str(torch.cuda.get_device_properties(self.index).uuid)
        except Exception:
            uuid = 'none'
        try:
            if os.environ.get('TFX_BENCH_NO_CLOCKS'): raise RuntimeError('clock sampling disabled (diagnosis only: the line is then not a valid bench line)')
            self.proc = subprocess.Popen([sys.executable, '-c', self.POLLER, uuid, str(self.index), self.Q, str(period)], stdout = subprocess.PIPE, stderr = subprocess.DEVNULL, text = True)
        except Exception:
            self.proc = None

    def start(self):
        self.t0 = time.time()

    def stop(self):
        """ends the sampling: terminates the poller and keeps the rows stamped inside [start(), now]"""
        if self.proc is None:
            return
        t1 = time.time()
        try:
            self.proc.terminate()
            out, _ = self.proc.communicate(timeout = 5)
            rows = [[c.strip() for c in ln.split(',')] for ln in out.strip().splitlines() if ln.strip()]
            inside = [r[1:] for r in rows if self.t0 is not None and self.t0 - 0.05 <= float(r[0]) <= t1 + 0.05]
            # a timed region shorter than one polling period: the sample nearest to it (taken under the same load: the warm-up runs the same step)
            self.rows = inside or [r[1:] for r in rows[-1:]]
        except Exception:
            pass
        self.proc = None

    def summary(self):
        sm = sorted(int(float(r[0])) for r in self.rows if r and r[0].replace('.', '').isdigit())
        reasons = set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for r in self.rows:
            for n, v in zip(names, r[3:7]):
                if v.lower().startswith('active'):
                    reasons.add(n)
        mx = [int(float(r[1])) for r in self.rows if len(r) > 1 and r[1].replace('.', '').isdigit()]
        return dict(sm_mhz = sm[len(sm) // 2] if sm else None, sm_max_mhz = max(mx) if mx else None, reasons = sorted(reasons), samples = len(self.rows))


# --------------------------------------------------------------------------------------------- reference arm / cpu baseline
def cpu_port_tokens_per_s(batch: int, steps: int, warmup: int):
    """Times the oracle port (the checker, here only as the reported CPU baseline) - fwd + bwd + Adam on the host cores; MEDIAN of `steps`
    timed steps after `warmup` (BASELINE.md section 3).  Threads: every core of the box (torch intra-op pool), stated in the record."""
    import statistics
    import torch
    from transfusion_pytorch_b200 import Transfusion, synth
    from oracle.torch_reference import OracleEngine
    cores = usable_cores()
    torch.set_num_threads(cores)
    torch.manual_seed(0)
    model = Transfusion(**CTOR, prob_uncond = 0.)
    synth.fill_parameters_(model, seed = 0)
    model._engine = OracleEngine(model)
    opt = torch.optim.Adam(model.parameters(), lr = 1e-4)
    times_ = []
    for s in range(warmup + steps):
        b = synth.config2_batch(batch, seed = 500 + s)
        t0 = time.perf_counter()
        opt.zero_grad(set_to_none = True)
        loss = model(b, times = synth.config2_times(batch, seed = s))
        loss.backward()
        opt.step()
        dt = time.perf_counter() - t0
        if s >= warmup:
            times_.append(dt)
    ms = 1e3 * statistics.median(times_)
    return batch * SEQ / (ms / 1e3), ms, torch.get_num_threads()


def usable_cores():
    """host threads the CPU arm may really use: the affinity mask, bounded by the cgroup CPU quota (a 128-thread pool on a container with a smaller
    quota thrashes: measured 15 tokens/s instead of ~400) """
    cores = os.cpu_count() or 1
    try:
        cores = len(os.sched_getaffinity(0))
    except AttributeError:
        pass
    try:
        quota, period = open('/sys/fs/cgroup/cpu.max').read().split()[:2]
        if quota != 'max':
            cores = max(1, min(cores, int(float(quota) / float(period))))
    except (OSError, ValueError):
        pass
    # a 128-thread intra-op pool across two NUMA nodes measured SLOWER (15 tokens/s) than 64 threads (~420 tokens/s) on this pool's hosts: one node's worth
    return min(cores, int(os.environ.get('TFX_CPU_THREADS', 64)))


def numa_note():
    try:
        nodes = [d for d in os.listdir('/sys/devices/system/node') if d.startswith('node')]
        return f'{len(nodes)} NUMA node(s), threads not pinned (torch intra-op pool over all cores)'
    except OSError:
        return 'NUMA layout unknown'


def run_reference_arm(args):
    rank = int(os.environ.get('RANK', 0))
    if rank != 0:
        return
    # b = 4, median of the timed fwd + bwd + Adam steps (BASELINE.md section 3 runs it with --warmup 2 --steps 3)
    b = 4
    steps, warm = args.steps, args.warmup
    tps, ms, cores = cpu_port_tokens_per_s(b, steps, warm)
    line = dict(impl = 'reference', metric = METRIC, value = tps, unit = 'tokens/s', n_gpus = args.gpus, steps = args.steps, warmup = args.warmup, ms_per_step = ms,
                higher_is_better = True, scaling = 'weak', vs_baseline = None, dtype = 'f32', data = 'synthetic',
                config = dict(workload = WORKLOADS['train'], global_batch = b, seq_len = SEQ, parallelism = 'cpu'),
                cpu_baseline = dict(value = tps, unit = 'tokens/s', cores = cores, kind = 'port',
                                    sample = f'{b} sequences x {SEQ} tokens per step, fwd+bwd+Adam, fp32, median of {steps} timed steps after {warm} warm-up; {numa_note()}'),
                e2e = dict(value = tps, unit = 'tokens/s', h2d_bytes_per_step = 0, d2h_bytes_per_step = 0))
    emit(line)


# --------------------------------------------------------------------------------------------- B200 arm
def family_model(name, args_, eng, rb):
    """(family, algorithmic flops, algorithmic bytes) of one C-ABI launch, from its arguments.  FLOPs use the UN-padded problem sizes (the engine
    pads the FFN inner dim 1365 -> 1408, the packed qkvg rows 1544 -> 1664, the time-MLP K 513 -> 576, vocab 390 -> 392: padding is not work).
    Bytes = the tensors the kernel must read + write once (DESIGN.md section 4), used for the GB/s of the HBM-bound kernels."""
    a = args_
    D, HI, H, Ip, inner, M = eng.D, eng.HI, eng.H, eng.Ip, eng.inner, rb.M
    real = {eng.Ip: eng.inner, 2 * eng.Ip: 2 * eng.inner, eng.NQ: 3 * HI + H, eng.Kt: D + 1, eng.Vp: eng.V}
    for dl, dlp in zip(eng.dls, eng.dlp):
        real.setdefault(dlp, dl)
    r = lambda d: real.get(d, d)
    if name == 'gemm_store':
        m, n, k = a[6], a[7], a[8]
        return 'gemm(tcgen05)', 2.0 * r(m) * r(n) * r(k), 2.0 * (m * k + n * k) + 4.0 * m * n
    if name == 'gemm_qkvg':
        m, h, d = a[4], a[5], a[6]
        return 'gemm(tcgen05)', 2.0 * m * (3 * h * 64 + h) * d, 2.0 * m * d + 2.0 * eng.NQ * d + 6.0 * m * h * 64
    if name == 'gemm_resid':
        m, n, k = a[7], a[8], a[9]
        return 'gemm(tcgen05)', 2.0 * m * n * r(k), 2.0 * m * k + 2.0 * n * k + 8.0 * m * n + 2.0 * m * n
    if name == 'gemm_geglu':
        m, k = a[5], a[7]
        return 'gemm(tcgen05)', 2.0 * m * 2 * inner * k, 2.0 * m * k + 4.0 * Ip * k + 6.0 * m * Ip
    pairs = float(((rb.kv_limit.astype('int64') - (rb.cu[:-1].repeat(rb.seq_lens))) + 1).sum())
    if name in ('attn_fwd_tc', 'attn_fwd_ts'):
        return 'attention', 4.0 * pairs * 64 * H, 8.0 * M * HI
    if name == 'attn_fwd':
        return 'attention', 0, 0          # general kernel: returns at once when the tcgen05 path is active (flops credited to attn_fwd_tc)
    if name in ('attn_bwd_tc', 'attn_bwd_ts'):
        return 'attention', 10.0 * pairs * 64 * H, 8.0 * M * HI + 8.0 * M * HI + 2.0 * M * HI      # q k v dO in; dq dk fp32 + dv bf16 out
    if name == 'attn_bwd':
        return 'attention', 0, 0
    fam = 'hbm-bound rows/elementwise'
    by = 0.0
    if name == 'adaln_fwd': by = M * (4 * D + 2 * D + 8)
    elif name == 'adaln_bwd': by = M * (4 * D + 4 * D + 8 * D + 8)
    elif name == 'resid_bwd': by = M * (4 * D + 2 * D + 2 * D) if a[1] is not None else M * (4 * D + 2 * D)
    elif name == 'attn_residual_fwd': by = M * (a[1] * 4 * D + 4 * D + 2 * D)
    elif name == 'attn_residual_bwd2': by = M * (a[1] * 2 * D * a[2] + a[7] * 4 * D + (8 * D if a[2] else 0) + 4 * D)
    elif name == 'attn_residual_fwd_h16': by = M * (a[1] * 2 * D + 4 * D + 2 * D)
    elif name == 'attn_residual_bwd_h16': by = M * (a[2] * 2 * D + a[2] * (4 * D if a[-1] else 8 * D) + 8 * D)
    elif name == 'attn_residual_bwd': by = M * (a[2] * 4 * D + a[2] * (4 * D if a[-1] else 8 * D) + 8 * D)
    elif name == 'geglu_bwd': by = M * (2 * Ip + 4 * Ip + 4 * Ip)
    elif name == 'qk_bwd_pack': by = M * (8 * HI + 4 * HI + 4 * HI + 16 * H)
    elif name == 'attn_bwd_prep': by = M * (4 * HI + 2 * HI + 4 * HI + 8 * H)
    elif name == 'rmsnorm_fwd': by = M * (4 * D + 4 * D + 2 * D)
    elif name == 'rmsnorm_bwd': by = M * 12 * D
    elif name == 'embed_assemble': by = M * (4 * D + 4 * D + 2 * D)
    elif name == 'embed_bwd': by = M * 8 * D
    elif name == 'axpy_f32': by = 12.0 * a[3]
    elif name == 'adam_step': by = 28.0 * a[4]
    elif name == 'ce_fwd_bwd': by = M * (4 * eng.Vp + 2 * eng.Vp)
    elif name == 'cast_pack_multi': by = 6.0 * eng.flat.numel()
    elif name == 'flow_noise': by = a[7] * a[8] * (8 + 2 + 4)
    elif name == 'mse_fwd_bwd': by = a[7] * a[8] * (8 + 2)
    elif name == 'scatter_add_rows': by = a[3] * 12 * D
    elif name in ('colsum_f32',): by = 4.0 * a[2] * a[3]
    elif name in ('colsum_bf16',): by = 2.0 * a[2] * a[3]
    return fam, 0, float(by)


def log(*a):
    print(f'[bench {time.strftime("%H:%M:%S")}]', *a, file = sys.stderr, flush = True)


# --------------------------------------------------------------------------------------------- --dump-outputs
DUMP_LIMIT = 64 << 20                 # bytes written by --dump-outputs in all
DUMP_PARAMS = 1 << 21                 # parameter values in the fixed sample (float32 values + float64 updates: 24 MB)


def param_sample(model):
    """the values of a fixed, seeded sample of every parameter element (named_parameters order, identical from run to run), float32 on the host"""
    import torch
    flat = torch.cat([p.detach().reshape(-1) for p in model.parameters()])
    idx = torch.randint(0, flat.numel(), (min(DUMP_PARAMS, flat.numel()),), generator = torch.Generator().manual_seed(0)).sort().values
    return flat[idx.to(flat.device)].float().cpu().numpy()


def write_outputs(out_dir, arrays):
    """writes every (name, array) as out_dir/<name>.npy (float32 stays float32, everything else becomes float64) while the total stays within DUMP_LIMIT"""
    import numpy as np
    os.makedirs(out_dir, exist_ok = True)
    total = 0
    for name, a in arrays:
        a = np.asarray(a)
        a = a.astype(np.float32 if a.dtype == np.float32 else np.float64)
        if total + a.nbytes > DUMP_LIMIT:
            log(f'--dump-outputs: {DUMP_LIMIT >> 20} MB reached, {name} and what follows it not written')
            return
        np.save(os.path.join(out_dir, name + '.npy'), a)
        total += a.nbytes
    log(f'--dump-outputs: {total / 2 ** 20:.1f} MB written to {out_dir}')


def run_b200_arm(args):
    import torch
    import torch.distributed as dist
    from transfusion_pytorch_b200 import Transfusion, synth
    from transfusion_pytorch_b200.data_parallel import DataParallelTrainer, AsyncScalar
    from transfusion_pytorch_b200.modality_processing import pack_batch

    world = int(os.environ.get('WORLD_SIZE', 1))
    rank = int(os.environ.get('RANK', 0))
    local = int(os.environ.get('LOCAL_RANK', 0))
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault('NCCL_DEBUG_FILE', '/dev/stderr')          # whatever NCCL_DEBUG the caller chose goes to stderr: stdout carries ONE JSON line
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id = torch.device('cuda', local))
    dev = torch.device('cuda', local)
    sampler = ClockSampler(local) if rank == 0 else None          # (the poller process starts now; rows are kept from sampler.start() on)
    B = args.batch if args.scaling == 'weak' else max(1, args.batch // world)      # strong scaling: --batch is the GLOBAL batch, split over the ranks
    torch.manual_seed(0)
    cfg4 = args.workload == 'config4'
    model = Transfusion(**(CTOR4 if cfg4 else CTOR)).to(dev)      # prob_uncond = 0.1 (reference default), train mode
    synth.fill_parameters_(model, seed = 0)
    model.train()
    trainer = DataParallelTrainer(model, lr = 1e-4, cuda_graph = not args.no_graph, overlap = not args.no_overlap)
    eng = model.engine
    eng.ensure_attached()

    POOL = 4
    if cfg4:
        host_batches = [synth.config4_batch(B, seed = 1000 * rank + i) for i in range(POOL)]
        nm = max(sum(isinstance(p, tuple) for p in s_) for b in host_batches for s_ in b)
        host_times = [torch.rand(B, nm, generator = torch.Generator().manual_seed(7 + 1000 * rank + i)) for i in range(POOL)]
        host_batches = [[[(p[0], p[1].pin_memory()) if isinstance(p, tuple) else p for p in s_] for s_ in b] for b in host_batches]
    else:
        host_batches = [synth.config2_batch(B, seed = 1000 * rank + i) for i in range(POOL)]
        host_batches = [[[p.pin_memory() if p.is_floating_point() else p for p in s_] for s_ in b] for b in host_batches]
        host_times = [synth.config2_times(B, seed = 1000 * rank + i) for i in range(POOL)]

    # ---- device-resident variant: packed descriptors + latents already in HBM
    packed = []
    for b, t in zip(host_batches, host_times):
        samples = [[torch.tensor([model.sos_id]), *s_, torch.tensor([model.eos_id])] for s_ in b]
        rb = pack_batch(samples, t, model, return_loss = True, return_embed = False)
        lat = model._latents_to_device(rb)
        eng.upload(rb)
        packed.append((rb, lat))
    assert packed[0][0].M == B * SEQ, packed[0][0].M
    log('packed', POOL, 'batches; M =', packed[0][0].M)

    profiling = [False]                                      # roofline pass: every rank launches eagerly (same collectives on all ranks)
    def step_resident(i):
        rb, lat = packed[i % POOL]
        if trainer.cuda_graph and not profiling[0]:
            return trainer.step_packed(rb, lat)              # CUDA-graph replay of the step (after two eager steps of this shape)
        return trainer.step_packed_eager(rb, lat)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing = True), torch.cuda.Event(enable_timing = True)
        e0.record()
        t_host = time.perf_counter()
        for i in range(steps):
            timed.last = fn(i)
        timed.host_ms = 1e3 * (time.perf_counter() - t_host) / steps      # CPU time to enqueue one step (no sync inside)
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device = dev)
        if world > 1:
            dist.all_reduce(ms, op = dist.ReduceOp.MAX)
        return ms.item()

    # a step graph is captured per shape signature after two eager steps of that shape: config 4's batches differ in span / condition-row counts, so every
    # one of the POOL rotating batches has to be seen three times before the timed region replays graphs only
    for i in range(max(args.warmup, 3 * POOL) if (cfg4 and trainer.cuda_graph) else args.warmup):
        step_resident(i)
        torch.cuda.synchronize(); log('warmup step', i, 'done')
    dump = args.dump_outputs and rank == 0
    params_before = param_sample(model) if dump else None
    if sampler: sampler.start()
    l0 = eng.ops.launches
    ms_total = timed(step_resident, args.steps)
    host_enqueue_ms = timed.host_ms
    launches = eng.ops.launches - l0
    if sampler:
        sampler.stop()
    if dump:                        # before the e2e and profiling steps below train the model further
        params = param_sample(model)
        write_outputs(args.dump_outputs, [('loss', timed.last.detach().float().reshape(1).cpu().numpy()), ('params', params),
                                          ('param_update', params.astype('float64') - params_before)])
    ms_step = ms_total / args.steps
    log('resident ms/step', ms_step)
    value = world * B * SEQ / (ms_step / 1e3)

    # ---- end to end through the public API (pack/route + H2D + D2H every step), over the SAME number of steps
    # Every step: Python pack/route of host samples, H2D of that step's inputs from pinned memory, fwd + bwd + optimizer, and a D2H
    # read of a loss.  The loss that is read inside step i is the one of step i-1 (asynchronous logging: the value is fetched while step i
    # runs on the device, so the host packs step i+1 instead of idling); the last loss is read before the timed region closes.
    h2d = [0]
    pending = [None]
    host_e2e = []
    def step_e2e(i):
        b, t = host_batches[i % POOL], host_times[i % POOL]
        t_h = time.perf_counter()
        loss = trainer.step(b, times = t)
        host_e2e.append(1e3 * (time.perf_counter() - t_h))
        rb = model._last_batch
        h2d[0] = rb.dev.get('h2d_bytes', 0) + getattr(rb, 'latent_h2d_bytes', 0)
        prev, pending[0] = pending[0], AsyncScalar(loss)      # D2H copy of this step's loss, on a side stream
        return prev.value() if prev is not None else None    # ... read one step later: waits for step i-1 only
    def e2e_loop(i):
        step_e2e(i)
        if i == e2e_loop.last:
            pending[0].value(); pending[0] = None              # drain: the final step's loss is read inside the timed region too
    for i in range(max(3, min(args.warmup, 3))):
        step_e2e(i)
    pending[0].value(); pending[0] = None
    e2e_steps = args.steps
    e2e_loop.last = e2e_steps - 1
    ms_e2e = timed(e2e_loop, e2e_steps) / e2e_steps
    e2e_value = world * B * SEQ / (ms_e2e / 1e3)
    log('e2e ms/step', ms_e2e)

    # replicas must still be identical after all those steps (every rank applied the same averaged gradient)
    spread = None
    if world > 1:
        cs = eng.flat.double().sum().reshape(1)
        lo, hi = cs.clone(), cs.clone()
        dist.all_reduce(lo, op = dist.ReduceOp.MIN); dist.all_reduce(hi, op = dist.ReduceOp.MAX)
        spread = float((hi - lo).item())

    # ---- per-kernel-family device time of one step (profiling pass, not part of the reported throughput)
    # every rank runs the step (it contains the gradient all-reduce); only rank 0 records per-launch events
    roof = None
    profiling[0] = True
    if rank == 0:
        eng.ops.timing = {}
        eng.ops.order = [] if args.dump_launches else None
    step_resident(0)
    barrier()
    if rank == 0:
        fam, inst = {}, {}
        rb = packed[0][0]
        for name, recs in eng.ops.timing.items():
            for e0, e1, a in recs:
                f, fl, by = family_model(name, a, eng, rb)
                ms = e0.elapsed_time(e1)
                d = fam.setdefault(f, dict(ms = 0., flops = 0., bytes = 0., launches = 0))
                d['ms'] += ms; d['flops'] += fl; d['bytes'] += by; d['launches'] += 1
                label = name + (f'[M={a[6]},N={a[7]},K={a[8]}]' if name == 'gemm_store' else f'[K={a[9]}]' if name == 'gemm_resid' else '[assemble]' if (name == 'attn_residual_bwd2' and not a[2]) else '')      # per kernel instance (entry point + problem shape)
                k = inst.setdefault(label, dict(ms = 0., flops = 0., bytes = 0., launches = 0, family = f))
                k['ms'] += ms; k['flops'] += fl; k['bytes'] += by; k['launches'] += 1
        if args.dump_launches:      # entry points of the profiled step in launch order, with the labels of the roofline table (tools/ncu_traffic.py aligns an ncu capture with it)
            seen, labels = {}, []
            for name in eng.ops.order:
                a = eng.ops.timing[name][seen.get(name, 0)][2]; seen[name] = seen.get(name, 0) + 1
                labels.append(name + (f'[M={a[6]},N={a[7]},K={a[8]}]' if name == 'gemm_store' else f'[K={a[9]}]' if name == 'gemm_resid' else '[assemble]' if (name == 'attn_residual_bwd2' and not a[2]) else ''))
            json.dump(dict(key = f'{args.workload}:b{B}', launches = labels), open(args.dump_launches, 'w'))
        eng.ops.timing = None
        eng.ops.order = None
        pk = peaks()
        tot = sum(d['ms'] for d in fam.values())
        top = max((f for f in fam if fam[f]['flops'] > 0), key = lambda f: fam[f]['ms'])
        ach = fam[top]['flops'] / (fam[top]['ms'] / 1e3) / 1e12
        # DRAM traffic per launch from the committed ncu `--set full` capture of THIS command line (profiles/r02_traffic.json: {batch: {label: bytes}})
        tpath = os.path.join(ROOT, 'profiles', 'r02_traffic.json')
        tmap = (json.load(open(tpath)) if os.path.isfile(tpath) else {}).get(f'{args.workload}:b{B}', {})
        def fam_row(d):
            row = dict(ms = round(d['ms'], 3), share = round(d['ms'] / tot, 3), launches = d['launches'])
            if d['flops']:
                row.update(tflops = round(d['flops'] / (d['ms'] / 1e3) / 1e12, 1), frac_of_tensor_peak = round(d['flops'] / (d['ms'] / 1e3) / 1e12 / pk['tf_sustained'], 3))
            else:
                row.update(gbs = round(d['bytes'] / (d['ms'] / 1e3) / 1e9, 1), frac_of_hbm_peak = round(d['bytes'] / (d['ms'] / 1e3) / 1e9 / pk['hbm'], 3))
            return row
        def inst_row(lbl, k):
            row = dict(kernel = lbl, family = k['family'], launches = k['launches'], us_per_launch = round(1e3 * k['ms'] / k['launches'], 1), share_of_step = round(k['ms'] / tot, 3))
            if k['flops']:
                a_ = k['flops'] / (k['ms'] / 1e3) / 1e12
                row.update(bound = 'tensor', achieved = round(a_, 1), unit = 'TFLOP/s', frac = round(a_ / pk['tf_sustained'], 3))
                if k['bytes']:      # the fused-epilogue GEMMs move fp32 residual rows: their HBM roofline is reported beside the tensor one
                    row.update(hbm_gbs = round(k['bytes'] / (k['ms'] / 1e3) / 1e9, 1), hbm_frac = round(k['bytes'] / (k['ms'] / 1e3) / 1e9 / pk['hbm'], 3))
            else:
                a_ = k['bytes'] / (k['ms'] / 1e3) / 1e9
                row.update(bound = 'hbm', achieved = round(a_, 1), unit = 'GB/s', frac = round(a_ / pk['hbm'], 3))
            row['algorithmic_bytes'] = int(k['bytes'] / k['launches'])
            row['traffic'] = tmap.get(lbl)
            return row
        ranked = sorted(inst.items(), key = lambda kv: -kv[1]['ms'])
        # DRAM traffic of the dominant family, per launch like `achieved`: every instance's ncu bytes x its launches (None when an instance was not captured)
        fam_inst = [(lbl, k) for lbl, k in inst.items() if k['family'] == top]
        fam_traffic = (int(sum(tmap[lbl] * k['launches'] for lbl, k in fam_inst) / max(1, sum(k['launches'] for _, k in fam_inst)))
                       if fam_inst and all(lbl in tmap for lbl, _ in fam_inst) else None)
        whole = value * ALGO_TRAIN_FLOP_PER_TOKEN / 1e12 / world
        roof = dict(bound = 'tensor', kernel = top, achieved = ach, peak = pk['tf_sustained'], unit = 'TFLOP/s', frac = ach / pk['tf_sustained'],
                    traffic = fam_traffic, traffic_kernel = top + ' (average per launch over the family: ncu DRAM bytes of every instance x its launches / launches)',
                    largest_kernel = dict(kernel = ranked[0][0], traffic = tmap.get(ranked[0][0])) if ranked else None,
                    peak_source = pk['src'] + ' (sustained bf16 GEMM; burst ' + str(pk['tf_burst']) + ', HBM copy ' + str(pk['hbm']) + ' GB/s)', share_of_step = fam[top]['ms'] / tot,
                    flops_model = 'un-padded problem sizes (FFN inner 1365, qkvg rows 1544, time-MLP K 513, vocab 390)',
                    families = {f: fam_row(d) for f, d in fam.items()},
                    whole_step_tflops = whole, whole_step_frac = whole / pk['tf_sustained'], whole_step_frac_of_burst = whole / pk['tf_burst'],
                    kernels = [inst_row(lbl, k) for lbl, k in ranked[:28]])

    if rank == 0:
        clocks = sampler.summary() if sampler else None
        cpu = None
        log('roofline pass done')
        if world == 1 and not args.no_cpu_baseline and not cfg4:
            tps, ms_cpu, cores = cpu_port_tokens_per_s(2, 2, 1)
            cpu = dict(value = tps, unit = 'tokens/s', cores = cores, kind = 'port',
                       sample = f'2 sequences x {SEQ} tokens per step (fwd+bwd+Adam, fp32), median of 2 timed steps after 1 warm-up; {numa_note()}; the full BASELINE.md section-3 protocol '
                                '(b=4, 2+3 steps) is `--impl reference`')
        line = dict(metric = METRIC if not cfg4 else METRIC + ' [config 4: two modalities, span-mask stress]', value = value, unit = 'tokens/s', n_gpus = world, steps = args.steps,
                    warmup = args.warmup, ms_per_step = ms_step, higher_is_better = True,
                    scaling = args.scaling, vs_baseline = None, dtype = 'bf16', data = 'synthetic',
                    config = dict(workload = WORKLOADS[args.workload], global_batch = world * B, per_gpu_batch = B,
                                  grad_allreduce = (f'fp32 flat buffer, ~{trainer.bucket_bytes >> 20} MB per-layer buckets on a side stream overlapped with backward inside the step graph'
                                                    if trainer.overlap else 'one fp32 all-reduce after backward') if world > 1 else None,
                                  seq_len = SEQ, parallelism = f'dp{world}', optimizer = 'fused Adam', launch = 'cuda graph replay' if trainer.cuda_graph else 'eager',
                                  l2 = 'per-step working set (>10 GB of activations) is far larger than the 126 MB L2; 4 rotating input batches'),
                    e2e = dict(value = e2e_value, unit = 'tokens/s', ms_per_step = ms_e2e, steps = e2e_steps, h2d_bytes_per_step = int(h2d[0]), d2h_bytes_per_step = 4,
                               loss_read = 'every step, deferred by one step (asynchronous logging)',
                               host_ms_per_step = round(sum(host_e2e[-e2e_steps:]) / e2e_steps, 3)),
                    gpu_launches = int(launches), host_enqueue_ms_per_step = round(host_enqueue_ms, 3), clocks = clocks, roofline = roof, cpu_baseline = cpu,
                    replica_checksum_spread = spread)
        emit(line)
        sys.stdout.flush()
    if world > 1:
        # captured graphs hold NCCL work: drop them and drain the device before the process group goes away.  The destructor has been
        # observed to hang after graph-captured collectives, so it runs under a watchdog; every rank has passed the barrier by then.
        trainer._graphs.clear()
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush(); sys.stderr.flush()
        done = threading.Event()
        def teardown():
            try:
                dist.destroy_process_group()
            finally:
                done.set()
        threading.Thread(target = teardown, daemon = True).start()
        if not done.wait(20):
            log('process-group teardown did not finish in 20 s: exiting without it')
            os._exit(0)


# --------------------------------------------------------------------------------------------- sample_many workload (BASELINE.json configs[4])
def config5_prompts(n_each, seed = 0):
    import torch
    g = torch.Generator().manual_seed(4242 + seed)
    prompts = []
    for _ in range(n_each):                                   # README.md:162-167 prompt forms, SURVEY.md 8(d) config 5
        prompts.append(torch.randint(0, 256, (16,), generator = g))
        prompts.append((0, torch.randn(int(torch.randint(4, 65, (1,), generator = g)), 384, generator = g)))
        prompts.append(None)
        prompts.append([torch.randint(0, 256, (8,), generator = g), (0, torch.randn(int(torch.randint(6, 33, (1,), generator = g)), 384, generator = g))])
    noise = torch.randn(256, 384, generator = g)
    return prompts, noise


def run_sample_many(args):
    """configs[4]: wall time and generated tokens/s of `sample_many` (32 mixed prompts, kv cache, cfg 3, 16 midpoint steps over a forced 256 x 384 modality, greedy
    text to max_length 512), KV-read bandwidth of the text loop, the FLOP saving over prefix recomputation, and the reference algorithm on the host beside it."""
    import copy
    import torch
    from transfusion_pytorch_b200 import Transfusion, synth
    dev = torch.device('cuda', int(os.environ.get('LOCAL_RANK', 0)))
    torch.cuda.set_device(dev)
    sampler = ClockSampler(dev.index or 0, period = 1.0)      # the loop is host-latency-bound: NVML queries take driver locks, one per second is enough here
    torch.manual_seed(0)
    model = Transfusion(**CTOR).to(dev).eval()
    synth.fill_parameters_(model, seed = 0)
    n_prompts, max_length, steps_ode, Lm = args.prompts, args.max_length, 16, 256
    prompts, noise = config5_prompts(n_prompts // 4)
    kw = dict(max_length = max_length, text_temperature = 0., cfg_scale = 3.0, modality_steps = steps_ode, init_modality_noise = noise, force_modality_at_start = (0, (Lm,)),
              return_unprocessed_modalities = True)
    eng = model.engine
    for _ in range(max(1, args.warmup)):
        out = model.sample_many(copy.deepcopy(prompts), **kw)
    torch.cuda.synchronize()
    sampler.start()
    times_ms, l0 = [], eng.ops.launches
    for _ in range(args.steps):
        e0, e1 = torch.cuda.Event(enable_timing = True), torch.cuda.Event(enable_timing = True)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        e0.record()
        out = model.sample_many(copy.deepcopy(prompts), **kw)          # host prompts in, host samples out: H2D / D2H inside the timed region
        e1.record(); torch.cuda.synchronize()
        times_ms.append((1e3 * (time.perf_counter() - t0), e0.elapsed_time(e1)))
    sampler.stop()
    if args.dump_outputs:
        # the samples of the last timed call, part by part (text ids, modality latents).  Whole samples only, and as many as fit in DUMP_LIMIT
        # by a per-sample bound that depends on the arguments alone (prompt modality < 65 rows, the forced modality, max_length float64 text ids),
        # so that two builds always write the same samples
        keep = min(len(out), DUMP_LIMIT // (4 * (64 + Lm) * 384 + 8 * max_length))
        if keep < len(out):
            log(f'--dump-outputs: the first {keep} of {len(out)} samples')
        write_outputs(args.dump_outputs, [(f'sample{i:03d}_part{j:02d}_text', p.cpu().numpy()) if torch.is_tensor(p) else
                                          (f'sample{i:03d}_part{j:02d}_modality{p[0]}', p[1].float().cpu().numpy())
                                          for i, s_ in enumerate(out[:keep]) for j, p in enumerate(s_)])
    launches = (eng.ops.launches - l0) // args.steps
    # one more (untimed) call with CUDA events around every text loop / modality round: where the wall time goes
    model._sampling_timer = {}
    model.sample_many(copy.deepcopy(prompts), **kw)
    torch.cuda.synchronize()
    phases = {k: dict(calls = len(v), ms = round(sum(a.elapsed_time(b) for a, b in v), 2)) for k, v in model._sampling_timer.items()}
    # (host hiccups stretch single calls by 2x now and then: the phase pass is repeated and the faster one kept)
    model._sampling_timer = {}
    model.sample_many(copy.deepcopy(prompts), **kw)
    torch.cuda.synchronize()
    again = {k: dict(calls = len(v), ms = round(sum(a.elapsed_time(b) for a, b in v), 2)) for k, v in model._sampling_timer.items()}
    if sum(v['ms'] for v in again.values()) < sum(v['ms'] for v in phases.values()): phases = again
    model._sampling_timer = None
    text_ms = phases.get('text_loop', {}).get('ms')
    wall_ms = sorted(t[0] for t in times_ms)[len(times_ms) // 2]
    # generated tokens: the 256 modality positions + every sampled text token of every sample
    prep = [model.prepare_prompt_sample(copy.deepcopy(p), kw['force_modality_at_start'])[0] for p in prompts]
    plen = [model._parts_len(p) for p in prep]
    total_len = [model._parts_len(s_) for s_ in out]
    gen = [t - p for t, p in zip(total_len, plen)]
    text_tokens = [g - Lm - 1 for g in gen]                             # minus the modality and the [eom] the sampler appends itself
    n_gen = sum(gen)
    # transformer FLOPs per generated token: kv-cache path vs re-running the packed prefix at every text step / ODE evaluation (round 1)
    FWD = 65.1e6 / 1.0                                                  # forward MFLOP per token (SURVEY.md 8(d)), linear layers dominate
    evals = 2 * (steps_ode - 1)
    cached = sum(p for p in plen) + n_prompts * (evals * 2 * Lm) + sum(text_tokens) + sum(p + 0 for p in plen)      # prefill + (cond+uncond) ODE tokens + text steps + uncond prefill
    recompute = n_prompts * evals * 2 * (sum(plen) / n_prompts + Lm) + sum(sum(range(p + Lm + 1, p + Lm + 1 + t)) for p, t in zip(plen, text_tokens))
    # KV bytes the text loop reads: every step reads the whole slab prefix of every sample, K and V, all layers
    kv_bytes = sum(sum(range(p + Lm + 1, p + Lm + 1 + t)) for p, t in zip(plen, text_tokens)) * eng.HI * 2 * 2 * eng.depth
    pk = peaks()
    cpu = None
    if not args.no_cpu_baseline:
        cpu = cpu_sample_many(args, prompts, noise)
    line = dict(metric = 'sample_many generated tokens/sec (text + latent positions), config 5', value = n_gen / (wall_ms / 1e3), unit = 'tokens/s', n_gpus = 1, steps = args.steps, warmup = args.warmup,
                ms_per_step = wall_ms, higher_is_better = True, scaling = 'weak', vs_baseline = None, dtype = 'bf16', data = 'synthetic',
                config = dict(workload = WORKLOADS['sample_many'], prompts = n_prompts, max_length = max_length, modality = [Lm, 384], modality_steps = steps_ode, cfg_scale = 3.0,
                              text = 'greedy', launch = 'captured text-step graph + captured ODE-evaluation graph'),
                e2e = dict(value = n_gen / (wall_ms / 1e3), unit = 'tokens/s', wall_ms = wall_ms, device_ms = sorted(t[1] for t in times_ms)[len(times_ms) // 2],
                           h2d_bytes_per_step = int(sum(p[1].numel() * 4 for pr in prompts for p in ([pr] if isinstance(pr, tuple) else (pr if isinstance(pr, list) else [])) if isinstance(p, tuple)) + noise.numel() * 4),
                           d2h_bytes_per_step = int(n_prompts * Lm * 384 * 4 + 4 * sum(text_tokens))),
                phases_ms = phases, gpu_launches = int(launches), generated = dict(total = n_gen, text = int(sum(text_tokens)), latent_positions = n_prompts * Lm),
                transformer_token_forwards = dict(kv_cache = int(cached), prefix_recompute = int(recompute), saving = round(recompute / cached, 1)),
                roofline = dict(bound = 'hbm', kernel = 'attn_decode (text loop, kv read)', achieved = (kv_bytes / (text_ms / 1e3) / 1e9 if text_ms else None), peak = pk['hbm'], unit = 'GB/s',
                                frac = (kv_bytes / (text_ms / 1e3) / 1e9 / pk['hbm'] if text_ms else None), traffic = None, kv_bytes_text_loop = int(kv_bytes), text_loop_ms = text_ms,
                                note = 'K / V bytes the decode attention reads over the whole text loop / device time of the loop: at 32 rows per step the loop is launch- and latency-bound, not bandwidth-bound'),
                clocks = sampler.summary(), cpu_baseline = cpu)
    emit(line)


def cpu_sample_many(args, prompts, noise):
    """the reference algorithm (oracle port: padded kv caches are replaced by slabs, everything else - per-token conditioning, dense masks - as the
    reference) on the host cores, on a BOUNDED sample: 4 of the prompts, 4 midpoint steps, 24 text tokens"""
    import copy
    import torch
    from transfusion_pytorch_b200 import Transfusion, synth
    from oracle.torch_reference import OracleEngine
    torch.set_num_threads(usable_cores())
    torch.manual_seed(0)
    model = Transfusion(**CTOR).eval()
    synth.fill_parameters_(model, seed = 0)
    model._engine = OracleEngine(model)
    sub = prompts[:4]
    kw = dict(max_length = 256 + 24, text_temperature = 0., cfg_scale = 3.0, modality_steps = 4, init_modality_noise = noise, force_modality_at_start = (0, (256,)),
              return_unprocessed_modalities = True)
    t0 = time.perf_counter()
    out = model.sample_many(copy.deepcopy(sub), **kw)
    dt = time.perf_counter() - t0
    prep = [model.prepare_prompt_sample(copy.deepcopy(p), kw['force_modality_at_start'])[0] for p in sub]
    n_gen = sum(model._parts_len(s_) - model._parts_len(p) for s_, p in zip(out, prep))
    return dict(value = n_gen / dt, unit = 'tokens/s', cores = torch.get_num_threads(), kind = 'port',
                sample = f'4 prompts, forced 256x384 modality with 4 midpoint steps (6 evaluations x cond/uncond), 24 greedy text tokens: {n_gen} generated positions in {dt:.1f} s')


_JSON_OUT = None


def emit(line: dict):
    """the ONE JSON line of the contract goes to the process's ORIGINAL stdout; everything else that libraries print on file descriptor 1 (the NCCL version
    banner is written there whatever NCCL_DEBUG_FILE says) has been routed to stderr by `claim_stdout`"""
    out = _JSON_OUT or sys.stdout
    out.write(json.dumps(line) + '\n')
    out.flush()


def claim_stdout():
    global _JSON_OUT
    if _JSON_OUT is None:
        sys.stdout.flush()
        _JSON_OUT = os.fdopen(os.dup(1), 'w')
        os.dup2(2, 1)


def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type = int, default = 1)
    ap.add_argument('--steps', type = int, default = 10)
    ap.add_argument('--warmup', type = int, default = 3)
    ap.add_argument('--batch', type = int, default = 128, help = 'sequences (x1024 tokens) per GPU per step (swept 32 / 64 / 128 on B200: 2.00 / 2.12 / 2.18 M tokens/s)')
    ap.add_argument('--impl', default = 'b200', choices = ['b200', 'reference'])
    ap.add_argument('--workload', default = 'train', choices = sorted(WORKLOADS), help = 'train = configs[1] (the graded metric); config4 = two-modality span stress; sample_many = configs[4]')
    ap.add_argument('--prompts', type = int, default = 32, help = 'sample_many: number of prompts (multiple of 4)')
    ap.add_argument('--max-length', type = int, default = 512, help = 'sample_many: max_length')
    ap.add_argument('--scaling', default = 'weak', choices = ['weak', 'strong'], help = 'strong: --batch is the global batch (fixed total work as N grows)')
    ap.add_argument('--no-overlap', action = 'store_true', help = 'N > 1: one all-reduce after backward instead of per-layer buckets overlapped with it')
    ap.add_argument('--no-cpu-baseline', action = 'store_true')
    ap.add_argument('--dump-launches', default = None, help = 'write the entry points of the profiled step in launch order (JSON) - input of tools/ncu_traffic.py')
    ap.add_argument('--no-graph', action = 'store_true', help = 'eager kernel launches instead of CUDA-graph replay (N = 1)')
    ap.add_argument('--dump-outputs', default = None, metavar = 'DIR',
                    help = 'after the timed steps write what they computed as DIR/<name>.npy (at most 64 MB; same arguments, same inputs): train / config4 = '
                           'loss of the last step, a fixed sample of the parameters after it and their change over the timed steps; sample_many = the samples of the last call '
                           '(with many prompts only the first ones, as many as --prompts / --max-length allow within 64 MB)')
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error('--steps must be at least 1 and --warmup at least 0')
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs writes the outputs of the B200 arm')
    if args.impl == 'reference':
        run_reference_arm(args)
    elif args.workload == 'sample_many':
        run_sample_many(args)
    else:
        run_b200_arm(args)


if __name__ == '__main__':
    main()

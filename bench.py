#!/usr/bin/env python
"""bench.py -- mel frames/sec of the fused STFT -> |.| -> mel -> dB hot path on B200.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

One step = one pass of the hot path over one batch of synthetic waveforms.  Workload (N=1 and
per rank for N>1, weak scaling): BASELINE.json configs[1] -- batch 256, mono, 22.05 kHz x 5 s,
n_fft=1024, hop=256, 128 mel bands, decibel output, through ``get_melspectrogram_layer``.
Rank 0 prints ONE JSON line (contract in the task statement):
  value      frames/s with inputs resident in HBM (CUDA events, max over ranks)
  e2e        frames/s through the public ``predict`` call with pinned HOST buffers: H2D of the
             waveforms and D2H of the log-mel tensor inside the timed region
  roofline   achieved algorithmic GB/s of the fused kernel (CUDA events around the kernel
             itself, recorded by the library) against the measured HBM copy bandwidth
  cpu_baseline  the oracle's multi-threaded CPU port on the same workload, timed on rank 0
``--impl reference`` times that CPU port alone (the reference itself needs TensorFlow + librosa,
which are not installable here; see DESIGN.md).
``--dump-outputs DIR`` writes what the last timed step returned (rank 0's log-mel tensor) to
DIR/logmel_db.npy, float32.  The inputs are seeded, so two builds run with the same arguments can be
compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

# NCCL's debug / banner output must not end up on stdout (one JSON line goes there)
os.environ.setdefault('NCCL_DEBUG_FILE', '/dev/stderr')

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# BASELINE.json configs[1] (the configuration the metric is quoted on; every rank runs one such batch: weak scaling)
# and configs[4] (batch 8192 x 10 s sharded over the ranks with kapre_b200.sharding.shard_range: 1024 items per
# rank on 8 GPUs).  Default: cfg2 below 8 ranks, cfg5 on 8.
CONFIGS = {
    'cfg2': dict(batch=256, sharded=False, length=110250, channels=1, sample_rate=22050, n_fft=1024, hop=256, n_mels=128,
                 workload='cfg2: batch=256 mono 22.05kHz 5s, n_fft=1024 hop=256 n_mels=128, '
                          'get_melspectrogram_layer(return_decibel=True), channels_last'),
    'cfg5': dict(batch=8192, sharded=True, length=160000, channels=1, sample_rate=16000, n_fft=1024, hop=256, n_mels=128,
                 workload='cfg5: batch=8192 mono 16kHz 10s log-mel, n_fft=1024 hop=256 n_mels=128, sharded over the ranks, '
                          'get_melspectrogram_layer(return_decibel=True), channels_last'),
}
CFG = dict(CONFIGS['cfg2'])
WORKLOAD = CFG['workload']


def select_config(name, rank, world):
    """Set the module-level CFG to this rank's share of the named configuration."""
    global CFG, WORKLOAD
    from kapre_b200.sharding import shard_range
    CFG = dict(CONFIGS[name])
    CFG['name'] = name
    CFG['global_batch'] = CFG['batch'] if CFG['sharded'] else CFG['batch'] * world
    if CFG['sharded']:
        lo, hi = shard_range(CFG['batch'], rank, world)
        CFG['batch'] = hi - lo
        CFG['shard'] = [lo, hi]
    WORKLOAD = CFG['workload']
DUMP_LIMIT = 60_000_000  # bytes of --dump-outputs, under 64 MB with the .npy header; beyond it, a sample of items
PROFILE_EVERY = 8  # every 8th fused-kernel launch of the timed loop is bracketed by CUDA events (roofline.kernel_ms)
N_SETS = 3  # rotating input/output sets: 3 x (113 MB in + 56 MB out) = 507 MB > 126 MB L2


def frames_per_step():
    return CFG['batch'] * CFG['channels'] * (1 + (CFG['length'] - CFG['n_fft']) // CFG['hop'])


def algorithmic_bytes_per_step():
    """SURVEY 8(d): every covered sample read once + every output written once (fp32)."""
    T = 1 + (CFG['length'] - CFG['n_fft']) // CFG['hop']
    covered = (T - 1) * CFG['hop'] + CFG['n_fft']
    return CFG['batch'] * CFG['channels'] * (4 * covered + 4 * T * CFG['n_mels'])


def measured_peaks():
    try:
        with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as f:
            d = json.load(f)
        return float(d['hbm_gbs']), 'MEASURED_PEAKS.json (measured copy bandwidth)'
    except Exception:
        return 6650.0, 'fallback 6.65 TB/s (B200_PROFILING.md)'


class ClockSampler:
    """Samples SM clock / throttle reasons through NVML while a region runs."""

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _once(self):
        nv = self.nv
        try:
            self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
            r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
            names = {'hw_slowdown': getattr(nv, 'nvmlClocksThrottleReasonHwSlowdown', 0x8),
                     'hw_thermal_slowdown': getattr(nv, 'nvmlClocksThrottleReasonHwThermalSlowdown', 0x40),
                     'sw_thermal_slowdown': getattr(nv, 'nvmlClocksThrottleReasonSwThermalSlowdown', 0x20),
                     'sw_power_cap': getattr(nv, 'nvmlClocksThrottleReasonSwPowerCap', 0x4)}
            for k, bit in names.items():
                if r & bit:
                    self.reasons.add(k)
        except Exception:
            pass

    def _run(self):
        while not self._stop.is_set():
            self._once()
            time.sleep(0.01)

    def start(self):
        if self.nv is None:
            return
        self._stop.clear()
        self._thread = threading.Thread(target=self._run, daemon=True)
        self._thread.start()

    def stop(self):
        if self.nv is None:
            return
        self._once()
        self._stop.set()
        if self._thread is not None:
            self._thread.join()

    def summary(self):
        if not self.samples:
            return {'sm_mhz': None, 'sm_max_mhz': self.max_mhz, 'reasons': sorted(self.reasons)}
        s = sorted(self.samples)
        return {'sm_mhz': s[len(s) // 2], 'sm_max_mhz': self.max_mhz, 'reasons': sorted(self.reasons),
                'samples': len(s)}


def dump_outputs(out_dir, y):
    """Write the device tensor `y` (batch first) to out_dir/logmel_db.npy as float32: whole if it fits in
    DUMP_LIMIT, otherwise the batch items np.random.default_rng(0).choice(batch, n, replace=False) picks, in
    increasing order, for the largest n that fits."""
    import numpy as np
    item_bytes = y[0].numel() * 4
    if y.shape[0] * item_bytes > DUMP_LIMIT:
        n = max(1, DUMP_LIMIT // item_bytes)
        items = np.sort(np.random.default_rng(0).choice(y.shape[0], n, replace=False))
        y = y[items.tolist()]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, 'logmel_db.npy'), y.float().cpu().numpy())


def cpu_port(threads=None):
    import torch
    from oracle.fast_cpu import MelSpectrogramCPU
    if threads:
        torch.set_num_threads(threads)
    return MelSpectrogramCPU(n_fft=CFG['n_fft'], hop_length=CFG['hop'], sample_rate=CFG['sample_rate'],
                             n_mels=CFG['n_mels'], return_decibel=True, input_data_format='channels_last',
                             output_data_format='channels_last')


def run_cpu(steps, warmup, budget_s):
    """Times the CPU port: `steps` passes over the cfg2 batch (stops early once budget_s is spent)."""
    import torch
    cores = os.cpu_count() or 1
    model = cpu_port()
    g = torch.Generator().manual_seed(1234)
    x = torch.rand((CFG['batch'], CFG['length'], CFG['channels']), generator=g) * 2 - 1
    # give the CPU arm its best thread count: torch's intra-op pool stops scaling (and can slow
    # down) on very wide hosts, so try a few widths up to all cores for one pass each
    best_n, best_t = cores, None
    for n in sorted({min(cores, c) for c in (8, 16, 32, 64, cores)}):
        torch.set_num_threads(n)
        model(x[:32])
        t0 = time.perf_counter()
        model(x)
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best_n, best_t = n, dt
    torch.set_num_threads(best_n)
    for _ in range(max(1, warmup)):
        model(x)
    done, t0 = 0, time.perf_counter()
    while done < steps:
        model(x)
        done += 1
        if time.perf_counter() - t0 > budget_s:
            break
    dt = time.perf_counter() - t0
    return dict(value=frames_per_step() * done / dt, unit='frames/s', cores=torch.get_num_threads(), host_cores=cores, kind='port',
                steps_timed=done,
                sample='%d passes over a %d-item batch of %s (%d frames each), torch-CPU fp32 op-by-op port of the '
                       'reference graph, best of {8,16,32,64,all=%d} threads, %.1f s' % (done, CFG['batch'], CFG.get('name', 'cfg2'), frames_per_step(), cores, dt)), dt / done


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=200)
    ap.add_argument('--warmup', type=int, default=10)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--config', default='auto', choices=['auto', 'cfg2', 'cfg5'],
                    help='auto: cfg2 per rank below 8 ranks (weak scaling), cfg5 (batch 8192 sharded) on 8 ranks')
    ap.add_argument('--no-numa-bind', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write the output of the last timed step to DIR/logmel_db.npy (float32)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'b200':
        ap.error('--dump-outputs writes the CUDA path\'s outputs (--impl b200)')
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    warmup = max(3, args.warmup)

    if args.impl == 'reference':
        if rank != 0:
            return 0
        select_config(('cfg5' if world >= 8 else 'cfg2') if args.config == 'auto' else args.config, 0, max(world, 1))
        if CFG['batch'] > 512:                            # bounded sample of this arm's workload: a 512-item slice per pass
            CFG['batch'] = 512
        base, s_per_step = run_cpu(args.steps, warmup, budget_s=150.0)
        line = {'impl': 'reference', 'metric': 'mel_frames_per_sec', 'value': base['value'], 'unit': 'frames/s',
                'n_gpus': args.gpus, 'steps': base['steps_timed'], 'warmup': warmup, 'ms_per_step': s_per_step * 1e3,
                'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32',
                'data': 'synthetic U(-1,1) waveforms', 'config': {'workload': WORKLOAD, 'name': CFG['name'], 'device': 'host CPU', 'items_per_pass': CFG['batch']},
                'cpu_baseline': base,
                'e2e': {'value': base['value'], 'unit': 'frames/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
                'gpu_launches': 0,
                'note': 'reference arm = the oracle CPU port (TensorFlow/librosa are not installed in this sandbox)'}
        print(json.dumps(line))
        return 0

    import torch
    import torch.distributed as dist

    import kapre_b200 as K
    from kapre_b200 import _native

    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    select_config(('cfg5' if world >= 8 else 'cfg2') if args.config == 'auto' else args.config, rank, world)
    # host side of the end-to-end path: this rank's CPU threads and page-locked pools on the GPU's NUMA node
    from kapre_b200 import hostmem
    numa = {'node': None} if args.no_numa_bind else hostmem.bind_to_gpu_node(local_rank)
    if world > 1:
        # stdout carries exactly one JSON line: NCCL prints its version banner (and any NCCL_DEBUG output) with
        # C stdio to fd 1, so fd 1 points at stderr while the communicator is created
        sys.stdout.flush()
        saved_fd = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group('nccl', device_id=dev)
            dist.barrier()                      # creates the communicator (lazy in torch)
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_fd, 1)
            os.close(saved_fd)
    _native.lib()
    layer = K.get_melspectrogram_layer(n_fft=CFG['n_fft'], hop_length=CFG['hop'], sample_rate=CFG['sample_rate'],
                                       n_mels=CFG['n_mels'], return_decibel=True, input_data_format='channels_last',
                                       output_data_format='channels_last')
    shape = (CFG['batch'], CFG['length'], CFG['channels'])
    xs = []
    for i in range(N_SETS):
        g = torch.Generator(device=dev).manual_seed(1234 + rank * N_SETS + i)
        xs.append(torch.rand(shape, generator=g, device=dev) * 2 - 1)
    frames = frames_per_step()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    from kapre_b200.sharding import reduce_max as _reduce_max

    def reduce_max(v):
        return _reduce_max(v, device=dev)

    def reduce_sum(v):
        if world > 1:
            t = torch.tensor([float(v)], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
            return float(t.item())
        return float(v)

    # ---------------- end to end through predict() with pinned host buffers ---------------------
    def run_e2e():
        xh = [torch.empty(shape, dtype=torch.float32, pin_memory=True) for _ in range(2)]
        for i, t in enumerate(xh):
            t.copy_(xs[i])
        torch.cuda.synchronize()
        n = max(3, min(args.steps, 20))
        y = None
        for i in range(max(3, args.warmup)):     # same pattern as the timed loop (the previous result is still
            y = layer.predict(xh[i % 2])         # alive when the next call starts), so the result pool is warm
        barrier()
        per_step = []
        t0 = time.perf_counter()
        for i in range(n):
            t1 = time.perf_counter()
            y = layer.predict(xh[i % 2])
            per_step.append(round((time.perf_counter() - t1) * 1e3, 3))
        torch.cuda.synchronize()
        secs = reduce_max(time.perf_counter() - t0)
        if os.environ.get('KAPRE_BENCH_DEBUG'):
            print('[e2e per-step ms]', per_step, file=sys.stderr)
        return xh, y, n, secs

    e2e_first = bool(os.environ.get('KAPRE_BENCH_E2E_FIRST'))
    if e2e_first:
        xh, y_host, e2e_steps, e2e_s = run_e2e()

    # ---------------- device-resident throughput ------------------------------------------------
    outs = [None] * N_SETS
    for i in range(warmup):
        outs[i % N_SETS] = layer(xs[i % N_SETS])
    _native.profile_read()
    sampler = ClockSampler(local_rank)
    barrier()
    n0 = _native.launch_count()
    _native.profile_enable(True, every=PROFILE_EVERY)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler.start()
    t_host0 = time.perf_counter()
    e0.record()
    for i in range(args.steps):
        outs[i % N_SETS] = layer(xs[i % N_SETS])
    e1.record()
    host_submit_ms = (time.perf_counter() - t_host0) * 1e3 / args.steps
    barrier()
    sampler.stop()
    _native.profile_enable(False)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, outs[(args.steps - 1) % N_SETS])
    ms_total = reduce_max(e0.elapsed_time(e1))
    launches = _native.launch_count() - n0
    kern_ms, kern_n = _native.profile_read()
    ms_per_step = ms_total / args.steps
    frames_all = reduce_sum(frames)                       # all ranks' frames per step (shards may differ by one item)
    value = frames_all * args.steps / (ms_total * 1e-3)

    if not e2e_first:
        xh, y_host, e2e_steps, e2e_s = run_e2e()
    e2e_value = frames_all * e2e_steps / e2e_s
    h2d = xh[0].numel() * 4
    d2h = int(y_host.size) * 4
    # PCIe ceiling of that call: the same two buffers copied concurrently on two streams, nothing else
    yd_probe = torch.empty(y_host.shape, dtype=torch.float32, device=dev)
    yh_probe = torch.empty(y_host.shape, dtype=torch.float32, pin_memory=True)
    s_a, s_b = torch.cuda.Stream(), torch.cuda.Stream()

    def _copies():
        with torch.cuda.stream(s_a):
            xs[0].copy_(xh[0], non_blocking=True)
        with torch.cuda.stream(s_b):
            yh_probe.copy_(yd_probe, non_blocking=True)
    _copies()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(5):
        _copies()
    torch.cuda.synchronize()
    pcie_s = (time.perf_counter() - t0) / 5
    pcie_bound = frames_all / pcie_s

    # ---------------- the same call on PAGEABLE memory (what a kapre user passes: a plain NumPy array) ----------
    pageable = None
    try:
        xn = xh[0].numpy().copy()                       # ordinary malloc'ed array, not page-locked
        layer.predict(xn)
        barrier()
        t0 = time.perf_counter()
        n_pg = 3
        for _ in range(n_pg):
            layer.predict(xn)
        torch.cuda.synchronize()
        pageable = frames_all * n_pg / reduce_max(time.perf_counter() - t0)
        del xn
    except Exception as e:  # noqa: BLE001  (a reported extra, never fatal for the bench line)
        print('[bench] pageable predict failed: %r' % (e,), file=sys.stderr)

    # ---------------- parity spot check of what was timed ---------------------------------------
    import oracle
    import numpy as np
    ref = oracle.melspectrogram_layer(xs[0][:2].cpu().numpy(), n_fft=CFG['n_fft'], hop_length=CFG['hop'],
                                      sample_rate=CFG['sample_rate'], n_mels=CFG['n_mels'], return_decibel=True)
    max_err_db = float(np.abs(outs[0][:2].cpu().numpy() - ref).max()) if outs[0] is not None else None

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    peak, peak_src = measured_peaks()
    kernel_ms = kern_ms / max(kern_n, 1)
    achieved = algorithmic_bytes_per_step() / (kernel_ms * 1e-3) / 1e9 if kern_n else None
    roofline = {'bound': 'hbm', 'achieved': achieved, 'peak': peak, 'unit': 'GB/s',
                'frac': (achieved / peak) if achieved else None, 'traffic': None, 'peak_source': peak_src,
                'kernel': 'kb_stft_kernel<16, FB_DB> (fused frame+window+FFT+|.|+mel+dB)',
                'kernel_ms': kernel_ms, 'kernel_launches_timed': kern_n,
                'algorithmic_bytes_per_launch': algorithmic_bytes_per_step(),
                'read_only_frac': (CFG['batch'] * 4.0 * ((1 + (CFG['length'] - CFG['n_fft']) // CFG['hop'] - 1) * CFG['hop'] + CFG['n_fft'])
                                   / (kernel_ms * 1e-3) / 1e9 / peak) if kern_n else None}
    traffic_file = os.path.join(ROOT, 'profiles', 'traffic_bytes_per_launch.json')
    if os.path.exists(traffic_file):
        try:
            roofline['traffic'] = json.load(open(traffic_file)).get(CFG['name'] + '_fb_db')
        except Exception:
            pass
    cpu = None
    if not args.no_cpu_baseline and world == 1:      # the CPU baseline is an N=1 measurement (rank 0 has the box to itself)
        hostmem.restore_affinity(numa)                # the CPU arm gets every host core
        cpu, _ = run_cpu(steps=40, warmup=1, budget_s=12.0)
    line = {
        'metric': 'mel_frames_per_sec', 'value': value, 'unit': 'frames/s', 'n_gpus': world, 'steps': args.steps,
        'warmup': warmup, 'ms_per_step': ms_per_step, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic U(-1,1) waveforms, generated on device (seeded)',
        'config': {'workload': WORKLOAD, 'name': CFG['name'], 'frames_per_step_per_gpu': frames,
                   'global_batch': CFG['global_batch'], 'items_per_gpu': CFG['batch'],
                   'parallelism': 'dp%d (batch sharded with kapre_b200.sharding.shard_range, no collective in the data path)' % world,
                   'numa': {'gpu_node': numa.get('node'), 'cpus_bound': numa.get('cpus')},
                   'l2': '%d rotating input/output sets (%.0f MB) > 126 MB L2' % (
                       N_SETS, N_SETS * algorithmic_bytes_per_step() / 1e6),
                   'launch': _native.last_launch_info(), 'host_submit_ms_per_step': host_submit_ms},
        'roofline': roofline,
        'cpu_baseline': cpu,
        'e2e': {'value': e2e_value, 'unit': 'frames/s', 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h,
                'steps': e2e_steps, 'api': 'Sequential.predict(pinned host tensor) -> host array',
                'pcie_bound': pcie_bound, 'frac_of_pcie_bound': e2e_value / pcie_bound,
                'pageable_numpy_input': pageable},
        'gpu_launches': launches,
        'clocks': sampler.summary(),
        'max_abs_err_db_vs_oracle': max_err_db,
    }
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == '__main__':
    sys.exit(main())

#!/usr/bin/env python
"""bench.py -- CSPN propagation throughput on B200 (contract: see the task brief / DESIGN.md section 6).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--algo auto|generic|cluster]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one pass of the hot path (24-iteration 2D CSPN, '8sum', with sparse depth) over one batch of
synthetic inputs of BASELINE.json configs[1]: 32 x 1216x352 (W x H) per GPU, fp32.  Weak scaling: every
rank owns its own 32 images (N=8 is configs[4], 256 images); no data-path collective.
Prints ONE JSON line on rank 0.  --dump-outputs DIR also writes what the last timed step returned on rank 0, the
propagated depth of its 32 images, as DIR/out.npy (float32, 54.8 MB); the inputs are seeded, so two builds can be
compared output for output.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

H, W, B_PER_GPU, ITERS, NORM = 352, 1216, 32, 24, '8sum'
ALGO_BYTES_PER_PX = 44          # SURVEY.md 8(d): read 8 guidance + blur + sparse, write out, fp32
METRIC = 'CSPN Mpixels/s (24-iter 2D, 1216x352)'


def workload_config(world):
    """The SAME dict in both arms (ours and --impl reference): the driver compares them."""
    return {'workload': f'2D CSPN 3x3, {ITERS} iters, {NORM}, with sparse depth (Bernoulli 500 samples/image), batch '
                        f'{B_PER_GPU}x{W}x{H} fp32 per GPU (BASELINE configs[1]; N=8 is configs[4])',
            'global_batch': world * B_PER_GPU,
            'parallelism': f'dp{world} (independent images per rank, no data-path collective)'}


def measured_hbm_peak():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    try:
        with open(p) as fh:
            return float(json.load(fh)['hbm_gbs']), 'measured (MEASURED_PEAKS.json, burst copy)'
    except Exception:
        return 6650.0, 'fallback (B200_PROFILING.md)'


def recorded_traffic(algo_name):
    """dram bytes per launch of the dominant kernel from the committed ncu --set full capture, or None."""
    try:
        with open(os.path.join(ROOT, 'profiles', 'traffic.json')) as fh:
            t = json.load(fh)
        return t.get(algo_name, {}).get('dram_bytes_per_launch')
    except Exception:
        return None


class ClockSampler:
    """Samples SM clock / throttle reasons of one GPU during the timed region (pynvml, ~2 ms period)."""
    REASONS = {0x1: 'gpu_idle', 0x2: 'applications_clocks_setting', 0x4: 'sw_power_cap', 0x8: 'hw_slowdown',
               0x10: 'sync_boost', 0x20: 'sw_thermal_slowdown', 0x40: 'hw_thermal_slowdown',
               0x80: 'hw_power_brake_slowdown', 0x100: 'display_clock_setting'}

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
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

    def _loop(self):
        while not self._stop.is_set():
            try:
                self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                mask = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for bit, name in self.REASONS.items():
                    if mask & bit and name != 'gpu_idle':
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.002)

    def __enter__(self):
        if self.nv:
            self._thr = threading.Thread(target=self._loop, daemon=True)
            self._thr.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._thr:
            self._thr.join()

    def summary(self):
        s = sorted(self.samples)
        return {'sm_mhz': (s[len(s) // 2] if s else None), 'sm_max_mhz': self.max_mhz,
                'reasons': sorted(self.reasons), 'samples': len(s)}


def physical_gpu_index(local_rank):
    vis = os.environ.get('CUDA_VISIBLE_DEVICES')
    if vis:
        try:
            return int(vis.split(',')[local_rank])
        except Exception:
            return local_rank
    return local_rank


# ---------------------------------------------------------------------------------------------
# CPU legs (the only places bench.py touches oracle/)
# ---------------------------------------------------------------------------------------------

def time_torch_port(nb, steps, warmup, threads):
    """The reference's own op sequence (oracle/cspn_torch_port.py == cspn.py minus `.cuda()`), all host threads."""
    import torch
    from cspn_b200.synth import make_inputs
    from oracle import cspn_torch_port as tp
    torch.set_num_threads(threads)
    g, d, s = make_inputs(0, nb, 1, H, W)
    with torch.no_grad():
        for _ in range(warmup):
            tp.cspn2d_torch(g, d, s, ITERS, NORM)
        t0 = time.perf_counter()
        for _ in range(steps):
            tp.cspn2d_torch(g, d, s, ITERS, NORM)
        dt = time.perf_counter() - t0
    return nb * H * W * steps / dt / 1e6, dt / steps


def median(xs):
    xs = sorted(xs)
    return xs[len(xs) // 2]


def time_torch_port_median(nb, reps, warmup, threads):
    """Median over `reps` single forwards after `warmup` (BASELINE.md section 3: warm-up + median)."""
    import torch
    from cspn_b200.synth import make_inputs
    from oracle import cspn_torch_port as tp
    torch.set_num_threads(threads)
    g, d, s = make_inputs(0, nb, 1, H, W)
    ts = []
    with torch.no_grad():
        for i in range(warmup + reps):
            t0 = time.perf_counter()
            tp.cspn2d_torch(g, d, s, ITERS, NORM)
            if i >= warmup:
                ts.append(time.perf_counter() - t0)
    t = median(ts)
    return nb * H * W / t / 1e6, t


def best_torch_threads():
    """The reference's op sequence is ~700 small ATen ops per forward: oversubscribing a 128-thread host makes it
    20x slower than a few threads.  'All the host threads it can use' = the count that maximises its throughput:
    per candidate one warm-up and the median of 3 single-image forwards."""
    ncpu = os.cpu_count() or 1
    best, best_t = 1, float('inf')
    for n in sorted({min(ncpu, c) for c in (8, 16, 32, 64)}):
        t = time_torch_port_median(1, 3, 1, n)[1]
        if t < best_t:
            best, best_t = n, t
    return best, best_t


def cpu_baseline_leg():
    """Bounded sample (about 20 s): the reference's op sequence at B=4 (BASELINE.md section 3's plan) and at B=1 (the
    reference's own eval batch, eval.py:39), plus the C/OpenMP oracle and the same ops run eagerly on this GPU for context."""
    import torch
    from cspn_b200.synth import make_inputs
    from oracle import c_oracle
    threads, _ = best_torch_threads()
    mpx4, t4 = time_torch_port_median(4, 3, 1, threads)
    mpx1, t1 = time_torch_port_median(1, 5, 2, threads)
    g, d, s = make_inputs(0, 4, 1, H, W)
    gn, dn, sn = g.numpy(), d.numpy(), s.numpy()
    ncpu = os.cpu_count() or 1
    c_mpx, c_thr = 0.0, 1
    for nt in sorted({min(ncpu, c) for c in (16, 32, 64)}):      # the OpenMP port also has a sweet spot
        c_oracle.cspn2d(gn[:1], dn[:1], sn[:1], ITERS, NORM, nthreads=nt)
        t0 = time.perf_counter()
        c_oracle.cspn2d(gn, dn, sn, ITERS, NORM, nthreads=nt)
        r = 4 * H * W / (time.perf_counter() - t0) / 1e6
        if r > c_mpx:
            c_mpx, c_thr = r, nt
    gpu_eager = None
    try:
        from oracle import cspn_torch_port as tp
        if torch.cuda.is_available():
            gg, dd, ss = [t.cuda() for t in (g, d, s)]
            with torch.no_grad():
                tp.cspn2d_torch(gg, dd, ss, ITERS, NORM)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                for _ in range(3):
                    tp.cspn2d_torch(gg, dd, ss, ITERS, NORM)
                torch.cuda.synchronize()
            gpu_eager = round(3 * 4 * H * W / (time.perf_counter() - t0) / 1e6, 1)
    except Exception:
        gpu_eager = None
    return {'value': round(mpx4, 3), 'unit': 'Mpixels/s', 'cores': threads, 'kind': 'port',
            'sample': f'4x{W}x{H} images (B=4: BASELINE.md section 3), {ITERS} iters, {NORM}, with sparse depth: 1 warm-up + median of '
                      f'3 forwards of oracle/cspn_torch_port.py (the reference op sequence of cspn.py:42-83 on CPU; '
                      f'/root/reference is absent on this box); {threads} torch threads = the fastest of 8/16/32/64 on this host '
                      f'(warm-up + median of 3 each)',
            'ms_per_forward': round(t4 * 1e3, 1),
            'b1_value': round(mpx1, 3), 'b1_ms_per_forward': round(t1 * 1e3, 1),
            'b1_note': 'batch 1 is the reference eval batch (eval.py:39); its ~700 small ops run several times faster per pixel '
                       'there than at larger batches',
            'reference_ops_eager_on_this_gpu_mpx_s': gpu_eager,
            'host_cpus': os.cpu_count(),
            'c_openmp_port_mpx_s': round(c_mpx, 3), 'c_openmp_threads': c_thr}


def run_reference_arm(args):
    """--impl reference: the reference's CPU implementation of the path (torch-op port), rank 0 only.  Each step is a
    B=4 sample of the workload (BASELINE.md section 3: Mpx/s is what is compared); K steps after W warm-up steps."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    threads, t1 = best_torch_threads()
    budget = 150.0                                               # seconds for the whole run
    nb = 4
    while nb > 1 and (args.steps + args.warmup) * nb * t1 * 2.0 > budget:   # larger batches run ~2x slower per image than B=1
        nb //= 2
    mpx, per = time_torch_port(nb, args.steps, args.warmup, threads)
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': round(mpx, 3), 'unit': 'Mpixels/s', 'n_gpus': args.gpus,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': round(per * 1e3, 3), 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': workload_config(args.gpus),
        'cpu_baseline': {'value': round(mpx, 3), 'unit': 'Mpixels/s', 'cores': threads, 'kind': 'port',
                         'sample': f'each step = {nb}x{W}x{H} images of the workload (same shape, iters, norm and sparse depth) through '
                                   f'oracle/cspn_torch_port.py (reference op sequence, cspn.py:42-83) with {threads} torch threads '
                                   f'(fastest of 8/16/32/64, warm-up + median of 3 each)', 'host_cpus': os.cpu_count()},
        'e2e': {'value': round(mpx, 3), 'unit': 'Mpixels/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    emit(line)


# ---------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------

_REAL_STDOUT = None


def quiet_stdout():
    """stdout carries exactly one JSON line: anything libraries print there (NCCL's version banner comes from C code)
    is diverted to stderr for the duration of the run."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    sys.stdout.flush()
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, (json.dumps(line) + '\n').encode())


def event_times(fn, reps, warmup, pre=None):
    """CUDA-event duration (ms) of each of `reps` calls of fn() after `warmup` calls; `pre(i)` runs untimed before call i."""
    import torch
    for i in range(warmup):
        if pre:
            pre(i)
        fn()
    evs = []
    for i in range(reps):
        if pre:
            pre(i)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        evs.append((a, b))
    torch.cuda.synchronize()
    return sorted(a.elapsed_time(b) for a, b in evs)


def other_configs(dev, peak, sm_max_mhz):
    """The BASELINE.json configs the headline value is not quoted on: configs[2] (NYU-shape iteration sweep), the 304x228
    single image of configs[0] (latency) and configs[3] (3D), each timed with CUDA events on this GPU."""
    import torch
    import cspn_b200
    from cspn_b200 import _lib
    from cspn_b200.synth import make_inputs, make_inputs_3d
    L = _lib.lib()
    out = {}
    fma_peak = 148 * 128 * (sm_max_mhz or 1965) * 1e6          # FMA/s at the maximum SM clock
    # ---- configs[2]: 64 x 304x228, N in {4,8,16,24,48}; two input sets alternate (2 x 195 MB > 126 MB L2) ----------------
    Bn, Hn, Wn = 64, 228, 304
    sets = [[t.to(dev) for t in make_inputs(sd, Bn, 1, Hn, Wn)] for sd in (1, 2)]
    px = Bn * Hn * Wn
    sweep = {}
    from cspn_b200 import torch_op
    torch_op.load()
    for n in (4, 8, 16, 24, 48):
        # these calls last 60-350 us: eager launches would be paced by the host (the queue runs dry between calls), so
        # 10 calls alternating the two input sets are captured into one CUDA graph and the replay is timed
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for g, d, s in sets:
                torch.ops.cspn_b200.propagate2d(g, d, s, n, 0, 0)
        torch.cuda.current_stream().wait_stream(side)
        launches, algo_name = L.cspn_last_launches(), _lib.ALGO_NAMES[L.cspn_last_algo()]
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            for i in range(10):
                g, d, s = sets[i & 1]
                torch.ops.cspn_b200.propagate2d(g, d, s, n, 0, 0)
        ms = event_times(graph.replay, 7, 2)
        t = ms[len(ms) // 2] * 1e-3 / 10
        rate = px / t
        sweep[str(n)] = {'us': round(t * 1e6, 1), 'mpx_s': round(rate / 1e6, 1),
                         'hbm_gbs': round(ALGO_BYTES_PER_PX * rate / 1e9, 1), 'hbm_frac': round(ALGO_BYTES_PER_PX * rate / 1e9 / peak, 4),
                         'fp32_ceiling_mpx_s': round(fma_peak / (8 * n + 30) / 1e6, 1),
                         'fp32_frac': round(rate / (fma_peak / (8 * n + 30)), 4),
                         'launches': launches, 'algo': algo_name}
        del graph
    out['cfg3_nyu_sweep'] = {'workload': f'2D CSPN 3x3, {NORM}, with sparse depth, batch {Bn}x{Wn}x{Hn} (BASELINE configs[2])',
                             'timing': 'one CUDA graph of 10 calls alternating two input sets (2 x 195 MB > 126 MB L2), median of 7 '
                                       'CUDA-event timed replays after 2 warm-up, per call',
                             'fp32_ceiling': f'148 SM x 128 FMA/clk x {sm_max_mhz} MHz / (8 N + 30) FMA per pixel (BASELINE.md section 2)',
                             'by_iters': sweep}
    del sets
    # ---- configs[0]'s shape on the GPU: one 304x228 image, latency of the call ------------------------------------------
    g, d, s = [t.to(dev) for t in make_inputs(0, 1, 1, Hn, Wn)]
    ms = event_times(lambda: cspn_b200.propagate2d(g, d, s, ITERS, NORM), 50, 5)
    lat = {'workload': f'2D CSPN 3x3, {ITERS} iters, 1x{Wn}x{Hn} (the shape of BASELINE configs[0])', 'us_median': round(ms[25] * 1e3, 1),
           'us_min': round(ms[0] * 1e3, 1), 'mpx_s': round(Hn * Wn / (ms[25] * 1e-3) / 1e6, 1), 'note': 'L2-resident (3 MB): a latency figure'}
    try:
        from cspn_b200 import torch_op
        torch_op.load()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            torch.ops.cspn_b200.propagate2d(g, d, s, ITERS, 0, 0)
        torch.cuda.current_stream().wait_stream(side)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            torch.ops.cspn_b200.propagate2d(g, d, s, ITERS, 0, 0)
        ms = event_times(graph.replay, 50, 5)
        lat['us_cuda_graph_replay'] = round(ms[25] * 1e3, 1)
    except Exception as e:          # the torch-op shim is optional
        lat['us_cuda_graph_replay'] = None
        lat['graph_note'] = str(e)[:120]
    out['cfg1_shape_latency'] = lat
    # ---- configs[3]: 3D, 8 x 64x96x312, 12 iters (parity unpinned: the Paddle op's source is not in the reference) --------
    B3, D3, H3, W3, N3 = 8, 64, 96, 312, 12
    g3, f3 = [t.to(dev) for t in make_inputs_3d(0, B3, 1, D3, H3, W3)]
    vox = B3 * D3 * H3 * W3
    r3 = {}
    for mode in ('26sum_abs', 'paddle'):
        ms = event_times(lambda: cspn_b200.propagate3d(g3, f3, N3, mode), 5, 2)
        t = ms[len(ms) // 2] * 1e-3
        r3[mode] = {'ms': round(t * 1e3, 3), 'mvox_s': round(vox / t / 1e6, 1), 'hbm_gbs': round(112 * vox / t / 1e9, 1),
                    'hbm_frac': round(112 * vox / t / 1e9 / peak, 4), 'launches': L.cspn_last_launches()}
    tr = recorded_traffic('step3d')
    out['cfg4_3d'] = {'workload': f'3D CSPN 3x3x3, {N3} iters, volume {B3}x{D3}x{H3}x{W3} [B,D,H,W], 26-channel guidance (BASELINE configs[3])',
                      'unit': 'Mvoxels/s; algorithmic 112 B/voxel (26 guidance + 1 read + 1 write, fp32)', 'parity': 'unpinned (3D arithmetic '
                      'is not in the reference tree; checked against the repo\'s own restatement)', 'by_norm': r3,
                      'traffic_per_step_launch_per_volume': tr,
                      'timing': 'median of 5 CUDA-event timed calls after 2 warm-up; inputs 1.7 GB > L2'}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--algo', default='auto', choices=['auto', 'generic', 'cluster'])
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-other-configs', action='store_true')
    ap.add_argument('--e2e-steps', type=int, default=5)
    ap.add_argument('--dump-outputs', metavar='DIR', help='write the output of the last timed step as DIR/out.npy')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'ours':
        ap.error('--dump-outputs writes the outputs of --impl ours')
    args.warmup = max(args.warmup, 3)
    quiet_stdout()

    if args.impl == 'reference':
        run_reference_arm(args)
        return

    import torch
    import torch.distributed as dist

    import cspn_b200
    from cspn_b200 import _lib
    from cspn_b200.sharding import bind_to_gpu_numa
    from cspn_b200.synth import make_inputs

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit('launch with torch.distributed.run --nproc-per-node N for --gpus N')
    if not torch.cuda.is_available():
        raise SystemExit('bench.py needs a CUDA device (no CPU fallback exists)')
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    numa = bind_to_gpu_numa(local_rank) if world > 1 else None      # before any pinned allocation (first touch)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        # keep stdout to the single JSON line: NCCL's version banner / debug log goes to stderr
        os.environ.setdefault('NCCL_DEBUG_FILE', '/dev/stderr')
        dist.init_process_group('nccl', device_id=dev)

    algo = {'auto': _lib.ALGO_AUTO, 'generic': _lib.ALGO_GENERIC, 'cluster': _lib.ALGO_CLUSTER}[args.algo]
    L = _lib.lib()

    # per-rank shard: its own 32 images (in the real pipeline the UNet produces them on this GPU)
    g_h, d_h, s_h = make_inputs(rank, B_PER_GPU, 1, H, W)
    g, d, s = g_h.to(dev), d_h.to(dev), s_h.to(dev)
    px = B_PER_GPU * H * W

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step():
        return cspn_b200.propagate2d(g, d, s, ITERS, NORM, algo)

    for _ in range(args.warmup):
        out = step()
    launches_per_step = L.cspn_last_launches()
    algo_used = _lib.ALGO_NAMES[L.cspn_last_algo()]
    plan = cspn_b200.describe_plan(B_PER_GPU, 1, H, W, ITERS, algo)

    # ---- timed region: K steps, inputs resident in HBM (602.7 MB per step > 126 MB L2) -------------
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(physical_gpu_index(local_rank)) as clocks:
        barrier()
        ev0.record()
        for _ in range(args.steps):
            out = step()
        ev1.record()
        barrier()
    last_out = out.cpu() if args.dump_outputs and rank == 0 else None
    ms = torch.tensor([ev0.elapsed_time(ev1)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_total = float(ms.item())
    ms_per_step = ms_total / args.steps
    value = world * px / (ms_per_step * 1e-3) / 1e6

    # ---- dominant-kernel roofline: events around each launch sequence of one step, averaged --------
    kern_ms = event_times(step, args.steps, 0)
    kern_ms_avg = sum(kern_ms) / len(kern_ms)
    peak, peak_src = measured_hbm_peak()
    achieved = ALGO_BYTES_PER_PX * px / (kern_ms_avg * 1e-3) / 1e9
    roofline = {'bound': 'hbm', 'achieved': round(achieved, 1), 'peak': peak, 'unit': 'GB/s',
                'frac': round(achieved / peak, 4), 'traffic': recorded_traffic(algo_used),
                'peak_source': peak_src, 'kernel': f'{algo_used} ({launches_per_step} launch(es) per step)',
                'algorithmic_bytes_per_launch_sequence': ALGO_BYTES_PER_PX * px,
                'launch_ms_avg': round(kern_ms_avg, 4), 'launch_ms_min': round(kern_ms[0], 4)}

    # ---- e2e: the reference-facing call with HOST buffers (pinned), H2D + kernels + D2H inside ------
    gp, dp, sp = g_h.pin_memory(), d_h.pin_memory(), s_h.pin_memory()
    out_h = torch.empty_like(dp).pin_memory()                                  # the serving loop's result buffer
    for _ in range(2):                                                         # warm-up (allocates pipeline slots)
        cspn_b200.propagate2d(gp, dp, sp, ITERS, NORM, algo, out=out_h)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.e2e_steps):
        cspn_b200.propagate2d(gp, dp, sp, ITERS, NORM, algo, out=out_h)         # H2D + kernels + D2H, blocking
    barrier()
    e2e_s = torch.tensor([(time.perf_counter() - t0) / args.e2e_steps], device=dev)
    if world > 1:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    e2e_launches = L.cspn_last_launches()
    e2e = {'value': round(world * px / float(e2e_s.item()) / 1e6, 1), 'unit': 'Mpixels/s',
           'h2d_bytes_per_step': world * 10 * px * 4, 'd2h_bytes_per_step': world * px * 4,
           'ms_per_step': round(float(e2e_s.item()) * 1e3, 3), 'launches_per_step': e2e_launches,
           'api': 'cspn_b200.propagate2d(cpu pinned tensors) -> C ABI cspn2d_fwd_f32_host', 'host_numa_binding': numa}
    same = bool(torch.equal(out_h, out.cpu()))

    # ---- the north_star's "NCCL only for the final gather" (eval.py:117), outside the timed value: three ways --------
    gather = None
    if world > 1:
        from cspn_b200.gather import ChunkedGather, FusedGather

        def timed(fn, reps=5, warm=3):
            for _ in range(warm):
                fn()
            barrier()
            ev0.record()
            for _ in range(reps):
                fn()
            ev1.record()
            barrier()
            t = torch.tensor([ev0.elapsed_time(ev1) / reps], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())

        full = torch.empty(world * B_PER_GPU, 1, H, W, device=dev)
        serial_ms = timed(lambda: dist.all_gather_into_tensor(full, step()))
        gather = {'bytes_received_per_rank': (world - 1) * px * 4,
                  'serial_nccl': {'ms_per_step': round(serial_ms, 4), 'what': 'kernel, then all_gather_into_tensor'}}
        ref_full = full.clone()
        try:
            cg = ChunkedGather(B_PER_GPU, 1, H, W, dev, n_chunks=4)
            chunk_ms = timed(lambda: cg.propagate(g, d, s, ITERS, NORM, algo))
            gather['chunked_nccl'] = {'ms_per_step': round(chunk_ms, 4), 'matches_serial': bool(torch.equal(cg.as_rank_major(), ref_full)),
                                      'what': '4 chunks of 8 images: kernel of chunk i+1 overlaps the all-gather of chunk i'}
        except Exception as e:
            gather['chunked_nccl'] = {'error': str(e)[:200]}
        try:
            fg = FusedGather(B_PER_GPU, 1, H, W, dev)
            fused_ms = timed(lambda: fg.propagate(g, d, s, ITERS, NORM))
            res = fg.propagate(g, d, s, ITERS, NORM)
            torch.cuda.synchronize()
            gather['fused_epilogue'] = {'ms_per_step': round(fused_ms, 4), 'mode': fg.mode, 'matches_serial': bool(torch.equal(res, ref_full)),
                                        'what': 'cspn2d_fwd_gather_f32: the kernel epilogue stores each tile into every GPU\'s gather buffer '
                                                '(symmetric memory over NVLink), one barrier across ranks after it'}
        except Exception as e:
            gather['fused_epilogue'] = {'error': str(e)[:300]}
        best = min((v['ms_per_step'], k) for k, v in gather.items() if isinstance(v, dict) and 'ms_per_step' in v)
        gather['ms_per_step_with_all_gather'] = best[0]
        gather['best'] = best[1]
        gather['mpx_s_with_all_gather'] = round(world * px / (best[0] * 1e-3) / 1e6, 1)
        gather['limiter'] = (f'each GPU receives {(world - 1) * px * 4 / 1e6:.0f} MB per step over NVLink: '
                             f'>= {(world - 1) * px * 4 / 900e9 * 1e3:.3f} ms at 900 GB/s per direction')

    cpu_baseline = None
    configs = None
    if rank == 0 and world == 1:
        if not args.no_other_configs:
            configs = other_configs(dev, peak, clocks.max_mhz)
        if not args.no_cpu_baseline:
            cpu_baseline = cpu_baseline_leg()

    if rank == 0:
        cfg = workload_config(world)
        line = {
            'metric': METRIC, 'value': round(value, 1), 'unit': 'Mpixels/s', 'n_gpus': world, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': round(ms_per_step, 4), 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': cfg,
            'detail': {'l2': 'inputs per step (602.7 MB/GPU) exceed the 126 MB L2; no flush needed', 'algo': algo_used, 'plan': plan},
            'roofline': roofline, 'cpu_baseline': cpu_baseline, 'e2e': e2e,
            'gpu_launches': world * args.steps * launches_per_step,
            'clocks': clocks.summary(), 'e2e_matches_device_path': same,
        }
        if configs:
            line['configs'] = configs
        if gather:
            line['gather'] = gather
        if last_out is not None:
            import numpy as np
            os.makedirs(args.dump_outputs, exist_ok=True)
            np.save(os.path.join(args.dump_outputs, 'out.npy'), last_out.numpy().astype(np.float32, copy=False))
        emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()

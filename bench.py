#!/usr/bin/env python
"""bench.py -- BASELINE.json metric: 2048x2048 pupil -> PSF propagations/sec.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--calls-per-step C] [--no-extras]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Headline workload (BASELINE configs[1], SURVEY.md 8d "C2"): one unit = `focus(pupil, Q=2)` of a 2048^2 complex64
Zernike-aberrated pupil -> 4096^2 complex64 field.  One step = CALLS public `prysm_b200.propagation.focus` calls,
each on a (16, 2048, 2048) stack of distinct pupils resident in HBM (512 MiB in, 2 GiB of distinct outputs per call,
>> 126 MB L2).  Multi-GPU = independent replicas on disjoint batches (weak scaling, no collective on the data path;
SURVEY.md 8e).

The JSON line carries: value (device-resident throughput, CUDA events, max over ranks), e2e (the same metric through
`Wavefront(...).focus()` with pinned HOST buffers, H2D + D2H inside the timed region), roofline (algorithmic bytes /
measured duration against the measured HBM peak), cpu_baseline (the unmodified reference from oracle/_ref on the
host cores), clocks, and -- at every N -- the other BASELINE configs as extras:
  mdft_c3 (N = 1), c4_polychromatic (64 wavelengths sharded over the ranks, ONE NCCL reduce inside the timed region),
  c5_free_space (32-plane screened angular-spectrum chain + CZT final focus, one chain per rank).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N = 2048
Q = 2
K = N * Q
HENE = 0.6328
EFL = 100.0
DX = 10.0 / N
BATCH = 16                       # pupils per library call (16 x 32 MiB = 512 MiB of distinct inputs)
ALG_BYTES = 8 * N * N + 8 * K * K  # SURVEY.md 8(d): read pupil + write field = 167 772 160 B / propagation
METRIC = '2048x2048 pupil->PSF propagations/sec'
WORKLOAD = 'C2: 2048x2048 complex64 pupil -> Wavefront.focus(Q=2) -> 4096x4096 field'


# ---------------------------------------------------------------------------------------------------------------
# synthetic inputs: plain numpy, shared by both arms (no oracle, no reference import)
# ---------------------------------------------------------------------------------------------------------------
def synthetic_pupil(n, seed=20260923):
    """SURVEY 8(d) aperture: unit disk of diameter 10 mm on an n x n grid, OPD [nm] = seeded low-order polynomial
    aberration (defocus, astigmatism, coma, trefoil, spherical) of ~180 nm RMS.  Returns (amp bool, opd float32)."""
    import numpy as np
    g = ((np.arange(n) - n // 2) * (10.0 / n) / 5.0).astype(np.float64)
    x, y = np.meshgrid(g, g)
    r2 = x * x + y * y
    amp = r2 <= 1.0
    c = np.random.default_rng(seed).normal(0, 60.0, 7)
    opd = (c[0] * (2 * r2 - 1) + c[1] * (x * x - y * y) + c[2] * 2 * x * y + c[3] * (3 * r2 - 2) * x +
           c[4] * (3 * r2 - 2) * y + c[5] * (x * x - 3 * y * y) * x + c[6] * (6 * r2 * r2 - 6 * r2 + 1))
    return amp, opd.astype(np.float32)


def make_pupils(count, seed0=20260923):
    """`count` distinct complex64 pupils: the aperture above with a per-pupil piston + tilt (|P| stays in {0, 1})."""
    import numpy as np
    amp, opd = synthetic_pupil(N)
    base = (amp * np.exp(1j * 2 * np.pi / (HENE * 1e3) * opd.astype(np.float64))).astype(np.complex64)
    rng = np.random.default_rng(seed0)
    out = []
    g = np.arange(N, dtype=np.float32) / N
    for _ in range(count):
        ph = rng.uniform(0, 2 * np.pi)
        tilt = rng.uniform(-3, 3, 2)
        mod = np.exp(1j * (ph + 2 * np.pi * (tilt[0] * g[:, None] + tilt[1] * g[None, :]))).astype(np.complex64)
        out.append(base * mod)
    return out


# ---------------------------------------------------------------------------------------------------------------
# host plumbing: clocks, NUMA
# ---------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md)."""

    def __init__(self, index, interval_ms=20):
        self.index = index
        self.interval_ms = interval_ms
        self.rows = []
        self.proc = None

    def start(self):
        q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
             'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
             'clocks_event_reasons.sw_power_cap')
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={q}', '--format=csv,noheader,nounits',
                                          '-i', str(self.index), '-lms', str(self.interval_ms)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [c.strip() for c in line.split(',')]))

    def stop(self, t0=None, t1=None):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.05)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, pw, mx, reasons = [], [], None, set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        rows = [r for (ts, r) in self.rows if t0 is None or t0 <= ts <= t1]
        window = 'timed region'
        if len(rows) < 2:   # nvidia-smi ticks are coarse against a short region: use every sample under the same load
            rows, window = [r for (_, r) in self.rows], 'warm-up + timed region (same workload)'
        for r in rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
                pw.append(float(r[2]))
                for nm, v in zip(names, r[3:7]):
                    if v.lower().startswith('active'):
                        reasons.add(nm)
            except Exception:
                pass
        sm.sort()
        med = sm[len(sm) // 2] if sm else None
        return {'sm_mhz': med, 'sm_min_mhz': sm[0] if sm else None, 'sm_max_mhz': mx, 'power_w_max': max(pw) if pw else None,
                'reasons': sorted(reasons), 'samples': len(sm), 'window': window}


def bind_to_gpu_numa_node(local):
    """Pin this rank's threads to the CPU set of its GPU's NUMA node BEFORE any pinned host buffer is allocated
    (first touch then lands on that node): on the 8-GPU box GPUs 0-3 hang off socket 0 and 4-7 off socket 1, and
    un-bound ranks all stage through one socket's memory / PCIe root (round-1 e2e efficiency 0.6 at N = 8)."""
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=pci.bus_id', '--format=csv,noheader', '-i', str(local)],
                             capture_output=True, text=True, timeout=10).stdout.strip().lower()
        # nvidia-smi prints an 8-digit domain (00000000:1B:00.0); sysfs uses 4 digits
        dom, rest = out.split(':', 1)
        path = f'/sys/bus/pci/devices/{dom[-4:]}:{rest}'
        node = int(open(f'{path}/numa_node').read())
        cpus = open(f'{path}/local_cpulist').read().strip()
        ids = set()
        for part in cpus.split(','):
            a, _, b = part.partition('-')
            ids.update(range(int(a), int(b or a) + 1))
        ids &= os.sched_getaffinity(0)
        if ids:
            os.sched_setaffinity(0, ids)
        return {'numa_node': node, 'cpus': len(ids)}
    except Exception as exc:
        return {'numa_node': None, 'error': repr(exc)[:80]}


# ---------------------------------------------------------------------------------------------------------------
# the reference on the host cores (cpu_baseline, --impl reference)
# ---------------------------------------------------------------------------------------------------------------
def reference_focus():
    """(callable pupil -> 4096^2 complex64 field, kind).  kind = "reference": the UNMODIFIED prysm installed in
    oracle/_ref by oracle/install_reference.sh, driven through its own public API
    (Wavefront(...).focus(efl, Q=2), prysm/propagation/wavefront.py:478-504) at config.precision = 32.
    Fallback when that directory is missing: the oracle port of the same call ("port")."""
    ref_dir = os.path.join(ROOT, 'oracle', '_ref')
    if os.path.isdir(os.path.join(ref_dir, 'prysm')):
        sys.path.insert(0, ref_dir)
        from prysm.conf import config as pconfig
        from prysm.propagation import Wavefront
        pconfig.precision = 32

        def run(pupil):
            return Wavefront(pupil, HENE, DX).focus(EFL, Q=Q).data
        return run, 'reference'
    sys.path.insert(0, os.path.join(ROOT, 'oracle'))
    import prysm_oracle as O
    return (lambda pupil: O.focus(pupil, Q)), 'port'


def cpu_focus_rate(run, seconds_budget, workers, pupils, min_reps=3):
    """Time `run` (one Wavefront.focus(Q=2) of a complex64 2048^2 pupil on the host) with scipy.fft workers."""
    import numpy as np
    from scipy import fft as sfft
    done, t_total = 0, 0.0
    with sfft.set_workers(workers):
        out = run(pupils[0])  # warm-up (plan caches, page faults)
        t_end = time.perf_counter() + seconds_budget
        while True:
            t0 = time.perf_counter()
            out = run(pupils[done % len(pupils)])
            t_total += time.perf_counter() - t0
            done += 1
            if time.perf_counter() > t_end and done >= min_reps:
                break
    assert out.dtype == np.complex64 and out.shape == (K, K)
    return done / t_total, done, t_total


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path (unmodified prysm from oracle/_ref,
    numpy + scipy.fft pocketfft), all host threads, same config / metric.  Rank 0 only."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    # torchrun exports OMP_NUM_THREADS=1 to every rank: undo it before numpy / scipy load so that the N > 1 launch of
    # this arm runs exactly like the N = 1 one (round 1: 3.3 vs 7.3 propagations/s)
    for var in ('OMP_NUM_THREADS', 'OPENBLAS_NUM_THREADS', 'MKL_NUM_THREADS'):
        os.environ[var] = str(cores)
    try:
        os.sched_setaffinity(0, range(cores))
    except Exception:
        pass
    import numpy as np
    from scipy import fft as sfft
    run, kind = reference_focus()
    per_step = 2                                   # bounded sample: 2 propagations per step
    pupils = make_pupils(2)
    with sfft.set_workers(cores):
        for _ in range(max(1, args.warmup)):
            run(pupils[0])
        t0 = time.perf_counter()
        for s in range(args.steps):
            for i in range(per_step):
                out = run(pupils[i % len(pupils)])
        dt = time.perf_counter() - t0
    assert out.dtype == np.complex64
    value = args.steps * per_step / dt
    shipped, n1, _ = cpu_focus_rate(run, 3.0, 1, pupils, min_reps=2)
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': 'propagations/s', 'n_gpus': args.gpus,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1e3 * dt / args.steps,
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'complex64',
        'data': 'synthetic',
        'config': {'workload': WORKLOAD, 'propagations_per_step': per_step, 'host_threads': cores,
                   'call': 'prysm.propagation.Wavefront(pupil, 0.6328, dx).focus(100, Q=2), config.precision = 32'
                           if kind == 'reference' else 'oracle port of Wavefront.focus'},
        'cpu_baseline': {'value': value, 'unit': 'propagations/s', 'cores': cores, 'kind': kind,
                         'sample': f'{args.steps * per_step} propagations, scipy.fft workers={cores}',
                         'as_shipped': {'value': shipped, 'unit': 'propagations/s', 'cores': 1,
                                        'sample': f'{n1} propagations, scipy.fft workers=1 (prysm never sets workers)'}},
        'e2e': {'value': value, 'unit': 'propagations/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------------
# extras: the other BASELINE configs
# ---------------------------------------------------------------------------------------------------------------
def timed(fn, reps, warm, barrier):
    """CUDA events around `reps` calls on torch's current stream, barrier + synchronize on both sides -> ms per call."""
    import torch
    for _ in range(warm):
        fn()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(reps):
        out = fn()
    e1.record()
    barrier()
    return e0.elapsed_time(e1) / reps, out


def measure_mdft_c3(peaks):
    """BASELINE configs[2]: 4096^2 -> 512^2 fixed-sampling focus via MDFT on the tcgen05 tensor cores.
    Algorithmic flops (SURVEY 8d): 8*(My*Ny*Nx + My*Nx*Mx) = 77 309 411 328 per apply."""
    import torch
    from prysm_b200 import propagation as P
    n, m = 4096, 512
    gen = torch.Generator(device='cuda').manual_seed(7)
    a = torch.complex(torch.randn((n, n), generator=gen, device='cuda'), torch.randn((n, n), generator=gen, device='cuda'))
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    ex = P.prepare_executor(10.0 / n, (n, n), HENE * 10.0 / 4, (m, m), HENE, EFL, kind='mdft')
    ex(a)
    torch.cuda.synchronize()
    build_ms = (time.perf_counter() - t0) * 1e3     # executor build + first apply (bases, expansion, descriptors)
    ms, _ = timed(lambda: ex(a), 20, 3, torch.cuda.synchronize)
    sec = ms * 1e-3
    flops = 8 * (m * n * n + m * n * m)
    peak = float(peaks.get('bf16_tflops', 1590.0))
    ach = flops / sec / 1e12
    return {'workload': 'C3: 4096x4096 complex64 -> 512x512 focus_dft(MDFT), 3xTF32 tcgen05 complex GEMM',
            'us_per_apply': sec * 1e6, 'applies_per_s': 1.0 / sec, 'tensor_core_path': ex._tc is not None,
            'executor_build_plus_first_apply_ms': build_ms,
            'roofline': {'bound': 'tensor', 'achieved': ach, 'peak': peak, 'unit': 'TFLOP/s', 'frac': ach / peak,
                         'traffic': None,
                         'peak_source': ('MEASURED_PEAKS.json bf16_tflops (measured, burst)' if 'bf16_tflops' in peaks
                                         else 'fallback 1590 TFLOP/s (B200_PROFILING.md; MEASURED_PEAKS.json absent)'),
                         'algorithmic_flops_per_apply': flops, 'issued_tf32_tflops': 3 * ach,
                         'note': 'algorithmic flops vs the bf16 peak; the path issues 3 TF32 MMAs per product (TF32 runs at half the bf16 rate)'}}


def measure_fused_psf(stack, peak):
    """SURVEY 8(d) 'fused PSF variant': unit = focus(...).intensity with |.|^2 formed in the last pass (fp32 out).
    Algorithmic bytes 8*N^2 + 4*K^2 = 100 663 296 per PSF."""
    import torch
    from prysm_b200 import propagation as P
    nb = stack.shape[0]
    ms, _ = timed(lambda: P.focus_intensity(stack, Q), 20, 3, torch.cuda.synchronize)
    sec = ms * 1e-3 / nb
    alg = 8 * N * N + 4 * K * K
    return {'workload': 'C2 fused PSF variant: 2048x2048 complex64 pupil -> |focus(Q=2)|^2 4096x4096 float32, batched',
            'us_per_psf': sec * 1e6, 'psf_per_s': 1.0 / sec,
            'roofline': {'bound': 'hbm', 'achieved': alg / sec / 1e9, 'peak': peak, 'unit': 'GB/s',
                         'frac': alg / sec / 1e9 / peak, 'traffic': None, 'algorithmic_bytes_per_psf': alg}}


def measure_c4(dev, world, rank, barrier, peak):
    """BASELINE configs[3]: 2048^2 pupil x 64 wavelengths -> common 2048^2 focal grid by CZT (K = 4096), weighted
    incoherent sum; wavelengths sharded round-robin over the ranks, ONE NCCL sum-reduce of the fp32 plane inside the
    timed region (recipe: docs/source/how-tos/Polychromatic Propagation.ipynb:86-98, prysm/polynomials/fitting.py:37).
    Algorithmic bytes per wavelength (SURVEY 8d): 8 N^2 + 4 M^2 = 50 331 648."""
    import numpy as np
    import torch
    import torch.distributed as dist
    from prysm_b200.polychromatic import polychromatic_psf
    amp_h, opd_h = synthetic_pupil(N)
    amp, opd = torch.from_numpy(amp_h).to(dev), torch.from_numpy(opd_h).to(dev)
    wvls = np.linspace(0.5, 0.7, 64)
    wts = np.full(64, 1 / 64)
    M = 2048

    def run(shard=True):
        return polychromatic_psf(amp, opd, wvls, wts, DX, EFL, 2.5, M, kind='czt', dst=0 if (world > 1 and shard) else None,
                                 shard=shard)
    reps = 5
    ms, out = timed(run, reps, 2, barrier)
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    res = {'workload': 'C4: 2048x2048 pupil x 64 wavelengths (0.5-0.7 um) -> 2048x2048 CZT focus (K=4096), weighted |.|^2 sum, '
                       'wavelengths sharded over the ranks, 1 NCCL reduce (16 MiB fp32) inside the timed region',
           'n_gpus': world, 'ms_per_polychromatic_psf': ms, 'psf_per_s': 1e3 / ms,
           'us_per_wavelength_per_gpu': ms * 1e3 / (64 / world)}
    alg = 50331648
    ach = alg * (64 / world) / (ms * 1e-3) / 1e9
    res['roofline'] = {'bound': 'hbm', 'achieved': ach, 'peak': peak, 'unit': 'GB/s', 'frac': ach / peak, 'traffic': None,
                       'algorithmic_bytes_per_wavelength': alg,
                       'note': 'per GPU; the path is FP32-ALU heavy (~40 flop/B, SURVEY 8d): the graded quantity is the speed-up'}
    if world > 1:
        # the same 64 wavelengths on rank 0 alone, in this very run: the denominator of the speed-up; and the reduce alone
        plane = torch.zeros((M, M), dtype=torch.float32, device=dev)
        rms, _ = timed(lambda: dist.reduce(plane, dst=0), 10, 2, barrier)
        tr = torch.tensor([rms], device=dev, dtype=torch.float64)
        dist.all_reduce(tr, op=dist.ReduceOp.MAX)
        res['nccl_reduce_ms'] = float(tr.item())
        res['nccl_reduce_share_of_step'] = float(tr.item()) / ms
        one = None
        if rank == 0:
            one, ref = timed(lambda: run(shard=False), 2, 1, torch.cuda.synchronize)
            denom = float(ref.abs().max())
            res['sharded_vs_single_gpu_rel_linf'] = float((out - ref).abs().max()) / denom
        barrier()
        if rank == 0:
            res['single_gpu_ms_same_run'] = one
            res['speedup_vs_1gpu_same_run'] = one / ms
    if rank == 0:
        res['checksum'] = float(out.double().sum())
    return res


def measure_c5(dev, world, barrier, peak):
    """BASELINE configs[4]: 4096^2 complex64 field, 32 planes of `wf = (wf * s_k).free_space(dz=5)` with distinct
    unit-modulus screens (8 distinct 128 MiB screens cycled: 1 GiB >> L2), then prepare_executor(kind='czt') +
    focus_dft to 512^2 (prysm/propagation/wavefront.py:381-383, 413-443; fttools.py:235-369).  One independent chain
    per rank.  Algorithmic bytes per plane (SURVEY 8d): 3 * 8 * 4096^2 = 402 653 184."""
    import torch
    import torch.distributed as dist
    from prysm_b200 import propagation as P
    n, planes, nscreens, m = 4096, 32, 8, 512
    gen = torch.Generator(device=dev).manual_seed(1000 + int(os.environ.get('RANK', '0')))
    field = torch.polar(torch.ones((n, n), device=dev), torch.randn((n, n), generator=gen, device=dev) * 0.3)
    screens = [torch.polar(torch.ones((n, n), device=dev), torch.randn((n, n), generator=gen, device=dev) * 0.1)
               for _ in range(nscreens)]
    dx = 10.0 / n
    wf0 = P.Wavefront(field, HENE, dx)
    ex = wf0.prepare_executor(EFL, HENE * 10.0 / 4, m, kind='czt')

    def chain():
        wf = wf0
        for k in range(planes):
            wf = (wf * screens[k % nscreens]).free_space(dz=5.0, Q=1)
        return wf

    def full():
        return chain().focus_dft(ex)
    ms_chain, _ = timed(chain, 3, 1, barrier)
    ms_full, psf = timed(full, 3, 1, barrier)
    t = torch.tensor([ms_chain, ms_full], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_chain, ms_full = float(t[0]), float(t[1])
    alg = 3 * 8 * n * n
    us_plane = ms_chain * 1e3 / planes
    ach = alg / (us_plane * 1e-6) / 1e9
    energy = float((psf.data.abs() ** 2).sum())
    return {'workload': 'C5: 4096x4096 complex64, 32 x (screen multiply + free_space(dz=5 mm, Q=1)) with 8 distinct screens cycled, '
                        'then CZT final focus to 512x512; one independent chain per GPU',
            'n_gpus': world, 'ms_per_chain_plus_focus': ms_full, 'us_per_plane': us_plane,
            'us_final_czt_focus': (ms_full - ms_chain) * 1e3, 'chains_per_s': world * 1e3 / ms_full,
            'psf_energy_check': energy,
            'roofline': {'bound': 'hbm', 'achieved': ach, 'peak': peak, 'unit': 'GB/s', 'frac': ach / peak, 'traffic': None,
                         'algorithmic_bytes_per_plane': alg, 'note': 'per GPU, per plane of the chain'}}


def dump_outputs(out, directory):
    """Write what the last timed call returned -- the (BATCH, K, K) complex64 fields -- as float32 [..., (re, im)]:
    focus_field_center.npy   the central 256 x 256 window of every field (8 MiB), where the PSF's energy is
    focus_field_sample.npy   2^21 samples of the whole stack at the flat indices in
    focus_field_index.npy    (float64, seeded, sorted; 16 MiB each)
    so that two builds run with the same arguments can be compared output for output."""
    import numpy as np
    import torch
    os.makedirs(directory, exist_ok=True)
    c, h = K // 2, 128
    np.save(os.path.join(directory, 'focus_field_center.npy'),
            torch.view_as_real(out[:, c - h:c + h, c - h:c + h]).cpu().numpy())
    idx = np.unique(np.random.default_rng(0).integers(0, out.numel(), 1 << 21))
    vals = out.reshape(-1)[torch.from_numpy(idx).to(out.device)]
    np.save(os.path.join(directory, 'focus_field_sample.npy'), torch.view_as_real(vals).cpu().numpy())
    np.save(os.path.join(directory, 'focus_field_index.npy'), idx.astype(np.float64))


# ---------------------------------------------------------------------------------------------------------------
# the B200 arm
# ---------------------------------------------------------------------------------------------------------------
def run_b200(args):
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    numa = bind_to_gpu_numa_node(local)

    import numpy as np  # noqa: F401
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=dev)

    import prysm_b200 as pb
    from prysm_b200 import propagation as P, _ops
    pb.config.precision = 32

    # ---- synthetic inputs: BATCH distinct pupils per rank, resident in HBM before timing
    host_pupils = make_pupils(2, seed0=20260923 + rank)
    base = [torch.from_numpy(p).to(dev) for p in host_pupils]
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    pupils = []
    for i in range(BATCH):  # distinct unit-modulus piston per pupil (built once, outside timing)
        ph = torch.rand((), generator=gen, device=dev) * 6.2831853
        pupils.append((base[i % 2] * torch.polar(torch.ones((), device=dev), ph)).contiguous())
    stack = torch.stack(pupils)                                   # (BATCH, N, N): 512 MiB of distinct inputs
    del pupils
    torch.cuda.synchronize()
    calls = max(1, args.calls_per_step)

    def step():  # CALLS public-API calls; each = one batched library call (pb_fft2_batch) writing 2 GiB of distinct outputs
        for _ in range(calls - 1):
            P.focus(stack, Q)
        return P.focus(stack, Q)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(max(3, args.warmup)):
        step()
    barrier()
    l0 = _ops.launch_count(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_start = time.perf_counter()
    e0.record()
    for _ in range(args.steps - 1):
        step()
    out = step()         # only the last step's result is held, as a caller of the timed path would receive it
    e1.record()
    barrier()
    t_end = time.perf_counter()
    if args.dump_outputs and rank == 0:
        dump_outputs(out, args.dump_outputs)
    del out
    ms = e0.elapsed_time(e1)
    launches = _ops.launch_count(dev) - l0
    clocks = sampler.stop(t_start, t_end) if rank == 0 else None
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    props = args.steps * calls * BATCH
    value = world * props / (ms_max * 1e-3)

    # ---- e2e: public API, pinned host buffers in, pinned host buffers out, copies inside the timed region
    e2e_props = 32
    hin = [torch.from_numpy(host_pupils[i % 2]).pin_memory() for i in range(2)]
    hout = [torch.empty((K, K), dtype=torch.complex64).pin_memory() for _ in range(2)]
    streams = [torch.cuda.Stream(dev) for _ in range(2)]

    def e2e_pass(n):
        for i in range(n):
            s = streams[i % 2]
            with torch.cuda.stream(s):  # double-buffered: copy-in, propagate, copy-out per stream
                d = hin[i % 2].to(dev, non_blocking=True)
                wf = P.Wavefront(d, HENE, DX).focus(EFL, Q=Q)
                hout[i % 2].copy_(wf.data, non_blocking=True)
        for s in streams:
            s.synchronize()

    e2e_pass(4)
    barrier()
    t0 = time.perf_counter()
    e2e_pass(e2e_props)
    torch.cuda.synchronize()
    t_e2e = time.perf_counter() - t0
    t2 = torch.tensor([t_e2e], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t2, op=dist.ReduceOp.MAX)
    e2e_value = world * e2e_props / float(t2.item())
    del hin, hout

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except Exception:
        pass
    peak = float(peaks.get('hbm_gbs', 6650.0))
    peak_src = 'MEASURED_PEAKS.json hbm_gbs (measured)' if 'hbm_gbs' in peaks else 'fallback 6650 GB/s'

    # ---- extras: the single-GPU ones first (rank 0 at N = 1), then the ones every rank takes part in (collectives / barriers).
    # No nvidia-smi sampling around them: NVML queries contend with kernel launches for the driver, and the launch-heavy
    # C4 loop (~10 launches per wavelength) measured 17-40 % slower with a sampler process starting beside it; they are
    # bursts of < 0.2 s that run at the maximum clock.
    extras = {}
    if not args.no_extras:
        if world == 1:
            for name, fn in (('fused_psf', lambda: measure_fused_psf(stack[:8], peak)),
                             ('mdft_c3', lambda: measure_mdft_c3(peaks))):
                try:
                    extras[name] = fn()
                except Exception as exc:  # an extra never takes the headline line down with it
                    extras[name] = {'error': repr(exc)[:300]}
        for name, fn in (('c4_polychromatic', lambda: measure_c4(dev, world, rank, barrier, peak)),
                         ('c5_free_space', lambda: measure_c5(dev, world, barrier, peak))):
            try:
                extras[name] = fn()
            except Exception as exc:
                extras[name] = {'error': repr(exc)[:300]}
                barrier()
            torch.cuda.empty_cache()

    if rank == 0:
        t_prop = ms_max * 1e-3 / props
        achieved = ALG_BYTES / t_prop / 1e9
        traffic, traffic_src = None, None
        try:   # DRAM bytes per propagation of the two focus kernels, from the committed ncu --set full capture of this command
            tr = json.load(open(os.path.join(ROOT, 'profiles', 'r02_focus_traffic.json')))
            traffic, traffic_src = tr['dram_bytes_per_propagation'], tr['source']
        except Exception:
            pass
        cpu = None
        if world == 1:
            cores = os.cpu_count() or 1
            try:
                os.sched_setaffinity(0, range(cores))   # undo the NUMA binding: the baseline gets every host core
            except Exception:
                pass
            run, kind = reference_focus()
            rate, n_done, secs = cpu_focus_rate(run, 10.0, cores, host_pupils)
            shipped, n1, s1 = cpu_focus_rate(run, 3.0, 1, host_pupils, min_reps=2)
            cpu = {'value': rate, 'unit': 'propagations/s', 'cores': cores, 'kind': kind,
                   'sample': f'{n_done} propagations of the same workload in {secs:.1f} s, scipy.fft workers={cores}',
                   'as_shipped': {'value': shipped, 'unit': 'propagations/s', 'cores': 1,
                                  'sample': f'{n1} propagations in {s1:.1f} s, scipy.fft workers=1 (prysm never sets workers)'}}
        line = {
            'metric': METRIC, 'value': value, 'unit': 'propagations/s', 'n_gpus': world, 'steps': args.steps,
            'warmup': max(3, args.warmup), 'ms_per_step': ms_max / args.steps, 'higher_is_better': True,
            'scaling': 'weak', 'vs_baseline': None, 'dtype': 'complex64', 'data': 'synthetic',
            'config': {'workload': WORKLOAD, 'propagations_per_step': calls * BATCH, 'parallelism': f'replicas x{world}',
                       'l2_policy': f'{BATCH} distinct 32 MiB inputs + {BATCH} distinct 128 MiB outputs per call (>> 126 MB L2)',
                       'call': f'{calls} x prysm_b200.propagation.focus(stack (16, 2048, 2048) complex64, Q=2) per step; '
                               'each is one pb_fft2_batch library call',
                       'numa': numa},
            'roofline': {'bound': 'hbm', 'achieved': achieved, 'peak': peak, 'unit': 'GB/s', 'frac': achieved / peak,
                         'traffic': traffic, 'traffic_source': traffic_src, 'peak_source': peak_src,
                         'algorithmic_bytes_per_propagation': ALG_BYTES,
                         'kernel': 'fused focus pipeline (column + row kernel of one propagation), per GPU',
                         'us_per_propagation': t_prop * 1e6},
            'e2e': {'value': e2e_value, 'unit': 'propagations/s', 'h2d_bytes_per_step': 8 * N * N,
                    'd2h_bytes_per_step': 8 * K * K,
                    'note': f'per propagation ({e2e_props} timed): pinned host pupil in, 4096^2 complex64 field back to pinned host memory'},
            'gpu_launches': launches,
            'clocks': clocks,
        }
        if cpu is not None:
            line['cpu_baseline'] = cpu
        line.update(extras)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--calls-per-step', type=int, default=32,
                    help='public-API calls per step (16 propagations each); 32 makes 20 steps last >= 0.5 s')
    ap.add_argument('--no-extras', action='store_true', help='headline only (for ncu captures)')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write the fields the last timed call returned (rank 0; sampled, float32) to DIR/*.npy')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_b200(args)


if __name__ == '__main__':
    main()

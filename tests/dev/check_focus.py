"""GPU: correctness of the tuned focus kernels against the oracle + timing of the single-field and batched calls."""
import os, sys, time
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, 'oracle'))
import prysm_oracle as O
import prysm_b200 as pb
from prysm_b200 import _ops, propagation as P

def rel(a, b): return float(np.abs(a - b).max() / np.abs(b).max())

check = '--check' in sys.argv
rng = np.random.default_rng(1)
if check:
    for N in (512, 1024, 2048):
        a = (rng.standard_normal((N, N)) + 1j * rng.standard_normal((N, N))).astype(np.complex64)
        a64 = a.astype(np.complex128)
        d = pb.asdevice(a)
        f = P.focus(d, 2); u = P.unfocus(d, 2)
        rf, ru = O.focus(a64, 2), O.unfocus(a64, 2)
        I = P.focus_intensity(d, 2)
        acc = torch.ones((2 * N, 2 * N), dtype=torch.float32, device='cuda')
        P.focus_intensity(d, 2, weight=0.5, out=acc)
        amp = rng.random((N, N)) > 0.3
        opd = (rng.standard_normal((N, N)) * 80).astype(np.float32)
        s = P.psf_from_amp_and_phase(amp, opd, 0.6328, 2, field=True)
        rs = O.focus(O.from_amp_and_phase(amp, opd.astype(np.float64), 0.6328), 2)
        print(f'N={N}: focus {rel(f.cpu().numpy(), rf):.2e} unfocus {rel(u.cpu().numpy(), ru):.2e} '
              f'intensity {rel(I.cpu().numpy(), O.intensity(rf)):.2e} accumulate {rel(acc.cpu().numpy(), 1 + 0.5 * O.intensity(rf)):.2e} '
              f'synth {rel(s.cpu().numpy(), rs):.2e}', flush=True)

N = 2048; K = 4096; B = 16
base = pb.asdevice((rng.standard_normal((N, N)) + 1j * rng.standard_normal((N, N))).astype(np.complex64))
ins = [(base * (1 + 0.01 * i)).contiguous() for i in range(B)]
outs = [torch.empty((K, K), dtype=torch.complex64, device='cuda') for _ in range(4)]
def step():
    for i in range(B):
        _ops.fft2(ins[i], (K, K), dir=-1, scale=1.0 / K, shift_in=True, shift_out=True, out=outs[i % 4])
for _ in range(3): step()
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
reps = 10
e0.record()
for _ in range(reps): step()
e1.record(); torch.cuda.synchronize()
us = e0.elapsed_time(e1) * 1e3 / (reps * B)
print(f'single: {us:.1f} us/propagation  {1e6 / us:.0f} prop/s  {167772160 / us / 1e3:.0f} GB/s algorithmic  frac {167772160 / us / 1e3 / 6571.2:.3f}')

# batched form: all B pupils in one pb_fft2_batch call (fields share launches, 8 per launch pair)
stack = torch.stack(ins)
out_b = torch.empty((B, K, K), dtype=torch.complex64, device='cuda')
def step_b():
    _ops.fft2_batch(stack, (K, K), dir=-1, scale=1.0 / K, shift_in=True, shift_out=True, out=out_b)
for _ in range(3): step_b()
torch.cuda.synchronize()
ref = _ops.fft2(ins[5], (K, K), dir=-1, scale=1.0 / K, shift_in=True, shift_out=True)
print('batched == single:', bool(torch.equal(out_b[5], ref)), bool(torch.equal(out_b[15], _ops.fft2(ins[15], (K, K), dir=-1, scale=1.0 / K, shift_in=True, shift_out=True))))
e0.record()
for _ in range(reps): step_b()
e1.record(); torch.cuda.synchronize()
us = e0.elapsed_time(e1) * 1e3 / (reps * B)
print(f'batched: {us:.1f} us/propagation  {1e6 / us:.0f} prop/s  '
      f'{167772160 / us / 1e3:.0f} GB/s algorithmic  frac {167772160 / us / 1e3 / 6571.2:.3f}')

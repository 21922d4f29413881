"""GPU timing of the other BASELINE paths: C5 free-space plane, C4 polychromatic wavelength, psf->mtf, plain fft2."""
import os, sys
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import prysm_b200 as pb
from prysm_b200 import _ops, propagation as P
from prysm_b200.polychromatic import polychromatic_psf

pb.config.precision = 32
def timeit(fn, reps=10, warm=2):
    for _ in range(warm): fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps): fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / reps

gen = torch.Generator(device='cuda').manual_seed(1)
def crand(n): return torch.complex(torch.randn((n, n), generator=gen, device='cuda'), torch.randn((n, n), generator=gen, device='cuda'))
a4 = crand(4096)
us = timeit(lambda: _ops.fft2(a4, (4096, 4096), dir=-1))
print(f'fft2 4096^2 c2c: {us:.0f} us  ({2*134217728/us/1e3:.0f} GB/s algorithmic r+w)')
wf = P.Wavefront(a4, 0.6328, 10.0 / 4096)
scr = crand(4096)
us = timeit(lambda: (wf * scr).free_space(dz=5.0, Q=1))
print(f'C5 plane (screen multiply + free_space 4096^2): {us:.0f} us  ({402653184/us/1e3:.0f} GB/s algorithmic)')
psf = torch.rand((4096, 4096), generator=gen, device='cuda')
us = timeit(lambda: pb.otf.mtf_from_psf(psf, 1.0))
print(f'mtf_from_psf 4096^2: {us:.0f} us')
N = 2048
amp = torch.ones((N, N), device='cuda'); opd = torch.randn((N, N), generator=gen, device='cuda') * 50
wvls = np.linspace(0.5, 0.7, 8); wts = np.full(8, 1 / 8)
us = timeit(lambda: polychromatic_psf(amp, opd, wvls, wts, 10.0 / N, 100.0, 2.5, N, kind='czt'), reps=3, warm=1) / 8
print(f'C4 per wavelength (synth + CZT 2048^2->2048^2 + weighted |.|^2): {us:.0f} us  ({50331648/us/1e3:.0f} GB/s algorithmic)')

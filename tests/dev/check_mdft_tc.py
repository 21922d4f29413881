"""GPU: tcgen05 MDFT vs the CUDA-core GEMM and the fp64 oracle; timing at the C3 size."""
import os, sys, time, hashlib
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, 'oracle'))
import prysm_oracle as O
import prysm_b200 as pb
from prysm_b200 import fttools as F, _ops

pb.config.precision = 32
rng = np.random.default_rng(0)
def rel(a, b): return float(np.abs(a - b).max() / np.abs(b).max())

for (N, M) in ((256, 128), (512, 256), (1024, 128)):
    x = (np.arange(N) - N // 2) * 0.1
    f = (np.arange(M) - M // 2) * (1.0 / (N * 0.1) * 0.37)
    a = (rng.standard_normal((N, N)) + 1j * rng.standard_normal((N, N))).astype(np.complex64)
    ref = O.MDFT(x, x, f, f, -1, 0.5)(a.astype(np.complex128))
    tc = F.MDFT(x, x, f, f, -1, 0.5)
    assert tc._tc is not None
    simt = F.MDFT(x, x, f, f, -1, 0.5, use_tensor_cores=False)
    o_tc = tc(a).cpu().numpy(); o_simt = simt(a).cpu().numpy()
    print('  sha1', hashlib.sha1(o_tc.tobytes()).hexdigest()[:12])
    print(f'N={N} M={M}: tc vs fp64 {rel(o_tc, ref):.2e}   simt vs fp64 {rel(o_simt, ref):.2e}   tc vs simt {rel(o_tc, o_simt):.2e}', flush=True)

if '--big' in sys.argv:
    N, M = 4096, 512
    amp, opd, dx = O.synthetic_pupil(N, np.float32)
    wf = pb.propagation.Wavefront.from_amp_and_phase(amp, opd, 0.6328, dx)
    fdx = 0.6328 * 10.0 / 4
    ex = wf.prepare_executor(100.0, fdx, M, kind='mdft')
    d = wf.data
    out = ex(d); torch.cuda.synchronize()
    g = np.load(os.path.join(ROOT, 'tests', 'golden', 'full_c3.npz'))
    o = out.cpu().numpy(); amax = float(g['field_absmax'])
    print('  sha1', hashlib.sha1(o.tobytes()).hexdigest()[:12])
    print('C3 tc vs reference fp64 (strided samples):', float(np.abs(o[::16, ::16] - g['field_stride']).max() / amax))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(3): ex(d)
    e0.record()
    for _ in range(20): ex(d)
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 20
    fl = 77309411328
    print(f'C3 MDFT apply: {ms*1e3:.1f} us  {fl/ms/1e9:.1f} TFLOP/s algorithmic ({3*fl/ms/1e9:.1f} TF32 TFLOP/s issued)')

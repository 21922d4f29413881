"""GPU: the drop-in path EXECUTED against the unmodified reference (SURVEY 8b).

The user code below is the example of INTEGRATION.md section 1, written against `prysm` only.  It runs twice in
the same process: once on the reference's stock numpy/scipy backend (fp64: the arbiter), once after
`prysm_b200.mathops.set_backend_to_b200()` at precision 32 -- same objects, same calls, CUDA underneath -- and the
results are compared at the north-star tolerance.  The reference is imported from oracle/_ref (installed by
oracle/install_reference.sh); where it is absent, the same user code runs on prysm_b200's own API against the
reference's stored fp64 outputs (tests/golden/dropin.npz).
"""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(ROOT, 'oracle', '_ref')

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def prysm_ref():
    if not os.path.isdir(os.path.join(REF, 'prysm')):
        pytest.skip('oracle/_ref is not installed (run oracle/install_reference.sh)')
    sys.path.insert(0, REF)
    try:
        import prysm
        import prysm.propagation  # noqa: F401
        import prysm.otf  # noqa: F401
        assert os.path.realpath(prysm.__file__).startswith(os.path.realpath(REF))
        yield prysm
    finally:
        sys.path.remove(REF)


def rel(a, b):
    return float(np.abs(np.asarray(a) - np.asarray(b)).max() / np.abs(np.asarray(b)).max())


def model_inputs(N=512):
    """Aperture and OPD [nm] from the reference's own builders (stock backend, fp64), the OPD rounded to float32 ONCE:
    every run below starts from these identical values, so the comparison measures the propagation path and not how
    each precision evaluates a Zernike recurrence."""
    from prysm.coordinates import make_xy_grid, cart_to_polar
    from prysm.geometry import circle
    from prysm.polynomials import zernike_nm_seq, noll_to_nm, sum_of_2d_modes
    x, y = make_xy_grid(N, diameter=10.0)
    r, t = cart_to_polar(x, y)
    amp = circle(5.0, r)
    nms = [noll_to_nm(j) for j in range(2, 12)]
    coefs = np.random.default_rng(3).normal(0, 30.0, len(nms))
    opd = sum_of_2d_modes(zernike_nm_seq(nms, r / 5.0, t), coefs)
    return np.asarray(amp), np.asarray(opd).astype(np.float32)


def user_model(amp, opd32):
    """Pure prysm user code: build a wavefront, focus it, take PSF / MTF, a screened free-space step, and
    fixed-sampling focuses.  Returns host arrays."""
    import prysm.mathops as mathops
    from prysm.propagation import Wavefront
    from prysm.otf import mtf_from_psf
    from prysm.conf import config
    tonp = mathops.array_to_true_numpy
    N = amp.shape[0]
    opd = opd32.astype(config.precision)
    dx = 10.0 / N
    wf = Wavefront.from_amp_and_phase(amp, opd, 0.6328, dx)
    out = {'pupil': tonp(wf.data)}
    psf = wf.focus(efl=100, Q=2)
    out['field'] = tonp(psf.data)
    inten = psf.intensity
    out['psf'] = tonp(inten.data)
    out['psf_dx'] = psf.dx
    mtf = mtf_from_psf(inten)
    out['mtf'] = tonp(mtf.data)
    out['mtf_type'] = type(mtf).__module__
    screen = Wavefront.phase_screen(np.asarray(tonp(opd)) * 0.1, 0.6328, dx)
    fs = (wf * screen).free_space(dz=5.0, Q=1)
    out['free_space'] = tonp(fs.data)
    for kind in ('mdft', 'czt'):
        ex = wf.prepare_executor(100.0, 0.6328 * 10.0 / 4, 128, kind=kind)
        out[kind] = tonp(wf.focus_dft(ex).data)
    out['wf_type'] = type(psf).__module__
    return out


def test_user_code_on_real_prysm_matches_its_numpy_path(prysm_ref):
    import torch
    from prysm.conf import config
    import prysm_b200.mathops as b200
    config.precision = 64
    amp, opd32 = model_inputs()
    ref = user_model(amp, opd32)               # the reference, stock backend, fp64
    config.precision = 32
    ref32 = user_model(amp, opd32)             # the reference's own fp32 run, for the record
    launches0 = None
    try:
        names = b200.set_backend_to_b200()
        assert ('prysm.propagation.wavefront', 'focus') in names
        from prysm_b200 import _ops
        launches0 = _ops.launch_count()
        got = user_model(amp, opd32)
        launches = _ops.launch_count() - launches0
    finally:
        b200.set_backend_to_defaults()
        config.precision = 64
    assert launches >= 10, 'the re-bound path must run on the CUDA kernels'
    assert got['wf_type'].startswith('prysm.') and got['mtf_type'].startswith('prysm.')   # reference classes come back
    assert abs(got['psf_dx'] - ref['psf_dx']) < 1e-9 * ref['psf_dx']
    report = {}
    for key, tol in (('pupil', 1e-6), ('field', 1e-6), ('psf', 1e-6), ('free_space', 1e-6), ('mdft', 1e-6), ('czt', 1e-6)):
        e, e32 = rel(got[key], ref[key]), rel(ref32[key], ref[key])
        report[key] = (e, e32)
        assert e <= tol, f'{key}: {e:.2e} from the reference fp64 result (reference fp32: {e32:.2e})'
    e = float(np.abs(got['mtf'] - ref['mtf']).max())
    assert e <= 2e-6, f'mtf: {e:.2e}'
    print('drop-in vs reference fp64 (ours, reference fp32):', {k: (f'{a:.1e}', f'{b:.1e}') for k, (a, b) in report.items()})
    # after the restore the reference is on numpy again
    from prysm.propagation import Wavefront
    w = Wavefront.from_amp_and_phase(np.ones((8, 8)), np.zeros((8, 8)), 0.5, 1.0)
    assert isinstance(w.data, np.ndarray) and isinstance(w.intensity.data, np.ndarray)
    assert not torch.is_tensor(w.focus(10, Q=2).data)


def b200_user_model(amp, opd32):
    """user_model's calls on prysm_b200's own classes (the same names prysm exports) at precision 32."""
    import prysm_b200 as pb
    from prysm_b200.propagation import Wavefront
    from prysm_b200.otf import mtf_from_psf
    N = amp.shape[0]
    dx = 10.0 / N
    wf = Wavefront.from_amp_and_phase(amp, opd32, 0.6328, dx)
    out = {'pupil': pb.asnumpy(wf.data)}
    psf = wf.focus(efl=100, Q=2)
    out['field'] = pb.asnumpy(psf.data)
    inten = psf.intensity
    out['psf'] = pb.asnumpy(inten.data)
    out['psf_dx'] = psf.dx
    out['mtf'] = pb.asnumpy(mtf_from_psf(inten).data)
    screen = Wavefront.phase_screen(opd32 * 0.1, 0.6328, dx)
    out['free_space'] = pb.asnumpy((wf * screen).free_space(dz=5.0, Q=1).data)
    for kind in ('mdft', 'czt'):
        ex = wf.prepare_executor(100.0, 0.6328 * 10.0 / 4, 128, kind=kind)
        out[kind] = pb.asnumpy(wf.focus_dft(ex).data)
    return out


def test_user_code_matches_reference_golden():
    """The user code above on prysm_b200's API, against the reference's stock fp64 run stored in
    tests/golden/dropin.npz (oracle/make_golden.py dropin): per output the central 16 x 16 window and 2048 seeded samples,
    normalised by the stored max |.| of the full reference array."""
    import torch
    from conftest import load_golden
    import prysm_oracle as O
    import prysm_b200 as pb
    from prysm_b200 import _ops
    if not torch.cuda.is_available():
        pytest.skip('needs a CUDA device')
    g = load_golden('dropin.npz')
    amp, opd32, _ = O.synthetic_pupil(512, np.float32, seed=3, nmodes=10)
    assert np.array_equal(opd32[::8, ::8], g['opd32_stride'])      # the inputs the reference ran on
    pb.config.precision = 32
    try:
        launches0 = _ops.launch_count()
        got = b200_user_model(amp, opd32)
        launches = _ops.launch_count() - launches0
    finally:
        pb.config.precision = 64
    assert launches >= 10, 'the user code must run on the CUDA kernels'
    assert abs(got['psf_dx'] - float(g['psf_dx'])) < 1e-9 * float(g['psf_dx'])
    report = {}
    for key, tol in (('pupil', 1e-6), ('field', 1e-6), ('psf', 1e-6), ('free_space', 1e-6), ('mdft', 1e-6), ('czt', 1e-6),
                     ('mtf', 2e-6)):
        a = np.asarray(got[key])
        cy, cx = a.shape[0] // 2, a.shape[1] // 2
        win = a[cy - 8:cy + 8, cx - 8:cx + 8]
        diff = max(float(np.abs(win - g[f'{key}_win']).max()), float(np.abs(a.ravel()[g[f'{key}_idx']] - g[f'{key}_val']).max()))
        # mtf: absolute (its maximum is 1); the others relative to the reference's max |.|
        e = diff if key == 'mtf' else diff / float(g[f'{key}_max'])
        report[key] = (e, float(g[f'{key}_e32']))
        assert e <= tol, f'{key}: {e:.2e} from the reference fp64 result (reference fp32: {float(g[f"{key}_e32"]):.2e})'
    print('user code vs reference fp64 golden (ours, reference fp32):', {k: (f'{a:.1e}', f'{b:.1e}') for k, (a, b) in report.items()})


def test_elementwise_members_never_touch_numpy_exp(prysm_ref, monkeypatch):
    """With the backend switched, Wavefront.from_amp_and_phase / phase_screen / thin_lens / intensity of the REAL
    prysm class run the kernels: numpy exp is poisoned for the duration and the results are device tensors."""
    import torch
    from prysm.conf import config
    import prysm.mathops as pm
    from prysm.propagation import Wavefront
    import prysm_b200.mathops as b200
    config.precision = 32
    N = 256
    rng = np.random.default_rng(5)
    amp = rng.random((N, N)) > 0.3
    opd = (rng.standard_normal((N, N)) * 50).astype(np.float32)
    g = (np.arange(N) - N // 2) * (10.0 / N)
    x, y = np.meshgrid(g, g)
    want = amp * np.exp(1j * 2 * np.pi / 0.6328 / 1e3 * opd.astype(np.float64))
    want_lens = np.exp(-1j * 2 * np.pi / (0.6328 / 1e3) * (x * x + y * y) / (2 * 500.0))
    try:
        b200.set_backend_to_b200()

        def boom(*a, **k):
            raise AssertionError('numpy exp reached on the re-bound path')
        monkeypatch.setattr(pm.np._srcmodule, 'exp', boom, raising=True)
        wf = Wavefront.from_amp_and_phase(amp, opd, 0.6328, 10.0 / N)
        ps = Wavefront.phase_screen(opd, 0.6328, 10.0 / N)
        tl = Wavefront.thin_lens(500.0, 0.6328, x, y)
        inten = wf.intensity
        prod = wf * ps
        assert all(torch.is_tensor(v) and v.is_cuda for v in (wf.data, ps.data, tl.data, inten.data, prod.data))
        assert isinstance(wf, Wavefront) and type(inten).__module__ == 'prysm._richdata'
        monkeypatch.undo()
        assert rel(wf.data.cpu().numpy(), want) <= 1e-6
        assert rel(tl.data.cpu().numpy(), want_lens) <= 1e-6
        assert rel(inten.data.cpu().numpy(), np.abs(want) ** 2) <= 1e-6
        assert rel(prod.data.cpu().numpy(), want * np.exp(1j * 2 * np.pi / 0.6328 / 1e3 * opd.astype(np.float64))) <= 1e-6
    finally:
        b200.set_backend_to_defaults()
        config.precision = 64

"""Full-array parity report of the BASELINE configs (C2..C5) on a GPU box -> profiles/r02_parity.json.

    python tools/parity_report.py [--out profiles/r02_parity.json] [--small]

Three runs per config on BIT-IDENTICAL inputs (built once by the reference's own fp64 code, the OPD / screen phase
rounded to float32 once, so that input rounding is the same on every side and the numbers below are transform error
only):

    ref64   the unmodified reference (oracle/_ref, numpy + scipy.fft), config.precision = 64   -- the arbiter
    ref32   the same reference at config.precision = 32                                          -- its own fp32 level
    gpu32   prysm_b200 at precision 32 (complex64 kernels)

Metric (SURVEY.md 8d): relative L-infinity over the FULL array, max|a - ref64| / max|ref64|, for the complex field and
for the intensity; the RMS error over the same normaliser is given beside it because at 4096^2 = 1.7e7 samples the
L-infinity of ANY fp32 transform chain sits ~5 sigma above its RMS.  The oracle is not touched:
the reference is imported from oracle/_ref (oracle/install_reference.sh).
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'oracle', '_ref'))

HENE, EFL = 0.6328, 100.0


def metrics(a, ref):
    a = np.asarray(a)
    d = np.abs(a.astype(ref.dtype, copy=False) - ref)
    den = float(np.abs(ref).max())
    return {'rel_linf': float(d.max()) / den, 'rel_rms': float(np.sqrt((d * d).mean())) / den}


def ref_inputs(N):
    from prysm.conf import config
    from prysm.coordinates import make_xy_grid, cart_to_polar
    from prysm.geometry import circle
    from prysm.polynomials import zernike_nm_seq, noll_to_nm, sum_of_2d_modes
    config.precision = 64
    x, y = make_xy_grid(N, diameter=10.0)
    r, t = cart_to_polar(x, y)
    amp = circle(5.0, r)
    nms = [noll_to_nm(j) for j in range(2, 38)]
    coefs = np.random.default_rng(20260923).normal(0, 30.0, 36)
    opd = np.zeros((N, N))
    for nm_chunk, c_chunk in zip(np.array_split(np.arange(36), 6), np.array_split(coefs, 6)):   # bounded memory at 4096^2
        opd += sum_of_2d_modes(zernike_nm_seq([nms[i] for i in nm_chunk], r / 5.0, t), c_chunk)
    return np.asarray(amp), opd.astype(np.float32), 10.0 / N


def run_reference(precision, fn):
    from prysm.conf import config
    from scipy import fft as sfft
    config.precision = precision
    with sfft.set_workers(os.cpu_count() or 1):
        out = fn()
    config.precision = 64
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'r02_parity.json'))
    ap.add_argument('--small', action='store_true', help='quarter-size run (smoke test of this script)')
    args = ap.parse_args()
    import torch
    import prysm
    from prysm.propagation import Wavefront as RW
    import prysm_b200 as pb
    from prysm_b200 import propagation as P
    assert os.path.realpath(prysm.__file__).startswith(os.path.realpath(os.path.join(ROOT, 'oracle', '_ref')))
    sc = 4 if args.small else 1
    rep = {'metric': 'max|a - ref64| / max|ref64| over the full array (rel_linf) and RMS over the same normaliser',
           'inputs': 'built once by the reference in fp64, OPD / screen phase rounded to float32 once, identical on all sides',
           'reference': f'prysm {getattr(prysm, "__version__", "0.22")} from oracle/_ref', 'configs': {}}
    t_all = time.time()

    def gpu(fn):
        pb.config.precision = 32
        out = fn()
        torch.cuda.synchronize()
        pb.config.precision = 64
        return out

    # ---- C2: 2048^2 pupil -> focus(Q=2) -> 4096^2
    N = 2048 // sc
    amp, opd32, dx = ref_inputs(N)

    def ref_c2(prec):
        def f():
            from prysm.conf import config
            wf = RW.from_amp_and_phase(amp, opd32.astype(config.precision), HENE, dx)
            return wf.focus(EFL, Q=2).data
        return run_reference(prec, f)
    r64, r32 = ref_c2(64), ref_c2(32)
    g = gpu(lambda: P.Wavefront.from_amp_and_phase(amp, opd32, HENE, dx).focus(EFL, Q=2).data).cpu().numpy()
    I64 = np.abs(r64) ** 2
    from prysm.otf import mtf_from_psf as ref_mtf
    psf_dx = dx * 0 + HENE * EFL / (dx * 2 * N)
    m64 = run_reference(64, lambda: ref_mtf(I64, psf_dx).data)
    m32 = run_reference(32, lambda: ref_mtf((np.abs(r32.astype(np.complex128)) ** 2).astype(np.float32), psf_dx).data)
    gm = gpu(lambda: pb.otf.mtf_from_psf(P.Wavefront.from_amp_and_phase(amp, opd32, HENE, dx).focus(EFL, Q=2).intensity).data).cpu().numpy()
    mtf = {'gpu32_abs_linf': float(np.abs(gm - m64).max()), 'ref32_abs_linf': float(np.abs(m32 - m64).max())}
    rep['configs']['C2_fft_focus'] = {
        'mtf_from_psf': mtf,
        'shape': [N, 2 * N], 'field': {'gpu32': metrics(g, r64), 'ref32': metrics(r32, r64)},
        'intensity': {'gpu32': metrics(np.abs(g.astype(np.complex128)) ** 2, I64), 'ref32': metrics(np.abs(r32.astype(np.complex128)) ** 2, I64)},
        'energy_conservation_gpu32': float((np.abs(g.astype(np.complex128)) ** 2).sum() / amp.sum() - 1)}
    print('C2', rep['configs']['C2_fft_focus'], flush=True)
    del r64, r32, g, I64

    # ---- C3: 4096^2 -> 512^2 MDFT (and the same window by CZT)
    N, M = 4096 // sc, 512 // sc
    amp, opd32, dx = ref_inputs(N)
    fdx = HENE * (EFL / 10.0) / 4
    out3 = {}
    for kind in ('mdft', 'czt'):
        def ref_c3(prec, kind=kind):
            def f():
                from prysm.conf import config
                wf = RW.from_amp_and_phase(amp, opd32.astype(config.precision), HENE, dx)
                return wf.focus_dft(wf.prepare_executor(EFL, fdx, M, kind=kind)).data
            return run_reference(prec, f)
        r64, r32 = ref_c3(64), ref_c3(32)

        def gfn(kind=kind):
            wf = P.Wavefront.from_amp_and_phase(amp, opd32, HENE, dx)
            return wf.focus_dft(wf.prepare_executor(EFL, fdx, M, kind=kind)).data
        g = gpu(gfn).cpu().numpy()
        out3[kind] = {'field': {'gpu32': metrics(g, r64), 'ref32': metrics(r32, r64)},
                      'intensity': {'gpu32': metrics(np.abs(g.astype(np.complex128)) ** 2, np.abs(r64) ** 2),
                                    'ref32': metrics(np.abs(r32.astype(np.complex128)) ** 2, np.abs(r64) ** 2)}}
    rep['configs']['C3_fixed_sampling_4096_to_512'] = {'shape': [N, M], **out3}
    print('C3', out3, flush=True)

    # ---- C5: screened free-space plane at 4096^2 and the final CZT focus of that plane (same amp / opd as C3)
    phi32 = np.random.default_rng(1000).normal(0, 0.1, (N, N)).astype(np.float32)
    scr_opd32 = (phi32.astype(np.float64) * (HENE * 1e3 / (2 * np.pi))).astype(np.float32)   # OPD [nm] of the screen

    def ref_c5(prec):
        def f():
            from prysm.conf import config
            wf = RW.from_amp_and_phase(amp, opd32.astype(config.precision), HENE, dx)
            scr = RW.phase_screen(scr_opd32.astype(config.precision), HENE, dx)
            plane = (wf * scr).free_space(dz=5.0, Q=1)
            psf = plane.focus_dft(plane.prepare_executor(EFL, fdx, M, kind='czt'))
            return plane.data, psf.data
        return run_reference(prec, f)
    (p64, f64), (p32, f32) = ref_c5(64), ref_c5(32)

    def g_c5():
        wf = P.Wavefront.from_amp_and_phase(amp, opd32, HENE, dx)
        scr = P.Wavefront.phase_screen(scr_opd32, HENE, dx)
        plane = (wf * scr).free_space(dz=5.0, Q=1)
        psf = plane.focus_dft(plane.prepare_executor(EFL, fdx, M, kind='czt'))
        return plane.data, psf.data
    gp, gf = gpu(g_c5)
    gp, gf = gp.cpu().numpy(), gf.cpu().numpy()
    rep['configs']['C5_free_space_plane_and_czt_focus'] = {
        'shape': [N, M],
        'plane_field': {'gpu32': metrics(gp, p64), 'ref32': metrics(p32, p64)},
        'final_focus_field': {'gpu32': metrics(gf, f64), 'ref32': metrics(f32, f64)},
        'final_focus_intensity': {'gpu32': metrics(np.abs(gf.astype(np.complex128)) ** 2, np.abs(f64) ** 2),
                                  'ref32': metrics(np.abs(f32.astype(np.complex128)) ** 2, np.abs(f64) ** 2)},
        'note': 'plane: |field| ~ 1 everywhere, so L-inf over 1.7e7 samples sits ~5 sigma above the RMS for any fp32 chain'}
    print('C5', rep['configs']['C5_free_space_plane_and_czt_focus'], flush=True)
    del p64, f64, p32, f32, gp, gf

    # ---- C4: 2048^2 pupil, CZT to a common 2048^2 grid at two wavelengths + their weighted sum
    N = M = 2048 // sc
    amp, opd32, dx = ref_inputs(N)
    out4 = {}
    tot = {k: 0 for k in ('r64', 'r32', 'g')}
    for w, wt in ((0.5, 0.25), (0.7, 0.75)):
        def ref_c4(prec, w=w):
            def f():
                from prysm.conf import config
                wf = RW.from_amp_and_phase(amp, opd32.astype(config.precision), w, dx)
                return wf.focus_dft(wf.prepare_executor(EFL, 2.5, M, kind='czt')).data
            return run_reference(prec, f)
        r64, r32 = ref_c4(64), ref_c4(32)

        def gfn(w=w):
            wf = P.Wavefront.from_amp_and_phase(amp, opd32, w, dx)
            return wf.focus_dft(wf.prepare_executor(EFL, 2.5, M, kind='czt')).data
        g = gpu(gfn).cpu().numpy()
        out4[f'wavelength_{w}'] = {'field': {'gpu32': metrics(g, r64), 'ref32': metrics(r32, r64)}}
        tot['r64'] = tot['r64'] + wt * np.abs(r64) ** 2
        tot['r32'] = tot['r32'] + wt * np.abs(r32.astype(np.complex128)) ** 2
        tot['g'] = tot['g'] + wt * np.abs(g.astype(np.complex128)) ** 2
    from prysm_b200.polychromatic import polychromatic_psf
    gsum = gpu(lambda: polychromatic_psf(amp, opd32, [0.5, 0.7], [0.25, 0.75], dx, EFL, 2.5, M, kind='czt')).cpu().numpy()
    out4['weighted_sum_intensity'] = {'gpu32_polychromatic_psf': metrics(gsum.astype(np.float64), tot['r64']),
                                      'gpu32_fields': metrics(tot['g'], tot['r64']), 'ref32': metrics(tot['r32'], tot['r64'])}
    rep['configs']['C4_polychromatic_czt_2048'] = {'shape': [N, M], **out4,
                                                  'note': 'the reference builds its fp32 CZT chirps from float32 arguments of ~1e3 rad '
                                                          '(fttools.py:373-379): its own fp32 run is not a 1e-6 arbiter here'}
    print('C4', out4, flush=True)
    rep['seconds'] = time.time() - t_all
    rep['device'] = torch.cuda.get_device_name(0)
    if not args.small:
        os.makedirs(os.path.dirname(args.out), exist_ok=True)
        json.dump(rep, open(args.out, 'w'), indent=1)
        print('written', args.out)


if __name__ == '__main__':
    main()

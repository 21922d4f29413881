"""Generate tests/golden/*.npz from the UNMODIFIED reference (prysm @ /root/reference).

    PYTHONDONTWRITEBYTECODE=1 python oracle/make_golden.py

The reference is Python and cannot travel to the GPU box, so its outputs on seeded inputs
are committed as small fixtures.  `small.npz` holds complete input/output pairs for every
hot-path function at test sizes; `full_*.npz` hold windows / strided samples / checksums of
the reference's fp64 outputs at the BASELINE.json sizes (C1, C2, C3) so that the CUDA path
can be compared with the real reference at full size without shipping 256 MB arrays.
"""
import os
import sys

import numpy as np

REF = os.environ.get('PRYSM_REFERENCE', '/root/reference')
sys.path.insert(0, REF)
sys.dont_write_bytecode = True
OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), '..', 'tests', 'golden')

from prysm.conf import config  # noqa: E402
from prysm import fttools, propagation, otf, psf  # noqa: E402
from prysm.propagation import Wavefront  # noqa: E402
from prysm.coordinates import make_xy_grid, cart_to_polar  # noqa: E402
from prysm.geometry import circle  # noqa: E402
from prysm.polynomials import zernike_nm_seq, noll_to_nm, sum_of_2d_modes  # noqa: E402
from prysm.wavelengths import HeNe  # noqa: E402

config.precision = 64


def crand(rng, shape):
    return rng.standard_normal(shape) + 1j * rng.standard_normal(shape)


def ref_pupil(N, round32=False):
    """SURVEY.md 8(d) builder, executed by the reference's own code in fp64.  round32: the OPD is rounded to float32
    once (and handed on as fp64), so that the fp64 reference run and a complex64 run start from bit-identical values
    and their difference is transform error, not input rounding."""
    x, y = make_xy_grid(N, diameter=10.0)
    r, t = cart_to_polar(x, y)
    amp = circle(5.0, r)
    nms = [noll_to_nm(j) for j in range(2, 38)]
    coefs = np.random.default_rng(20260923).normal(0, 30.0, 36)
    # mode by mode in a fixed order (opd += c_j * Z_j): the summation order of a tensordot is an implementation detail, a
    # loop of IEEE multiply-adds is not -- the fp32-rounded OPD below must be reproducible bit for bit by the tests
    opd = np.zeros((N, N))
    for idx in np.array_split(np.arange(36), 6):      # bounded memory at 4096^2
        for z, c in zip(zernike_nm_seq([nms[i] for i in idx], r / 5.0, t), coefs[idx]):
            opd += c * z
    if round32:
        opd = opd.astype(np.float32).astype(np.float64)
    return amp, opd, 10.0 / N


def small():
    rng = np.random.default_rng(20260923)
    g = {}
    # --- fft focus family (reference tests/test_propagation.py:24-55 shapes and Qs)
    for i, (shp, Q) in enumerate((((8, 8), 1), ((8, 8), 2), ((9, 12), 1.5), ((7, 9), 2), ((16, 16), 2),
                                  ((64, 64), 2), ((12, 5), 3), ((32, 64), 1), ((9, 9), 1))):
        a = crand(rng, shp)
        g[f'focus{i}_in'] = a
        g[f'focus{i}_Q'] = np.float64(Q)
        g[f'focus{i}_focus'] = propagation.focus(a, Q)
        g[f'focus{i}_unfocus'] = propagation.unfocus(a, Q)
        b = crand(rng, g[f'focus{i}_focus'].shape)
        g[f'focus{i}_gin'] = b
        g[f'focus{i}_focus_adjoint'] = propagation.focus_adjoint(b, Q)
        g[f'focus{i}_unfocus_adjoint'] = propagation.unfocus_adjoint(b, Q)
    # --- Wavefront object path on the seeded pupil at N=64
    amp, opd, dx = ref_pupil(64)
    wf = Wavefront.from_amp_and_phase(amp, opd, HeNe, dx)
    psfwf = wf.focus(100.0, Q=2)
    g['wf_amp'], g['wf_opd'], g['wf_dx'] = amp, opd, np.float64(dx)
    g['wf_field'] = wf.data
    g['wf_psf_field'] = psfwf.data
    g['wf_psf_dx'] = np.float64(psfwf.dx)
    g['wf_psf_intensity'] = psfwf.intensity.data
    back = psfwf.unfocus(100.0, Q=1)
    g['wf_back_field'], g['wf_back_dx'] = back.data, np.float64(back.dx)
    mt = otf.mtf_from_psf(psfwf.intensity)
    g['wf_mtf'], g['wf_mtf_df'] = mt.data, np.float64(mt.dx)
    g['wf_ptf'] = otf.ptf_from_psf(psfwf.intensity).data
    g['wf_otf'] = otf.otf_from_psf(psfwf.intensity).data
    g['wf_ee_radii'] = np.array([1.0, 5.0, 12.5, 40.0])
    g['wf_ee'] = otf.encircled_energy(psfwf.intensity.data, psfwf.dx, g['wf_ee_radii'])
    g['wf_centroid'] = np.asarray(psf.centroid(psfwf.intensity.data, psfwf.dx))
    g['wf_centroid_px'] = np.asarray(psf.centroid(psfwf.intensity.data, unit='pixels'))
    x, y = make_xy_grid(64, diameter=10.0)
    g['lens'] = Wavefront.thin_lens(250.0, HeNe, x, y).data
    # --- angular spectrum (reference tests/test_propagation.py:178-243)
    f = crand(rng, (24, 32))
    g['as_in'] = f
    for Q in (1, 2):
        g[f'as_Q{Q}'] = propagation.angular_spectrum(f, HeNe, 0.05, 12.5, Q)
    tf = propagation.angular_spectrum_transfer_function((24, 32), HeNe, 0.05, 12.5)
    g['as_tf'] = tf
    g['as_with_tf'] = propagation.angular_spectrum(f, HeNe, 0.05, 12.5, tf=tf)
    gq = crand(rng, (48, 64))
    g['as_gin'] = gq
    g['as_adjoint_Q2'] = propagation.angular_spectrum_adjoint(gq, HeNe, 0.05, 12.5, 2)
    f9 = crand(rng, (9, 12))
    g['as9_in'] = f9
    g['as9_Q1'] = propagation.angular_spectrum(f9, HeNe, 0.05, 3.0, 1)
    g['as9_Q15'] = propagation.angular_spectrum(f9, HeNe, 0.05, 3.0, 1.5)
    # --- executors
    cases = (((16, 16), (8, 8), 2.0, (0.0, 0.0)), ((9, 12), (8, 11), 1.7, (3.0, -2.0)),
             ((32, 24), (40, 12), 0.9, (0.5, 0.25)), ((64, 64), (32, 32), 3.164, (0.0, 0.0)))
    for i, (pn, fn, fdx, shift) in enumerate(cases):
        a = crand(rng, pn)
        gg = crand(rng, fn)
        g[f'ex{i}_in'], g[f'ex{i}_gin'] = a, gg
        g[f'ex{i}_params'] = np.array([0.1, fdx, HeNe, 100.0, shift[0], shift[1]])
        for kind in ('mdft', 'czt'):
            ex = propagation.prepare_executor(0.1, pn, fdx, fn, HeNe, 100.0, shift, kind)
            g[f'ex{i}_{kind}_fwd'] = ex(a)
            g[f'ex{i}_{kind}_adj'] = ex.adjoint(gg)
    K = 32
    pdx = 0.1
    fdx = HeNe * 100.0 / (pdx * K)
    for i, (pn, fn) in enumerate((((16, 16), (32, 32)), ((20, 16), (12, 32)))):
        a = crand(rng, pn)
        gg = crand(rng, fn)
        ex = propagation.prepare_executor(pdx, pn, fdx, fn, HeNe, 100.0, (0, 0), 'fftdft')
        g[f'fd{i}_in'], g[f'fd{i}_gin'] = a, gg
        g[f'fd{i}_params'] = np.array([pdx, fdx, HeNe, 100.0, 0.0, 0.0])
        g[f'fd{i}_fwd'], g[f'fd{i}_adj'] = ex(a), ex.adjoint(gg)
    # --- incoherent sum
    modes = rng.random((6, 12, 10))
    wts = rng.random(6)
    g['modes'], g['weights'], g['modes_sum'] = modes, wts, sum_of_2d_modes(modes, wts)
    np.savez_compressed(os.path.join(OUT, 'small.npz'), **g)
    print('small.npz', len(g), 'arrays')


def window(a, w):
    cy, cx = a.shape[0] // 2, a.shape[1] // 2
    return a[cy - w // 2:cy + w // 2, cx - w // 2:cx + w // 2]


def full():
    # C1: 256^2 -> 512^2 fp64 FFT focus;  C2: 2048^2 -> 4096^2 (fp64 arbiter for the fp32 GPU path)
    for name, N in (('c1', 256), ('c2', 2048)):
        amp, opd, dx = ref_pupil(N, round32=(name != 'c1'))
        wf = Wavefront.from_amp_and_phase(amp, opd, HeNe, dx)
        ps = wf.focus(100.0, Q=2)
        I = ps.intensity.data
        mt = otf.mtf_from_psf(I, ps.dx).data
        g = dict(N=np.int64(N), psf_dx=np.float64(ps.dx),
                 field_win=window(ps.data, 64), field_stride=ps.data[::N // 16, ::N // 16],
                 field_absmax=np.float64(np.abs(ps.data).max()),
                 I_win=window(I, 64), I_max=np.float64(I.max()), I_sum=np.float64(I.sum()),
                 I_rowsum=I.sum(axis=1)[::8], I_colsum=I.sum(axis=0)[::8],
                 E_in=np.float64((np.abs(wf.data) ** 2).sum()),
                 mtf_win=window(mt, 64), mtf_row=mt[mt.shape[0] // 2, ::8])
        np.savez_compressed(os.path.join(OUT, f'full_{name}.npz'), **g)
        print(f'full_{name}.npz written; I_max={I.max():.6e}')
    # C3: 4096^2 -> 512^2 MDFT (focal_dx = wvl*F#/4)
    N = 4096
    amp, opd, dx = ref_pupil(N, round32=True)
    wf = Wavefront.from_amp_and_phase(amp, opd, HeNe, dx)
    fdx = HeNe * (100.0 / 10.0) / 4
    ex = wf.prepare_executor(100.0, fdx, 512, kind='mdft')
    out = wf.focus_dft(ex).data
    g = dict(N=np.int64(N), M=np.int64(512), focal_dx=np.float64(fdx), norm=np.float64(ex.norm),
             field_win=window(out, 64), field_stride=out[::16, ::16],
             field_absmax=np.float64(np.abs(out).max()),
             I_sum=np.float64((np.abs(out) ** 2).sum()))
    np.savez_compressed(os.path.join(OUT, 'full_c3.npz'), **g)
    print('full_c3.npz written')


def full_c45():
    """BASELINE configs C4 (2048^2 x wavelengths, CZT -> 2048^2) and C5 (4096^2 free-space plane with a phase screen):
    windows / strided samples / sums of the reference's fp64 outputs -> full_c4.npz, full_c5.npz."""
    N = M = 2048
    amp, opd, dx = ref_pupil(N, round32=True)
    g = dict(N=np.int64(N), M=np.int64(M), focal_dx=np.float64(2.5), efl=np.float64(100.0))
    tot = 0
    for w, wt in ((0.5, 0.25), (0.7, 0.75)):
        wf = Wavefront.from_amp_and_phase(amp, opd, w, dx)
        ex = wf.prepare_executor(100.0, 2.5, M, kind='czt')
        f = wf.focus_dft(ex).data
        I = np.abs(f) ** 2
        tot = tot + wt * I
        tag = f'w{int(w * 10)}_'
        g.update({tag + 'field_win': window(f, 64), tag + 'field_stride': f[::64, ::64], tag + 'absmax': np.float64(np.abs(f).max()),
                  tag + 'I_sum': np.float64(I.sum())})
    g.update(sum_win=window(tot, 64), sum_stride=tot[::64, ::64], sum_max=np.float64(tot.max()), sum_total=np.float64(tot.sum()))
    np.savez_compressed(os.path.join(OUT, 'full_c4.npz'), **g)
    print('full_c4.npz written')
    N = 4096
    amp, opd, dx = ref_pupil(N, round32=True)
    wf = Wavefront.from_amp_and_phase(amp, opd, HeNe, dx)
    # the screen exp(i phi), phi ~ N(0, 0.1 rad), expressed as an OPD in nm and rounded to float32 once (see ref_pupil)
    phi32 = np.random.default_rng(1000).normal(0, 0.1, (N, N)).astype(np.float32)
    scr_opd = (phi32.astype(np.float64) * (HeNe * 1e3 / (2 * np.pi))).astype(np.float32).astype(np.float64)
    scr = Wavefront.phase_screen(scr_opd, HeNe, dx)
    plane = (wf * scr).free_space(dz=5.0, Q=1)
    out = plane.data
    fdx = HeNe * (100.0 / 10.0) / 4
    foc = plane.focus_dft(plane.prepare_executor(100.0, fdx, 512, kind='czt')).data      # the chain's final CZT focus
    g = dict(N=np.int64(N), dz=np.float64(5.0), field_win=window(out, 64), field_stride=out[::128, ::128],
             absmax=np.float64(np.abs(out).max()), E_out=np.float64((np.abs(out) ** 2).sum()),
             E_in=np.float64((np.abs(wf.data) ** 2).sum()), edge=out[N // 2, 1000:1100],
             focal_dx=np.float64(fdx), focus_win=window(foc, 64), focus_stride=foc[::16, ::16],
             focus_absmax=np.float64(np.abs(foc).max()), focus_I_sum=np.float64((np.abs(foc) ** 2).sum()))
    np.savez_compressed(os.path.join(OUT, 'full_c5.npz'), **g)
    print('full_c5.npz written')


def coronagraph():
    """Adjoint twins + Lyot-coronagraph compositions (SURVEY.md 8(f) rows) -> coronagraph.npz."""
    from prysm.polynomials import sum_of_2d_modes_adjoint
    rng = np.random.default_rng(20260924)
    g = {}
    # elementwise adjoints
    a = rng.random((18, 24))
    a[2, 3] = 0
    ph = rng.standard_normal((18, 24)) * 40
    wf = Wavefront.from_amp_and_phase(a, ph, 0.55, 0.1)
    bar = Wavefront(crand(rng, (18, 24)), 0.55, 0.1)
    ibar = rng.random((18, 24))
    g.update(ea_amp=a, ea_opd=ph, ea_bar=bar.data, ea_ibar=ibar,
             ea_intensity_adjoint=wf.intensity_adjoint(ibar).data,
             ea_phase=wf.from_amp_and_phase_adjoint_phase(bar),
             ea_amp_nophase=wf.from_amp_and_phase_adjoint_amp(bar),
             ea_amp_phase=wf.from_amp_and_phase_adjoint_amp(bar, phase=ph))
    xg, yg = make_xy_grid((18, 24), dx=0.1)
    g['ea_lens_adjoint'] = np.float64(Wavefront.thin_lens_adjoint(250.0, 0.55, xg, yg, bar))
    # otf adjoints
    pp = rng.random((20, 26))
    D = otf.transform_psf(pp, 1.5)[0]
    rb = rng.standard_normal((20, 26))
    cb = crand(rng, (20, 26))
    g.update(oa_psf=pp, oa_rbar=rb, oa_cbar=cb,
             oa_mtf=otf.mtf_from_psf_adjoint(rb, data=D), oa_ptf=otf.ptf_from_psf_adjoint(rb, data=D),
             oa_otf=otf.otf_from_psf_adjoint(cb, data=D),
             oa_ee=otf.encircled_energy_adjoint([0.3, -1.2], dx=1.5, radius=[2.0, 7.5], data=D))
    modes = rng.random((5, 18, 24))
    g.update(ma_modes=modes, ma_out=sum_of_2d_modes_adjoint(modes, ibar))
    # single-executor compositions
    w = crand(rng, (28, 24))
    gb = crand(rng, (28, 24))
    lyot = rng.random((28, 24))
    fpm_r = rng.random((20, 32))
    fpm_c = crand(rng, (20, 32))
    g.update(co_w=w, co_g=gb, co_lyot=lyot, co_fpm_real=fpm_r, co_fpm_cplx=fpm_c,
             co_params=np.array([0.25, 0.8, 0.55, 20.0]))
    for kind in ('mdft', 'czt'):
        ex = propagation.prepare_executor(0.25, (28, 24), 0.8, (20, 32), 0.55, 20.0, kind=kind)
        for fname, fpm in (('real', fpm_r), ('cplx', fpm_c)):
            t = f'co_{kind}_{fname}_'
            nxt, at, after = propagation.to_fpm_and_back(w, fpm, ex, return_more=True)
            Ea, Eb, it, fb = propagation.to_fpm_and_back_adjoint(gb, fpm, ex, return_more=True, return_fpm_grad=True, field_at_fpm=at)
            al, at2, af2, atl = propagation.babinet(w, lyot, fpm, ex, return_more=True)
            ab, fbb, lb = propagation.babinet_adjoint(gb, lyot, fpm, ex, field_at_fpm=at2, field_at_lyot=atl,
                                                      return_fpm_grad=True, return_lyot_grad=True)
            g.update({t + 'next': nxt, t + 'at_fpm': at, t + 'after_fpm': after, t + 'Eabar': Ea, t + 'Ebbar': Eb,
                      t + 'inter': it, t + 'fpm_bar': fb, t + 'bab_after_lyot': al, t + 'bab_at_fpm': at2,
                      t + 'bab_at_lyot': atl, t + 'bab_abar': ab, t + 'bab_fpm_bar': fbb, t + 'bab_lyot_bar': lb})
    # multi-resolution vortex stack (reference tests/test_propagation.py:544-556 geometry, 3 levels)
    npup = 64
    x = crand(rng, (npup, npup))
    y = crand(rng, (npup, npup))
    g.update(mr_x=x, mr_y=y, mr_params=np.array([0.1, 2.0, HeNe, 10.0]))
    fpm = propagation.vortex_phase_mask(2)
    for kind in ('mdft', 'czt'):
        mr = propagation.prepare_multiresolution(0.1, npup, 2.0, 32, HeNe, 10.0, num_levels=3, fine_samples=32, kind=kind)
        out, at, after = propagation.to_fpm_and_back_multiresolution(x, fpm, mr, return_more=True)
        Ea, Ebs, its, fbs = propagation.to_fpm_and_back_multiresolution_adjoint(y, fpm, mr, return_more=True,
                                                                                return_fpm_grad=True, field_at_fpm=at)
        t = f'mr_{kind}_'
        g.update({t + 'out': out, t + 'Eabar': Ea})
        for k in range(3):
            g.update({t + f'at{k}': at[k], t + f'after{k}': after[k], t + f'Ebbar{k}': Ebs[k], t + f'inter{k}': its[k],
                      t + f'fpm_bar{k}': fbs[k]})
            if kind == 'mdft':
                g.update({f'mr_win{k}': mr.windows[k], f'mr_xf{k}': mr.xf[k], f'mr_yf{k}': mr.yf[k]})
    g['mr_vortex1'] = fpm(mr.xf[1], mr.yf[1])
    # measured-mask resampling (reference tests/test_propagation.py:648-676)
    mm = crand(rng, (41, 37))
    qx = rng.random((24, 30)) * 20 - 10
    qy = rng.random((24, 30)) * 20 - 10
    g.update(mf_map=mm, mf_qx=qx, mf_qy=qy,
             mf_vortex=propagation.prepare_measured_fpm(mm, 0.4, center=(0.3, -0.2), charge=2)(qx, qy),
             mf_scalar=propagation.prepare_measured_fpm(mm, 0.4, center=(0.3, -0.2), fill=0.25)(qx, qy),
             mf_default=propagation.prepare_measured_fpm(mm, 0.4)(qx, qy))
    np.savez_compressed(os.path.join(OUT, 'coronagraph.npz'), **g)
    print(f'coronagraph.npz written, {len(g)} arrays')


def synthesis():
    """Pupil synthesis by recurrence (SURVEY.md 8(f) rank 3) -> synthesis.npz."""
    from prysm import geometry
    from prysm.polynomials import jacobi_seq, zernike_nm, zernike_sum
    rng = np.random.default_rng(20260925)
    g = {}
    x, y = make_xy_grid((33, 40), dx=0.06)
    r, t = cart_to_polar(x, y)
    g.update(grid_x=x, grid_y=y, grid_r=r, grid_t=t, circle=geometry.circle(1.0, r),
             grey=geometry.antialias(geometry.circle_sdf(1.0, r), 0.06))
    xd, yd = make_xy_grid(32, diameter=2.0)
    g.update(grid_xd=xd, grid_yd=yd)
    xs = np.linspace(-1, 1, 65)
    g['jac_x'] = xs
    for i, (al, be) in enumerate(((0, 0), (0, 3), (1.5, 0.5), (-0.5, -0.5))):
        g[f'jac{i}_ab'] = np.array([al, be], dtype=np.float64)
        g[f'jac{i}'] = jacobi_seq([0, 1, 2, 5, 9, 14], al, be, xs)
    nms = [noll_to_nm(j) for j in range(1, 38)]
    rn = r / 1.2
    g['z_nms'] = np.array(nms)
    g['z_seq_norm'] = zernike_nm_seq(nms, rn, t, norm=True)
    g['z_seq_raw'] = zernike_nm_seq(nms, rn, t, norm=False)
    g['z_single'] = zernike_nm(5, -3, rn, t)
    c = rng.standard_normal(37) * 20
    c[4] = 0
    g['z_coefs'] = c
    g['z_sum'] = zernike_sum(c, nms, x / 1.2, y / 1.2)
    np.savez_compressed(os.path.join(OUT, 'synthesis.npz'), **g)
    print(f'synthesis.npz written, {len(g)} arrays')


def imagechain():
    """Image-chain consumers of the path's FFTs (SURVEY.md 8(f) rank 4) -> imagechain.npz."""
    from prysm import convolution
    rng = np.random.default_rng(20260926)
    g = {}
    ob = rng.random((36, 30))
    ps = rng.random((36, 30))
    obc = crand(rng, (36, 30))
    odd = rng.random((15, 9))
    g.update(obj=ob, psf=ps, obj_c=obc, odd_obj=odd, odd_psf=rng.random((15, 9)))
    g['conv_real'] = convolution.conv(ob, ps)
    g['conv_cplx'] = convolution.conv(obc, ps)
    g['conv_odd'] = convolution.conv(odd, g['odd_psf'])
    tf1 = rng.random((36, 30))
    tf2 = crand(rng, (36, 30))
    g.update(tf1=tf1, tf2=tf2)
    for sh in (False, True):
        g[f'atf_shift{int(sh)}'] = convolution.apply_transfer_functions(ob, 0.5, [tf1, tf2], shift=sh)
        g[f'atf_c_shift{int(sh)}'] = convolution.apply_transfer_functions(obc, 0.5, [tf1], shift=sh)
        seen = {}

        def probe(fx, fy, fr, ft):
            seen.update(fx=fx, fy=fy, fr=fr, ft=ft)
            return np.exp(-(fr / 0.7) ** 2)                     # a Gaussian MTF
        g[f'atf_callable_shift{int(sh)}'] = convolution.apply_transfer_functions(ob, 0.5, [probe], shift=sh)
        for k, v in seen.items():
            g[f'grid_{k}_shift{int(sh)}'] = v
    for i, zoom in enumerate((0.5, 2, (2, 1.5))):
        g[f'resample{i}'] = fttools.fourier_resample(ob, zoom)
    g['resample_c'] = fttools.fourier_resample(obc, 2)
    from prysm import detector
    for i, fac in enumerate((2, 3, (2, 3), (4, 6))):
        g[f'bin{i}_avg'] = detector.bindown(ob, fac, 'avg')
        g[f'bin{i}_sum'] = detector.bindown(ob, fac, 'sum')
        g[f'tile{i}_sum'] = detector.tile(ps[:6, :5], fac, 'sum')
    ufy, ufx = (fttools.forward_ft_unit(2.0, n, shift=False) for n in ob.shape)
    g['pixel_ft'] = detector.pixel_ft(ufx.reshape(1, -1), ufy.reshape(-1, 1), 3.0, 2.5)
    g['olpf_ft'] = detector.olpf_ft(ufx.reshape(1, -1), ufy.reshape(-1, 1), 0.7, 0.9)
    np.savez_compressed(os.path.join(OUT, 'imagechain.npz'), **g)
    print(f'imagechain.npz written, {len(g)} arrays')


DROPIN_KEYS = ('pupil', 'field', 'psf', 'mtf', 'free_space', 'mdft', 'czt')


def dropin():
    """The user code of tests/test_gpu_dropin.py (INTEGRATION.md section 1) on the reference's stock backend, fp64,
    from the oracle's synthetic pupil (N = 512, Noll 2..11, seed 3, OPD rounded to float32): per output its max |.|,
    the central 16 x 16 window and 2048 seeded samples, plus the reference's own fp32 error for the record."""
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__))))
    import prysm_oracle as O
    amp, opd32, dx = O.synthetic_pupil(512, np.float32, seed=3, nmodes=10)

    def user_model():
        opd = opd32.astype(config.precision)
        wf = Wavefront.from_amp_and_phase(amp, opd, HeNe, dx)
        psf = wf.focus(efl=100, Q=2)
        inten = psf.intensity
        out = {'pupil': wf.data, 'field': psf.data, 'psf': inten.data, 'mtf': otf.mtf_from_psf(inten).data}
        out['free_space'] = (wf * Wavefront.phase_screen(opd * 0.1, HeNe, dx)).free_space(dz=5.0, Q=1).data
        for kind in ('mdft', 'czt'):
            out[kind] = wf.focus_dft(wf.prepare_executor(100.0, HeNe * 10.0 / 4, 128, kind=kind)).data
        return out, psf.dx
    config.precision = 32
    r32, _ = user_model()
    config.precision = 64
    r64, psf_dx = user_model()
    g = dict(psf_dx=np.float64(psf_dx), opd32_stride=opd32[::8, ::8])
    for k in DROPIN_KEYS:
        a = np.asarray(r64[k])
        idx = np.sort(np.random.default_rng(len(k)).choice(a.size, 2048, replace=False))
        g.update({f'{k}_max': np.float64(np.abs(a).max()), f'{k}_win': window(a, 16), f'{k}_idx': idx.astype(np.int32),
                  f'{k}_val': a.ravel()[idx],
                  f'{k}_e32': np.float64(np.abs(np.asarray(r32[k]) - a).max() / np.abs(a).max())})
    np.savez_compressed(os.path.join(OUT, 'dropin.npz'), **g)
    print('dropin.npz written', {k: f'{float(g[k + "_e32"]):.1e}' for k in DROPIN_KEYS})


if __name__ == '__main__':
    os.makedirs(OUT, exist_ok=True)
    which = sys.argv[1:] or ['small', 'full', 'full_c45', 'coronagraph', 'synthesis', 'imagechain', 'dropin']   # name the fixtures to (re)write
    for name in which:
        {'small': small, 'full': full, 'full_c45': full_c45, 'coronagraph': coronagraph, 'synthesis': synthesis,
         'imagechain': imagechain, 'dropin': dropin}[name]()

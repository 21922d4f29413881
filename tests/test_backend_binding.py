"""CPU: set_backend_to_b200() re-binds prysm's hot-path names and set_backend_to_defaults() restores them.
Runs only where an unmodified prysm is importable: oracle/_ref (oracle/install_reference.sh) or its source tree."""
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_INSTALLED = os.path.join(ROOT, 'oracle', '_ref')
REF = os.environ.get('PRYSM_REFERENCE', _INSTALLED if os.path.isdir(os.path.join(_INSTALLED, 'prysm')) else '/root/reference')


@pytest.fixture()
def prysm_pkg():
    if not os.path.isdir(os.path.join(REF, 'prysm')):
        pytest.skip('the reference prysm is not installed')
    sys.dont_write_bytecode = True
    sys.path.insert(0, REF)
    try:
        import prysm.propagation  # noqa: F401
        import prysm
        yield prysm
    finally:
        sys.path.remove(REF)


def test_rebinding_round_trip(prysm_pkg):
    import prysm.propagation as pp
    import prysm.propagation.wavefront as pw
    import prysm.fttools as pf
    import prysm.otf as po
    from prysm_b200 import mathops, propagation as bp, fttools as bf, otf as bo
    orig = (pp.focus, pw.focus, pw.angular_spectrum, pf.MDFT, po.mtf_from_psf, pw.prepare_executor)
    cls = pw.Wavefront
    patched = ('from_amp_and_phase', 'phase_screen', 'thin_lens', 'intensity', 'phase', 'real', 'imag',
               '__numerical_operation__', 'intensity_adjoint', 'from_amp_and_phase_adjoint_phase')
    orig_cls = {n: cls.__dict__[n] for n in patched}
    names = mathops.set_backend_to_b200()
    try:
        # the reference's Wavefront class is patched IN PLACE (user code that imported it earlier sees the change)
        assert pp.Wavefront is cls and all(cls.__dict__[n] is not orig_cls[n] for n in patched)
        assert isinstance(cls.__dict__['intensity'], property) and isinstance(cls.__dict__['thin_lens'], classmethod)
        assert ('prysm.propagation.wavefront', 'focus') in names
        assert pp.focus is bp.focus and pw.focus is bp.focus            # Wavefront.focus resolves this global
        assert pw.angular_spectrum is bp.angular_spectrum and pw.prepare_executor is bp.prepare_executor
        assert pf.MDFT is bf.MDFT and po.mtf_from_psf.__wrapped_engine__ is bo.mtf_from_psf
        import prysm.propagation.dft as pd
        assert pd.MDFT is bf.MDFT and pd.CZT is bf.CZT                  # prepare_executor's constructors
        import prysm.propagation.coronagraph as pc
        assert pc.babinet is bp.babinet and pw.to_fpm_and_back is bp.to_fpm_and_back   # Wavefront.babinet resolves pw.*
        assert pp.prepare_multiresolution is bp.prepare_multiresolution and pp.vortex_phase_mask is bp.vortex_phase_mask
        assert po.encircled_energy_adjoint.__wrapped_engine__ is bo.encircled_energy_adjoint
    finally:
        mathops.set_backend_to_defaults()
    assert (pp.focus, pw.focus, pw.angular_spectrum, pf.MDFT, po.mtf_from_psf, pw.prepare_executor) == orig
    assert mathops._saved == {} and mathops._saved_cls == {}
    assert all(cls.__dict__[n] is orig_cls[n] for n in patched)

"""Load the reference's numeric core (``/root/reference/muse_psfr/psfrec.py``) in a
container that lacks astropy / mpdaf / matplotlib (SURVEY F3).

TEST INFRASTRUCTURE ONLY: used by ``oracle/make_goldens.py`` to write the reference's
outputs into ``tests/golden/ref_*.npz``, which the tests compare against.

The third-party symbols the numeric core never touches are replaced by stubs that
fail loudly if used, so only the reference's own numpy/scipy code runs:
``simul_psd_wfm``, ``dsp4muse``, ``psd_fit``, ``pupil_mask``, ``psd_to_psf``,
``psf_muse``, ``muse_intrinsic_psf``, ``fit_psf_with_polynom``.
"""
import importlib.util
import sys
import types

REFERENCE_FILE = '/root/reference/muse_psfr/psfrec.py'


class _Missing:
    def __init__(self, *a, **k):
        raise RuntimeError('third-party symbol stubbed out: not part of the numeric core')


def load_reference():
    """Return the reference ``psfrec`` module object (numeric core usable)."""
    if 'ref_psfrec' in sys.modules:
        return sys.modules['ref_psfrec']
    saved = {}

    def stub(name, **attrs):
        saved[name] = sys.modules.get(name)
        mod = types.ModuleType(name)
        mod.__dict__.update(attrs)
        sys.modules[name] = mod
        return mod

    stub('astropy')
    stub('astropy.convolution', Moffat2DKernel=_Missing)
    stub('astropy.io')
    fits = stub('astropy.io.fits', HDUList=type('HDUList', (), {}))
    sys.modules['astropy.io'].fits = fits
    stub('astropy.table', Column=_Missing, Table=_Missing, vstack=_Missing)
    stub('mpdaf')
    stub('mpdaf.obj', Cube=_Missing)
    try:
        spec = importlib.util.spec_from_file_location('ref_psfrec', REFERENCE_FILE)
        ref = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(ref)
    finally:
        for name, old in saved.items():
            if old is None:
                sys.modules.pop(name, None)
            else:
                sys.modules[name] = old
    sys.modules['ref_psfrec'] = ref
    return ref

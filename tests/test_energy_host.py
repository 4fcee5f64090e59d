"""CPU tests of the encircled energy: the overlap geometry of csrc/ee_geometry.h (compiled for the host by nvcc
through tools/ee_check.cu) and the CPU restatement tests/ee_oracle.py, both against scipy.integrate.quad of
the chord length; the restatement's known answers; and the Python surface that needs no device (record
slots, table units, argument refusals, EE_MEAN / EE_FIELD through the FITS writer and reader)."""
import io
import os
import shutil
import subprocess

import numpy as np
import pytest
from numpy.testing import assert_allclose
from scipy.integrate import quad

import ee_oracle as eo
from muse_psfr_b200 import _fits, _lib, psfrec

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LBDA = np.array([500., 700.])


def quad_area(dy, dx, r):
    """Overlap of the pixel centred at (dy, dx) with the disc of radius r: quad of the chord length inside
    [dy - 1/2, dy + 1/2] over x in [dx - 1/2, dx + 1/2], with the chord's kinks as breakpoints."""
    y0, y1, x0, x1 = dy - 0.5, dy + 0.5, dx - 0.5, dx + 0.5

    def chord(x):
        s = np.sqrt(max(r * r - x * x, 0.0))
        return max(0.0, min(y1, s) - max(y0, -s))

    pts = [x for x in (-r, r) + tuple(s * np.sqrt(r * r - y * y) for y in (y0, y1) if abs(y) < r for s in (-1, 1))
           if x0 < x < x1]
    val, err = quad(chord, x0, x1, points=sorted(pts) or None, epsabs=1e-15, epsrel=1e-15, limit=200)
    return val


def cases():
    """(dy, dx, r): random pixels and radii, radii through pixel corners and tangent to pixel edges, pixels
    across the axes, tiny and zero radii."""
    rng = np.random.default_rng(7)
    out = []
    for _ in range(160):
        dy, dx = rng.uniform(-21, 21, 2)
        d = np.hypot(dy, dx)
        out.append((dy, dx, max(0.0, d + rng.uniform(-0.8, 0.8))))
    for k in range(0, 20, 3):
        for m in range(0, 20, 4):
            rc = np.hypot(k + 0.5, m + 0.5)          # circle through a corner of pixel (k, m) and its neighbours
            for dy, dx in ((k, m), (k + 1, m), (k, m + 1), (k + 1, m + 1), (-k, m), (k, -m - 1)):
                out.append((float(dy), float(dx), rc))
    for k in range(0, 20, 2):
        rt = k + 0.5                                # tangent to the edges of the pixels on the axes
        for dy, dx in ((k, 0), (k + 1, 0), (0, -k), (k, 1), (k + 1, 2), (-k - 1, 1)):
            out.append((float(dy), float(dx), rt))
    for dy, dx in ((0.0, 0.0), (0.3, -0.2), (0.5, 0.5), (-0.49, 0.1), (1.2, 0.0)):
        for r in (0.0, 1e-9, 0.1, 0.5, 0.70710678118654757, 1.0, 1.7):
            out.append((dy, dx, r))
    return np.array(out)


@pytest.fixture(scope='module')
def geometry():
    """Area, circle length and area-only result of the library's geometry for every case."""
    nvcc = next((c for c in (os.environ.get('NVCC'), shutil.which('nvcc'), '/usr/local/cuda/bin/nvcc')
                 if c and os.path.exists(c)), None)
    if nvcc is None:
        pytest.skip('nvcc not found')
    import tempfile
    with tempfile.TemporaryDirectory() as tmp:
        exe = os.path.join(tmp, 'ee_check')
        subprocess.run([nvcc, '-O2', '-I', os.path.join(ROOT, 'muse_psfr_b200', 'csrc'),
                        os.path.join(ROOT, 'tools', 'ee_check.cu'), '-o', exe], check=True, cwd=tmp)
        c = cases()
        run = subprocess.run([exe], input='\n'.join('%.17g %.17g %.17g' % tuple(v) for v in c), capture_output=True,
                             text=True, timeout=120, check=True)
    return c, np.array([[float(t) for t in line.split()] for line in run.stdout.splitlines()])


def test_geometry_matches_quad(geometry):
    c, res = geometry
    assert len(res) == len(c) > 400
    ref = np.array([quad_area(*v) for v in c])
    assert np.max(np.abs(res[:, 0] - ref)) <= 1e-13
    assert np.array_equal(res[:, 0], res[:, 2])         # the area does not depend on whether the arc is formed
    assert np.all((res[:, 0] >= 0) & (res[:, 0] <= 1))


def test_geometry_arc_is_the_area_derivative(geometry):
    c, res = geometry
    # the random cases only: corner-through and tangent radii sit on kinks of the area, where the one-sided
    # slopes differ
    h = 1e-5
    dy, dx, r = c[:160].T
    r = np.asarray(r, dtype=eo.LD)
    fd = np.asarray((eo.pixel_area(dy, dx, r + h) - eo.pixel_area(dy, dx, r - h)) / (2 * h), dtype=float)
    assert np.mean(np.abs(res[:160, 1] - fd) < 1e-8) > 0.97


def test_oracle_geometry_matches_quad():
    c = cases()
    ref = np.array([quad_area(*v) for v in c])
    got = np.array([float(eo.pixel_area(dy, dx, r)) for dy, dx, r in c])
    assert np.max(np.abs(got - ref)) <= 1e-13


@pytest.mark.parametrize('r', [0.5, 3.0, np.hypot(7.5, 2.5), 10.5, 15.0, np.hypot(13.5, 13.5), 19.5])
def test_oracle_uniform_image(r):
    img = np.ones((40, 40))
    assert_allclose(float(eo.ee(img, r)), np.pi * r * r, rtol=1e-13)


def test_oracle_known_answers():
    img = np.ones((40, 40))
    assert eo.ee(img, 0.0) == 0
    assert float(eo.ee(img, 40.0)) == 1600.0
    for q in (0.1, 0.5, 0.7):
        assert_allclose(eo.r_at(img, q), np.sqrt(q * 1600 / np.pi), rtol=1e-12)
    one = np.zeros((40, 40))
    one[22, 17] = 2.0
    assert_allclose(float(eo.ee(one, 3.1)), 2.0 * float(eo.pixel_area(2, -3, 3.1)), rtol=1e-15)
    assert np.isnan(eo.r_at(np.zeros((40, 40)), 0.5))


# ---------------------------------------------------------------- Python surface without a device
def test_record_slots_match_header():
    header = open(os.path.join(ROOT, 'include', 'psfr.h')).read()
    assert '#define PSFR_EE_MAX_RADII %d' % _lib.EE_MAX_RADII in header
    assert '#define PSFR_EE_MAX_FRACTIONS %d' % _lib.EE_MAX_FRACTIONS in header
    sl_ee, i_tot, sl_r, rec = _lib.ee_slots(3, 2)
    assert (sl_ee, i_tot, sl_r, rec) == (slice(0, 3), 3, slice(4, 6), 6)
    assert _lib.ee_slots(0, 1)[3] == 2
    for name in ('psfr_encircled_energy', 'psfr_compute_energy'):
        assert name in _lib.exported_symbols() and name in header


def test_table_units():
    rec = np.arange(12, dtype=float).reshape(2, 6) + 1
    tab = psfrec._ee_table(LBDA, rec, [0.2, 0.5, 1.0], [0.5, 0.8])
    assert tab.colnames == ['lbda', 'ee', 'ee_total', 'r_ee']
    assert np.array_equal(tab['ee'], rec[:, :3]) and np.array_equal(tab['ee_total'], rec[:, 3])
    assert_allclose(tab['r_ee'], rec[:, 4:] * 0.2)         # px -> arcsec
    assert np.array_equal(tab.meta['radii'], [0.2, 0.5, 1.0]) and np.array_equal(tab.meta['fractions'], [0.5, 0.8])
    rad, frac = psfrec._ee_params([0.2, 1.0], (0.5,))
    assert_allclose(rad, [1.0, 5.0]) and np.array_equal(frac, [0.5])


BAD = [dict(radii=np.arange(65) * 0.1), dict(radii=[0.5], fractions=np.linspace(0.05, 0.95, 17)),
       dict(radii=[np.nan]), dict(radii=[-0.1]), dict(radii=[np.inf]), dict(radii=[0.5], fractions=[0.0]),
       dict(radii=[0.5], fractions=[1.0]), dict(radii=[0.5], fractions=[0.5, np.nan])]


@pytest.mark.parametrize('bad', BAD)
def test_refusals_before_any_device_call(bad, monkeypatch):
    def no_device(*a, **k):
        raise AssertionError('a device context was requested')
    monkeypatch.setattr(psfrec, 'get_context', no_device)
    monkeypatch.setattr(psfrec, '_planes_context', no_device)
    args = dict(fractions=(0.5, 0.8))
    args.update(bad)
    with pytest.raises(ValueError):
        psfrec.encircled_energy(LBDA, np.ones((2, 40, 40)), args['radii'], args['fractions'])
    with pytest.raises(ValueError):
        psfrec.compute_psf_batch(LBDA, [1.0], [0.7], [25.], ee_radii=args['radii'], ee_fractions=args['fractions'])
    with pytest.raises(ValueError):
        psfrec.compute_psf_field(LBDA, [1.0], [0.7], [25.], ee_radii=args['radii'], ee_fractions=args['fractions'])
    with pytest.raises(ValueError):
        psfrec.compute_psf_from_sparta(psfrec.create_sparta_table(nlines=2), ee_radii=args['radii'],
                                       ee_fractions=args['fractions'])


@pytest.mark.parametrize('center', [(20.0, np.nan), [[20.0, 20.0]], np.zeros((2, 3)), (np.inf, 1.0)])
def test_bad_centres_refused(center, monkeypatch):
    monkeypatch.setattr(psfrec, 'get_context', lambda *a, **k: pytest.fail('device context requested'))
    with pytest.raises(ValueError, match='center'):
        psfrec.encircled_energy(LBDA, np.ones((2, 40, 40)), [0.5], center=center)


def test_empty_inputs():
    tab = psfrec.encircled_energy([], np.empty((0, 40, 40)), [0.2, 0.4], [0.5])
    assert len(tab) == 0 and tab['ee'].shape == (0, 2) and tab['r_ee'].shape == (0, 1)
    fit, cube, ee = psfrec.compute_psf_batch(LBDA, [], [], [], ee_radii=[0.2, 0.4, 0.6])
    assert fit.shape == (0, 2, 16) and ee.shape == (0, 2, 6)
    fit, cube, efit, ee = psfrec.compute_psf_field(LBDA, [], [], [], positions=[[0., 10.], [0., 5.]], elliptical=True,
                                                   ee_radii=[0.5], ee_fractions=[0.5])
    assert efit.shape == (0, 2, 2, 24) and ee.shape == (0, 2, 2, 3)
    fit, cube, ee = psfrec.compute_psf_field([], [1.0], [0.7], [25.], want_cube=False, ee_radii=[0.5])
    assert cube is None and ee.shape == (1, 9, 0, 4)


def test_ee_hdus_round_trip():
    rng = np.random.default_rng(3)
    radii, fracs = np.array([0.2, 0.6, 1.0]), np.array([0.5, 0.8])
    ee_mean = rng.random((2, 6))
    ee_field = rng.random((3, 2, 6))
    meta = psfrec._ee_cards({'SEEING': 0.8, 'GL': 0.7, 'L0': 25.0}, radii, fracs)
    cols = psfrec._ee_columns(LBDA, ee_field, radii, fracs)
    cols['x'] = np.repeat([-30., 0., 12.5], 2)
    cols['y'] = np.repeat([0., 30., -7.3], 2)
    hdul = _fits.HDUList([_fits.PrimaryHDU(),
                          _fits.table_to_hdu(psfrec._ee_columns(LBDA, ee_mean, radii, fracs), meta=meta, name='EE_MEAN'),
                          _fits.table_to_hdu(cols, meta=meta, name='EE_FIELD')])
    buf = io.BytesIO()
    hdul.writeto(buf)
    back = _fits.open(buf.getvalue())
    m = back['EE_MEAN']
    assert np.array_equal(m.data['ee'], ee_mean[:, :3]) and np.array_equal(m.data['ee_total'], ee_mean[:, 3])
    assert np.array_equal(m.data['r_ee'], ee_mean[:, 4:] * 0.2) and np.array_equal(m.data['lbda'], LBDA)
    assert m.header['SEEING'] == 0.8 and m.header['EERAD2'] == 0.6 and m.header['EEFRAC2'] == 0.8
    f = back['EE_FIELD']
    assert f.data['ee'].shape == (6, 3) and np.array_equal(f.data['ee'], ee_field.reshape(6, 6)[:, :3])
    assert np.array_equal(f.data['x'], cols['x']) and np.array_equal(f.data['lbda'], np.tile(LBDA, 3))

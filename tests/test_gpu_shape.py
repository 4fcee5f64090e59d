"""GPU tests of the elliptical Moffat fit: ``psfr_moffat_fit_elliptical``, ``psfr_compute_field_shapes`` and
their Python surface (``fit_psf_cube(circular=False)``, ``compute_psf_field(elliptical=True)``, SHAPE_MEAN /
SHAPE_FIELD of the SPARTA shell).

The fitter is checked on exact model images (known answers), against the CPU reference of tests/efit_oracle.py
on the same GPU-produced PSFs (so that PSF parity does not enter), and the fused outputs against the standalone
call bit for bit."""
import io

import numpy as np
import pytest
from numpy.testing import assert_allclose

import efit_oracle as eo
import psfr_oracle as orc
from test_gpu_field import GROUPS3, GRID3, LBDA6, POS7, draws5, group_inputs, oracle_field, own_context
from test_gpu_sparta_batch import assert_same_result, config2_table

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def psfrec():
    import torch
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    from muse_psfr_b200 import psfrec as mod
    mod.set_device(0)
    mod.release_contexts()
    yield mod
    mod.release_contexts()


def efit_of(ctx, imgs):
    from muse_psfr_b200 import _lib
    imgs = np.ascontiguousarray(imgs, dtype=float)
    n, ny, nx = imgs.reshape(-1, imgs.shape[-2], imgs.shape[-1]).shape
    out = np.full((n, _lib.EFIT_NPAR), np.nan)
    ctx.moffat_fit_elliptical(n, ny, nx, imgs, out)
    return out


def pa_diff_rad(a_deg, b_deg):
    """Distance of two position angles [deg] modulo 180, in radians."""
    d = np.mod(np.asarray(a_deg) - np.asarray(b_deg) + 90.0, 180.0) - 90.0
    return np.abs(np.deg2rad(d))


# ---------------------------------------------------------------- 1. known answers
CASES = [(q, pa, n) for q in (0.999, 0.98, 0.7) for pa in (0., 30., 45., 90., 135., 179.9) for n in (1.5, 2.5, 4.)]


def test_known_answers(psfrec):
    from muse_psfr_b200 import _lib
    ctx = psfrec.get_context()
    centres = [(19.3, 20.6), (17.8, 21.25), (20.0, 18.4)]
    truth = [(2.0 + 0.1 * i, *centres[i % 3], 3.0, 3.0 * q, pa, n) for i, (q, pa, n) in enumerate(CASES)]
    imgs = np.stack([eo.render((40, 40), *t) for t in truth])
    rec = efit_of(ctx, imgs)
    for i, (I, y0, x0, amaj, amin, pa, n) in enumerate(truth):
        r, q = rec[i], amin / amaj
        assert r[_lib.EFIT_ITER] > 0, i
        for slot, ref in ((_lib.EFIT_PEAK, I), (_lib.EFIT_Y0, y0), (_lib.EFIT_X0, x0), (_lib.EFIT_A_MAJOR, amaj),
                          (_lib.EFIT_A_MINOR, amin), (_lib.EFIT_N, n), (_lib.EFIT_AXIS_RATIO, q)):
            assert_allclose(r[slot], ref, rtol=1e-8, err_msg='case %d slot %d' % (i, slot))
        assert 0 <= r[_lib.EFIT_PA] < 180
        assert pa_diff_rad(r[_lib.EFIT_PA], pa) <= 1e-6 / (1 - q), (i, r[_lib.EFIT_PA], pa)
        kf = 2 * np.sqrt(2 ** (1 / n) - 1)
        assert_allclose(r[[_lib.EFIT_FWHM_MAJOR, _lib.EFIT_FWHM_MINOR]], [amaj * kf, amin * kf], rtol=1e-8)
        assert_allclose(r[_lib.EFIT_FLUX], np.pi * I * amaj * amin / (n - 1), rtol=1e-8)
    # a circle: the axis ratio stays at 1 and the orientation is undetermined
    circ = efit_of(ctx, np.stack([eo.render((40, 40), 1.7, 19.3, 20.6, 2.6, 2.6, 0., n) for n in (1.5, 2.5, 4.)]))
    assert np.all(circ[:, _lib.EFIT_AXIS_RATIO] >= 1 - 1e-8) and np.all(circ[:, _lib.EFIT_AXIS_RATIO] <= 1)
    assert_allclose(circ[:, _lib.EFIT_A_MAJOR], 2.6, rtol=1e-8)
    for r in circ:
        assert (r[_lib.EFIT_PA] == 0 and r[_lib.EFIT_ERR_PA] == np.inf) or r[_lib.EFIT_ERR_PA] > 1.0, r


# ---------------------------------------------------------------- 2. parity with the CPU reference, same images
@pytest.fixture(scope='module')
def field7(psfrec):
    seeing, GL, L0, three, h = draws5()
    psfrec.release_contexts()
    return psfrec.compute_psf_field(LBDA6, seeing, GL, L0, positions=POS7, h=h, three_lgs_mode=three, elliptical=True)


def assert_matches_reference(rec, ref):
    from muse_psfr_b200 import _lib
    assert_allclose(rec[:, [_lib.EFIT_FWHM_MAJOR, _lib.EFIT_FWHM_MINOR, _lib.EFIT_N]],
                    ref[:, [eo.FWHM_MAJOR, eo.FWHM_MINOR, eo.N]], rtol=1e-5)
    assert_allclose(rec[:, _lib.EFIT_AXIS_RATIO], ref[:, eo.AXIS_RATIO], rtol=0, atol=1e-5)
    q = ref[:, eo.AXIS_RATIO]
    sel = 1 - q >= 1e-3
    assert np.all(pa_diff_rad(rec[sel, _lib.EFIT_PA], ref[sel, eo.PA]) <= 1e-5 / (1 - q[sel]))
    errs = [_lib.EFIT_ERR_PEAK, _lib.EFIT_ERR_Y0, _lib.EFIT_ERR_X0, _lib.EFIT_ERR_A_MAJOR, _lib.EFIT_ERR_A_MINOR,
            _lib.EFIT_ERR_N, _lib.EFIT_ERR_FWHM_MAJOR, _lib.EFIT_ERR_FWHM_MINOR, _lib.EFIT_ERR_AXIS_RATIO,
            _lib.EFIT_ERR_FLUX]
    assert_allclose(rec[:, errs], ref[:, errs], rtol=1e-4)
    assert_allclose(rec[sel, _lib.EFIT_ERR_PA], ref[sel, eo.ERR_PA], rtol=1e-4)
    assert_allclose(rec[:, [_lib.EFIT_PEAK, _lib.EFIT_FLUX]], ref[:, [eo.PEAK, eo.FLUX]], rtol=1e-5)


def test_parity_with_reference_on_field_psfs(field7):
    from muse_psfr_b200 import _lib
    fit, cube, efit = field7
    imgs = cube.reshape(-1, 40, 40)
    rec = efit.reshape(-1, _lib.EFIT_NPAR)
    assert np.all(rec[:, _lib.EFIT_ITER] > 0)
    ref = np.stack([eo.moffat_fit_elliptical(im)[0] for im in imgs])
    assert_matches_reference(rec, ref)
    # the PSFs are elliptical and their orientation varies over the field
    assert rec[:, _lib.EFIT_AXIS_RATIO].min() < 0.999
    assert np.ptp(rec[rec[:, _lib.EFIT_AXIS_RATIO] < 0.999, _lib.EFIT_PA]) > 20


def test_elliptical_chisq_not_above_circular(field7):
    from muse_psfr_b200 import _lib
    fit, _, efit = field7
    assert np.all(efit[..., _lib.EFIT_CHISQ] <= fit[..., _lib.FIT_CHISQ] * (1 + 1e-12))


def test_end_to_end_off_axis_against_oracle_cube(psfrec):
    from muse_psfr_b200 import _lib
    pos = np.array([[12.5, -30.], [-7.3, 30.]])
    lam = np.array([490., 930.])
    _, _, efit = psfrec.compute_psf_field(lam, [0.8], [0.7], [22.], positions=pos, elliptical=True)
    ref_cubes = oracle_field(lam, 0.8, 0.7, 22., False, pos)
    ref = np.stack([eo.moffat_fit_elliptical(im)[0] for _, psf in ref_cubes for im in psf])
    rec = efit[0].reshape(-1, _lib.EFIT_NPAR)
    assert_allclose(rec[:, [_lib.EFIT_FWHM_MAJOR, _lib.EFIT_FWHM_MINOR, _lib.EFIT_N]],
                    ref[:, [eo.FWHM_MAJOR, eo.FWHM_MINOR, eo.N]], rtol=1e-5)
    assert_allclose(rec[:, _lib.EFIT_AXIS_RATIO], ref[:, eo.AXIS_RATIO], rtol=0, atol=1e-5)


def test_fit_psf_cube_elliptical_table(psfrec, field7):
    from muse_psfr_b200 import _lib
    _, cube, efit = field7
    tab = psfrec.fit_psf_cube(LBDA6, cube[2, 3], circular=False)
    assert np.array_equal(tab['fwhm'], efit[2, 3][:, [_lib.EFIT_FWHM_MAJOR, _lib.EFIT_FWHM_MINOR]] * 0.2)
    assert np.array_equal(tab['pa'], efit[2, 3][:, _lib.EFIT_PA])
    assert np.array_equal(tab['converged'], np.ones(LBDA6.size, dtype=np.int64))
    circ = psfrec.fit_psf_cube(LBDA6, cube[2, 3])
    assert 'axis_ratio' not in circ.colnames


# ---------------------------------------------------------------- 3. fused = standalone, bit for bit
def shape_outputs(nd, npos, nl, ngroup):
    from muse_psfr_b200 import _lib
    return dict(out_cube=np.full((nd, npos, nl, 40, 40), np.nan), out_fit=np.full((nd, npos, nl, _lib.FIT_NPAR), np.nan),
                out_mean=np.full((ngroup, npos, nl, 40, 40), np.nan),
                out_mean_fit=np.full((ngroup, npos, nl, _lib.FIT_NPAR), np.nan),
                out_efit=np.full((nd, npos, nl, _lib.EFIT_NPAR), np.nan),
                out_mean_efit=np.full((ngroup, npos, nl, _lib.EFIT_NPAR), np.nan))


def test_fused_equals_standalone(psfrec):
    """3 positions: at 3 planes one draw per chunk, at 6 two draws (the exposures of 4 and 6 draws span chunk
    edges), at 128 all draws in one chunk."""
    recs, lgs = group_inputs(psfrec)
    pos = np.ascontiguousarray(POS7[:, [1, 5, 6]])
    nl, nd, ng = LBDA6.size, len(recs), len(GROUPS3)
    first = None
    for max_planes in (3, 6, 128):
        ctx = own_context(psfrec, max_planes)
        try:
            out = shape_outputs(nd, 3, nl, ng)
            ctx.compute_field(recs, pos, lgs, LBDA6, GROUPS3, **out)
            plain = {k: np.full(v.shape, np.nan) for k, v in out.items() if 'efit' not in k}
            ctx.compute_field(recs, pos, lgs, LBDA6, GROUPS3, **plain)
            for k, v in plain.items():
                assert np.array_equal(out[k], v), (max_planes, k)
            assert np.array_equal(out['out_efit'].reshape(-1, 24), efit_of(ctx, out['out_cube'].reshape(-1, 40, 40)))
            assert np.array_equal(out['out_mean_efit'].reshape(-1, 24),
                                  efit_of(ctx, out['out_mean'].reshape(-1, 40, 40)))
        finally:
            ctx.close()
        if first is None:
            first = out
        for k in out:
            assert np.array_equal(out[k], first[k]), (max_planes, k)


def test_device_mixed_and_partial_outputs(psfrec):
    import torch
    recs, lgs = group_inputs(psfrec)
    pos = np.ascontiguousarray(POS7[:, :3])
    nl = LBDA6.size
    ctx = own_context(psfrec, 8)
    try:
        full = shape_outputs(len(recs), 3, nl, len(GROUPS3))
        ctx.compute_field(recs, pos, lgs, LBDA6, GROUPS3, **full)
        dev = {n: torch.full(a.shape, np.nan, dtype=torch.float64, device='cuda') for n, a in full.items()}
        ctx.compute_field(recs, pos, lgs, LBDA6, GROUPS3, **dev)
        torch.cuda.synchronize()
        for n, a in full.items():
            assert np.array_equal(dev[n].cpu().numpy(), a), n
        for keep in (('out_efit',), ('out_mean_efit',), ('out_efit', 'out_mean_efit'), ('out_fit', 'out_mean_efit'),
                     ('out_cube', 'out_efit')):
            part = {n: np.full(full[n].shape, np.nan) for n in keep}
            ctx.compute_field(recs, pos, lgs, LBDA6, GROUPS3, **part)
            for n in keep:
                assert np.array_equal(part[n], full[n]), (keep, n)
        mixed = {'out_efit': torch.full(full['out_efit'].shape, np.nan, dtype=torch.float64, device='cuda'),
                 'out_mean_efit': np.full(full['out_mean_efit'].shape, np.nan)}
        ctx.compute_field(recs, pos, lgs, LBDA6, GROUPS3, **mixed)
        torch.cuda.synchronize()
        assert np.array_equal(mixed['out_efit'].cpu().numpy(), full['out_efit'])
        assert np.array_equal(mixed['out_mean_efit'], full['out_mean_efit'])
        # the standalone fit with device images and device records
        imgs = torch.from_numpy(full['out_cube'].reshape(-1, 40, 40)).cuda()
        recs_dev = torch.full((imgs.shape[0], 24), np.nan, dtype=torch.float64, device='cuda')
        ctx.moffat_fit_elliptical(imgs.shape[0], 40, 40, imgs, recs_dev)
        torch.cuda.synchronize()
        assert np.array_equal(recs_dev.cpu().numpy(), full['out_efit'].reshape(-1, 24))
    finally:
        ctx.close()


def test_standalone_chunks_through_staging(psfrec):
    """More host images than the staging buffers hold (1 plane x 35 wavelengths = 35 images per chunk)."""
    _, cube, efit = psfrec.compute_psf_field(LBDA6, [0.9], [0.6], [20.], positions=GRID3, elliptical=True)
    ctx = own_context(psfrec, 1)
    try:
        imgs = np.ascontiguousarray(np.concatenate([cube.reshape(-1, 40, 40)] * 2))
        assert len(imgs) > 35
        rec = efit_of(ctx, imgs)
        assert np.array_equal(rec, np.concatenate([efit.reshape(-1, 24)] * 2))
    finally:
        ctx.close()


# ---------------------------------------------------------------- 4. refusals
def test_refusals(psfrec):
    from muse_psfr_b200 import _lib
    recs, lgs = group_inputs(psfrec)
    pos = np.ascontiguousarray(POS7[:, :3])
    nl = LBDA6.size
    SENT = 12345.0
    ctx = own_context(psfrec, 8)
    outs = {n: np.full(a.shape, SENT) for n, a in shape_outputs(len(recs), 3, nl, len(GROUPS3)).items()}

    def untouched():
        for n, a in outs.items():
            assert np.all(a == SENT), n

    def raw(ndir, dirs, ngroup=3, group_end=GROUPS3.ctypes.data, **kw):
        ptrs = {n: _lib.ptr(outs[n]) for n in outs}
        ptrs.update(kw)
        rc = ctx._lib.psfr_compute_field_shapes(
            ctx._handle(), len(recs), _lib.ptr(recs), 4, _lib.ptr(np.ascontiguousarray(lgs)), ndir, dirs, nl,
            _lib.ptr(np.ascontiguousarray(LBDA6)), ngroup, group_end,
            *[ptrs[n] for n in ('out_cube', 'out_fit', 'out_mean', 'out_mean_fit', 'out_efit', 'out_mean_efit')], None)
        untouched()
        return rc
    try:
        assert raw(3, None) == _lib.E_ARG
        assert raw(9, _lib.ptr(np.ascontiguousarray(GRID3))) == _lib.E_CAPACITY
        for ge in ([4, 4, 11], [5, 4, 11], [4, 5, 10]):
            assert raw(3, _lib.ptr(pos), group_end=np.array(ge, dtype=np.int32).ctypes.data) == _lib.E_ARG
        # an elliptical mean alone needs exposures too
        assert raw(3, _lib.ptr(pos), ngroup=0, group_end=None, out_mean=None, out_mean_fit=None) == _lib.E_ARG
        with pytest.raises(ValueError, match='out_efit'):
            ctx.compute_field(recs, pos, lgs, LBDA6, GROUPS3, out_efit=np.zeros((len(recs), 3, nl, 23)))
        with pytest.raises(ValueError, match='out_mean_efit'):
            ctx.compute_field(recs, pos, lgs, LBDA6, GROUPS3, out_mean_efit=np.zeros((3, 2, nl, 24)))
        # the standalone fit
        img = np.ones((2, 40, 40))
        rec = np.full((2, 24), SENT)
        fn = ctx._lib.psfr_moffat_fit_elliptical
        for args in ((0, 40, 40, _lib.ptr(img), _lib.ptr(rec)), (2, 2, 40, _lib.ptr(img), _lib.ptr(rec)),
                     (2, 40, 2, _lib.ptr(img), _lib.ptr(rec)), (2, 40, 40, None, _lib.ptr(rec)),
                     (2, 40, 40, _lib.ptr(img), None)):
            assert fn(ctx._handle(), *args, None) == _lib.E_ARG, args
            assert np.all(rec == SENT)
        big = np.ones((1, 81, 81))
        assert fn(ctx._handle(), 1, 81, 81, _lib.ptr(big), _lib.ptr(rec), None) == _lib.E_UNSUPPORTED
        assert np.all(rec == SENT)
        assert fn(None, 2, 40, 40, _lib.ptr(img), _lib.ptr(rec), None) == _lib.E_ARG
        # the context still works
        ctx.compute_field(recs, pos, lgs, LBDA6, GROUPS3, out_efit=outs['out_efit'])
        assert np.all(outs['out_efit'][..., _lib.EFIT_ITER] > 0)
    finally:
        ctx.close()


# ---------------------------------------------------------------- 5. the SPARTA shell
def test_sparta_shapes(psfrec):
    from muse_psfr_b200 import _fits, _lib
    tbl = config2_table()
    plain = psfrec.compute_psf_from_sparta_batch([tbl], lbda=LBDA6, verbose=False, field_positions=GRID3)[0]
    got = psfrec.compute_psf_from_sparta_batch([tbl], lbda=LBDA6, verbose=False, field_positions=GRID3,
                                               elliptical=True)[0]
    names = ['PRIMARY', 'SPARTA_ATM_DATA', 'FIT_ROWS', 'FIT_MEAN', 'PSF_MEAN', 'FIT_FIELD', 'PSF_FIELD']
    assert [h.name for h in got] == names + ['SHAPE_MEAN', 'SHAPE_FIELD']
    assert_same_result(_fits.HDUList(list(got)[:7]), plain)
    ctx = psfrec.get_context()
    nl = LBDA6.size
    mean = np.ascontiguousarray(got['PSF_MEAN'].data)
    ref_mean = psfrec._shape_columns(LBDA6, efit_of(ctx, mean))
    ref_field = psfrec._shape_columns(LBDA6, efit_of(ctx, np.ascontiguousarray(got['PSF_FIELD'].data)))
    ref_field['x'] = np.repeat(GRID3[0], nl)
    ref_field['y'] = np.repeat(GRID3[1], nl)

    def check(hdul):
        for name, ref in (('SHAPE_MEAN', ref_mean), ('SHAPE_FIELD', ref_field)):
            tab = hdul[name].data
            assert list(tab.dtype.names) == list(ref), name
            for col, v in ref.items():
                assert np.array_equal(tab[col], v), (name, col)
            for key in ('SEEING', 'GL', 'L0'):
                assert hdul[name].header[key] == got['FIT_MEAN'].header[key]
    check(got)
    buf = io.BytesIO()
    got.writeto(buf)
    check(_fits.open(buf.getvalue()))
    # without field positions only SHAPE_MEAN is appended
    one = psfrec.compute_psf_from_sparta(tbl, lbda=LBDA6, verbose=False, elliptical=True)
    assert [h.name for h in one] == names[:5] + ['SHAPE_MEAN']
    assert_same_result(_fits.HDUList(list(one)[:5]), _fits.HDUList(list(plain)[:5]))
    for col, v in ref_mean.items():
        assert np.array_equal(one['SHAPE_MEAN'].data[col], v), col

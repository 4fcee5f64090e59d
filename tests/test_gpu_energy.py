"""GPU tests of the encircled energy: ``psfr_encircled_energy``, ``psfr_compute_energy`` and their Python surface
(``encircled_energy``, ``compute_psf_batch`` / ``compute_psf_field(ee_radii=...)``, EE_MEAN / EE_FIELD of the
SPARTA shell).

Known answers on synthetic images, parity with the CPU restatement of tests/ee_oracle.py on GPU-produced PSFs,
the fused records against the standalone call bit for bit, and every other output of the fused call against
the existing entry points bit for bit."""
import io

import numpy as np
import pytest
from numpy.testing import assert_allclose

import ee_oracle as eo
from test_gpu_field import GROUPS3, GRID3, LBDA6, POS7, draws5, group_inputs, own_context
from test_gpu_sparta_batch import assert_same_result, config2_table

pytestmark = pytest.mark.gpu

RADII_PX = np.array([0.0, 0.5, 1.0, np.hypot(1.5, 0.5), 2.5, 4.0, np.hypot(3.5, 2.5), 6.5, 10.0, 15.0, 19.5, 25.0,
                     30.0])          # 30 px lies beyond the farthest pixel corner, hypot(20.5, 20.5)
FRACS = np.array([0.5, 0.8, 0.2])
EE_RADII = RADII_PX * 0.2            # arcsec for the Python surface


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


def ee_of(ctx, imgs, radii=RADII_PX, fracs=FRACS, centres=None):
    from muse_psfr_b200 import _lib
    imgs = np.ascontiguousarray(imgs, dtype=float)
    n, ny, nx = imgs.reshape(-1, imgs.shape[-2], imgs.shape[-1]).shape
    out = np.full((n, _lib.ee_slots(len(radii), len(fracs))[3]), np.nan)
    ctx.encircled_energy(n, ny, nx, imgs, radii, fracs, out, centres=centres)
    return out


def assert_oracle_parity(imgs, recs, radii=RADII_PX, fracs=FRACS, centres=None):
    """EE and TOTAL to 1e-14 absolute (the images are unit-sum PSFs), radii at fractions to 1e-9 px."""
    imgs = np.asarray(imgs).reshape(-1, 40, 40)
    recs = np.asarray(recs).reshape(len(imgs), -1)
    nrad = len(radii)
    for i, img in enumerate(imgs):
        ref = eo.record(img, radii, fracs, None if centres is None else centres[i])
        assert np.max(np.abs(recs[i, :nrad + 1] - ref[:nrad + 1])) <= 1e-14, i
        assert np.max(np.abs(recs[i, nrad + 1:] - ref[nrad + 1:])) <= 1e-9, i


# ---------------------------------------------------------------- 1. known answers
def test_uniform_image_is_pi_r_squared(psfrec):
    ctx = psfrec.get_context()
    corners = [np.hypot(k + 0.5, m + 0.5) for k in range(0, 14, 3) for m in range(0, 14, 4)]
    tangents = [k + 0.5 for k in range(20)]
    radii = np.array(sorted(corners + tangents + [0.0, 0.3, 7.77, 19.5]))
    assert len(radii) <= 64
    rec = ee_of(ctx, np.full((1, 40, 40), 1.0), radii, [0.5, 0.25])[0]
    assert rec[0] == 0.0
    assert_allclose(rec[1:len(radii)], np.pi * radii[1:] ** 2, rtol=1e-13)
    assert rec[len(radii)] == 1600.0
    assert_allclose(rec[len(radii) + 1:], np.sqrt(np.array([0.5, 0.25]) * 1600 / np.pi), atol=1e-9)


def test_single_pixel_zero_radius_and_full_aperture(psfrec):
    ctx = psfrec.get_context()
    imgs = np.zeros((3, 40, 40))
    imgs[0, 22, 17] = 2.0
    imgs[1, 20, 20] = 1.0
    rng = np.random.default_rng(4)
    imgs[2] = rng.random((40, 40))
    radii = np.array([0.0, 0.5, 1.3, np.hypot(2.5, 3.5), 3.9, 5.0, 29.0, 29.5, 100.0])
    rec = ee_of(ctx, imgs, radii, [0.5])
    area = np.array([float(eo.pixel_area(2, -3, r)) for r in radii])
    assert_allclose(rec[0, :len(radii)], 2.0 * area, atol=1e-15, rtol=1e-14)
    assert np.all(rec[:, 0] == 0.0)
    assert_allclose(rec[1, 1], np.pi / 4, rtol=1e-15)       # r = 0.5 is inscribed in the lit pixel (20, 20)
    for i in range(3):                      # beyond the farthest corner (hypot(20.5, 20.5) = 28.99): EE == TOTAL
        assert np.all(rec[i, 6:9] == rec[i, len(radii)]), i
    assert rec[2, len(radii)] == ee_of(ctx, imgs[2:], [1e3], [])[0, 0]


def test_centres_and_nonpositive_totals(psfrec):
    ctx = psfrec.get_context()
    rng = np.random.default_rng(9)
    imgs = rng.random((4, 40, 40))
    imgs[3] = -imgs[3]
    centres = np.array([[20.0, 20.0], [17.3, 22.65], [0.0, 39.5], [12.25, 8.0]])
    radii = np.array([0.0, 0.75, 2.5, np.hypot(1.5, 2.5), 6.0, 12.5, 60.0])
    rec = ee_of(ctx, imgs, radii, [0.5, 0.9], centres=centres)
    assert np.array_equal(rec[0], ee_of(ctx, imgs[:1], radii, [0.5, 0.9])[0])     # default centre = (20, 20)
    assert_oracle_parity(imgs[:3] / 1600, ee_of(ctx, imgs[:3] / 1600, radii, [0.5, 0.9], centres=centres[:3]),
                         radii, [0.5, 0.9], centres[:3])
    assert np.all(np.isnan(rec[3, -2:]))    # TOTAL < 0
    uni = ee_of(ctx, np.ones((1, 40, 40)), [3.3, 7.25], [], centres=np.array([[17.6, 21.2]]))[0]
    assert_allclose(uni[:2], np.pi * np.array([3.3, 7.25]) ** 2, rtol=1e-13)


def test_broad_moffat_half_light_radius(psfrec):
    """A Moffat with a = 6 px and n = 3 sampled at the pixel centres: the half-light radius of the continuous
    profile is a sqrt(2^(1/(n-1)) - 1).  The box holds all but 0.7 % of the flux and the pixels are point
    samples, so r_50 of the image is not exactly that: it lies 7e-4 above (tests/ee_oracle.py gives the same)."""
    ctx = psfrec.get_context()
    a, n = 6.0, 3.0
    p, q = np.mgrid[:40, :40]
    img = (1 + ((p - 20) ** 2 + (q - 20) ** 2) / a ** 2) ** (-n)
    rec = ee_of(ctx, img[None], [], [0.5])[0]
    assert abs(rec[1] / (a * np.sqrt(2 ** (1 / (n - 1)) - 1)) - 1) < 1e-3
    assert abs(rec[1] - eo.r_at(img, 0.5)) < 1e-9


# ---------------------------------------------------------------- 2. parity with the restatement on GPU PSFs
def test_parity_batch_field_and_means(psfrec):
    seeing, GL, L0, three, h = draws5()
    fit, cube, ee = psfrec.compute_psf_batch(LBDA6, seeing[:2], GL[:2], L0[:2], ee_radii=EE_RADII,
                                             ee_fractions=FRACS)
    assert ee.shape == (2, LBDA6.size, len(RADII_PX) + 1 + len(FRACS))
    assert_oracle_parity(cube, ee)
    fit, cube, ee = psfrec.compute_psf_field(LBDA6, seeing[:1], GL[:1], L0[:1], positions=POS7, ee_radii=EE_RADII,
                                             ee_fractions=FRACS)
    assert ee.shape == (1, 7, LBDA6.size, len(RADII_PX) + 1 + len(FRACS))
    assert_oracle_parity(cube, ee)
    recs, lgs = group_inputs(psfrec)
    ctx = own_context(psfrec, 6)
    try:
        out = energy_outputs(len(recs), 3, LBDA6.size, len(GROUPS3))
        ctx.compute_energy(True, recs, np.ascontiguousarray(POS7[:, :3]), lgs, LBDA6, RADII_PX, FRACS, GROUPS3,
                           out_mean=out['out_mean'], out_mean_ee=out['out_mean_ee'])
        assert_oracle_parity(out['out_mean'], out['out_mean_ee'])
    finally:
        ctx.close()


# ---------------------------------------------------------------- 3. fused = standalone, bit for bit
def energy_outputs(nd, npos, nl, ngroup, rec=len(RADII_PX) + 1 + len(FRACS)):
    from muse_psfr_b200 import _lib
    return dict(out_cube=np.full((nd, npos, nl, 40, 40), np.nan), out_fit=np.full((nd, npos, nl, _lib.FIT_NPAR), np.nan),
                out_mean=np.full((ngroup, npos, nl, 40, 40), np.nan),
                out_mean_fit=np.full((ngroup, npos, nl, _lib.FIT_NPAR), np.nan),
                out_efit=np.full((nd, npos, nl, _lib.EFIT_NPAR), np.nan),
                out_mean_efit=np.full((ngroup, npos, nl, _lib.EFIT_NPAR), np.nan),
                out_ee=np.full((nd, npos, nl, rec), np.nan), out_mean_ee=np.full((ngroup, npos, nl, rec), np.nan))


def launches(ctx, fn, *args, **kw):
    n0 = ctx.kernel_launches()
    fn(*args, **kw)
    return ctx.kernel_launches() - n0


def run_energy(ctx, field, recs, pos, lgs, out):
    ctx.compute_energy(field, recs, pos, lgs, LBDA6, RADII_PX, FRACS, GROUPS3, **out)


@pytest.mark.parametrize('field', [False, True])
def test_fused_equals_standalone_and_existing_entry_points(psfrec, field):
    """At 3 planes one draw per chunk (field) or three, at 8 several with the exposures across chunk edges, at 128
    all draws in one chunk.  The other outputs equal psfr_compute_groups / psfr_compute_field_shapes bit for bit,
    and the EE stage adds one launch per chunk and one per chunk where exposures end."""
    recs, lgs = group_inputs(psfrec)
    npos = 3
    pos = np.ascontiguousarray(POS7[:, [1, 5, 6]] if field else GRID3[:, [0, 4, 8]])
    P = npos if field else 1
    nl, nd, ng = LBDA6.size, len(recs), len(GROUPS3)
    first = None
    for max_planes in (3, 8, 128):
        ctx = own_context(psfrec, max_planes)
        try:
            out = energy_outputs(nd, P, nl, ng)
            ctx.compute_groups(recs, pos, lgs, LBDA6, GROUPS3, out_fit=out['out_fit'])   # builds the MUSE kernels once
            n_energy = launches(ctx, run_energy, ctx, field, recs, pos, lgs, out)
            plain = {k: np.full(v.shape, np.nan) for k, v in out.items() if '_ee' not in k}
            if field:
                n_plain = launches(ctx, ctx.compute_field, recs, pos, lgs, LBDA6, GROUPS3, **plain)
            else:
                plain = {k: v for k, v in plain.items() if 'efit' not in k}
                n_plain = launches(ctx, ctx.compute_groups, recs, pos, lgs, LBDA6, GROUPS3, **plain)
                efit = ctx.moffat_fit_elliptical
                efit(nd * nl, 40, 40, out['out_cube'], efit_ref := np.full(out['out_efit'].shape, np.nan))
                efit(ng * nl, 40, 40, out['out_mean'], mefit_ref := np.full(out['out_mean_efit'].shape, np.nan))
                assert np.array_equal(out['out_efit'], efit_ref) and np.array_equal(out['out_mean_efit'], mefit_ref)
            for k, v in plain.items():
                assert np.array_equal(out[k], v), (max_planes, k)
            assert np.array_equal(out['out_ee'].reshape(nd * P * nl, -1), ee_of(ctx, out['out_cube']))
            assert np.array_equal(out['out_mean_ee'].reshape(ng * P * nl, -1), ee_of(ctx, out['out_mean']))
            # launches: with the outputs of the existing entry point only, the same count; the EE stage adds one
            # launch per chunk and one per chunk in which exposures end
            same = {k: np.full(v.shape, np.nan) for k, v in plain.items()}
            assert launches(ctx, run_energy, ctx, field, recs, pos, lgs, same) == n_plain, max_planes
            per_chunk = max_planes // npos
            chunks = -(-nd // per_chunk)
            ends = len({(int(e) - 1) // per_chunk for e in GROUPS3})
            with_efit = {k: np.full(v.shape, np.nan) for k, v in out.items() if '_ee' not in k}
            n_efit = launches(ctx, run_energy, ctx, field, recs, pos, lgs, with_efit)
            assert n_efit + chunks + ends == n_energy, (max_planes, n_efit, n_energy)
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
        full = energy_outputs(len(recs), 3, nl, len(GROUPS3))
        run_energy(ctx, True, recs, pos, lgs, full)
        dev = {n: torch.full(a.shape, np.nan, dtype=torch.float64, device='cuda') for n, a in full.items()}
        run_energy(ctx, True, recs, pos, lgs, dev)
        torch.cuda.synchronize()
        for n, a in full.items():
            assert np.array_equal(dev[n].cpu().numpy(), a), n
        for keep in (('out_ee',), ('out_mean_ee',), ('out_ee', 'out_mean_ee'), ('out_fit', 'out_mean_ee'),
                     ('out_cube', 'out_ee', 'out_mean_efit')):
            part = {n: np.full(full[n].shape, np.nan) for n in keep}
            run_energy(ctx, True, recs, pos, lgs, part)
            for n in keep:
                assert np.array_equal(part[n], full[n]), (keep, n)
        mixed = {'out_ee': torch.full(full['out_ee'].shape, np.nan, dtype=torch.float64, device='cuda'),
                 'out_mean_ee': np.full(full['out_mean_ee'].shape, np.nan)}
        run_energy(ctx, True, recs, pos, lgs, mixed)
        torch.cuda.synchronize()
        assert np.array_equal(mixed['out_ee'].cpu().numpy(), full['out_ee'])
        assert np.array_equal(mixed['out_mean_ee'], full['out_mean_ee'])
        # the standalone call with device images, centres and records, and through the staging in chunks
        imgs = torch.from_numpy(full['out_cube'].reshape(-1, 40, 40)).cuda()
        rec_dev = torch.full((imgs.shape[0], full['out_ee'].shape[-1]), np.nan, dtype=torch.float64, device='cuda')
        cen = torch.full((imgs.shape[0], 2), 20.0, dtype=torch.float64, device='cuda')
        ctx.encircled_energy(imgs.shape[0], 40, 40, imgs, RADII_PX, FRACS, rec_dev, centres=cen)
        torch.cuda.synchronize()
        assert np.array_equal(rec_dev.cpu().numpy(), full['out_ee'].reshape(imgs.shape[0], -1))
        small = own_context(psfrec, 1)
        try:
            many = np.concatenate([full['out_cube'].reshape(-1, 40, 40)] * 2)
            assert len(many) > 35
            assert np.array_equal(ee_of(small, many), np.concatenate([full['out_ee'].reshape(len(many) // 2, -1)] * 2))
        finally:
            small.close()
    finally:
        ctx.close()


# ---------------------------------------------------------------- 4. nothing else moves
@pytest.mark.parametrize('mode', ['four', 'three', 'per_draw'])
def test_compute_psf_batch_fit_and_cube_unchanged(psfrec, mode):
    """The EE path runs the groups entry point, with DRAW_NGS filled in scalar mode: the fit and the cube equal
    psfr_compute_batch's bit for bit, and want_cube=False gives the same records."""
    seeing, GL, L0, three, _ = draws5()
    flag = {'four': False, 'three': True, 'per_draw': three}[mode]
    fit0, cube0 = psfrec.compute_psf_batch(LBDA6, seeing, GL, L0, npsflin=3, three_lgs_mode=flag, max_planes=18)
    fit, cube, ee = psfrec.compute_psf_batch(LBDA6, seeing, GL, L0, npsflin=3, three_lgs_mode=flag, max_planes=18,
                                             ee_radii=EE_RADII, ee_fractions=FRACS)
    assert np.array_equal(fit, fit0) and np.array_equal(cube, cube0)
    fit2, none, ee2 = psfrec.compute_psf_batch(LBDA6, seeing, GL, L0, npsflin=3, three_lgs_mode=flag, max_planes=18,
                                               ee_radii=EE_RADII, ee_fractions=FRACS, want_cube=False)
    assert none is None and np.array_equal(fit2, fit0) and np.array_equal(ee2, ee)
    radii_px = psfrec._ee_params(EE_RADII, FRACS)[0]        # EE_RADII / 0.2, as compute_psf_batch converts them
    assert np.array_equal(ee.reshape(-1, ee.shape[-1]), ee_of(psfrec.get_context(), cube, radii_px))


def test_compute_psf_field_outputs_unchanged(psfrec):
    seeing, GL, L0, three, h = draws5()
    base = psfrec.compute_psf_field(LBDA6, seeing[:2], GL[:2], L0[:2], positions=POS7[:, :4], elliptical=True)
    got = psfrec.compute_psf_field(LBDA6, seeing[:2], GL[:2], L0[:2], positions=POS7[:, :4], elliptical=True,
                                   ee_radii=EE_RADII, ee_fractions=FRACS)
    assert len(got) == 4
    for a, b in zip(base, got[:3]):
        assert np.array_equal(a, b)
    tab = psfrec.encircled_energy(np.tile(LBDA6, 8), got[1].reshape(-1, 40, 40), EE_RADII, FRACS)
    ref = psfrec._ee_table(np.tile(LBDA6, 8), got[3], EE_RADII, FRACS)
    for col in tab.colnames:
        assert np.array_equal(tab[col], ref[col]), col


# ---------------------------------------------------------------- 5. refusals
def test_refusals(psfrec):
    from muse_psfr_b200 import _lib
    recs, lgs = group_inputs(psfrec)
    pos = np.ascontiguousarray(POS7[:, :3])
    nl = LBDA6.size
    SENT = 12345.0
    ctx = own_context(psfrec, 8)
    outs = {n: np.full(a.shape, SENT) for n, a in energy_outputs(len(recs), 3, nl, len(GROUPS3), rec=64 + 17).items()}
    img = np.ones((2, 40, 40))
    rec = np.full((2, 64 + 17 + 1), SENT)

    def untouched():
        for n, a in outs.items():
            assert np.all(a == SENT), n
        assert np.all(rec == SENT)

    def fused(nrad, radii, nfrac, fracs):
        rc = ctx._lib.psfr_compute_energy(
            ctx._handle(), 1, len(recs), _lib.ptr(recs), 4, _lib.ptr(np.ascontiguousarray(lgs)), 3, _lib.ptr(pos), nl,
            _lib.ptr(np.ascontiguousarray(LBDA6)), 3, GROUPS3.ctypes.data, nrad, _lib.ptr(radii), nfrac,
            _lib.ptr(fracs), *[_lib.ptr(outs[n]) for n in ('out_cube', 'out_fit', 'out_mean', 'out_mean_fit',
                                                           'out_efit', 'out_mean_efit', 'out_ee', 'out_mean_ee')],
            None)
        untouched()
        return rc

    def alone(nrad, radii, nfrac, fracs, centres=None):
        rc = ctx._lib.psfr_encircled_energy(ctx._handle(), 2, 40, 40, _lib.ptr(img), _lib.ptr(centres), nrad,
                                            _lib.ptr(radii), nfrac, _lib.ptr(fracs), _lib.ptr(rec), None)
        untouched()
        return rc
    good_r, good_f = np.array([1.0, 2.0]), np.array([0.5])
    bad = [(65, np.ones(65), 1, good_f), (2, good_r, 17, np.full(17, 0.5)), (2, np.array([1.0, np.nan]), 1, good_f),
           (2, np.array([-1.0, 2.0]), 1, good_f), (2, np.array([1.0, np.inf]), 1, good_f), (2, good_r, 1, np.zeros(1)),
           (2, good_r, 1, np.ones(1)), (-1, good_r, 1, good_f), (2, None, 1, good_f)]
    try:
        for args in bad:
            assert fused(*args) == _lib.E_ARG, args
            assert alone(*args) == _lib.E_ARG, args
        for c in ([20.0, np.nan, 20.0, 20.0], [np.inf, 20.0, 20.0, 20.0]):
            assert alone(2, good_r, 1, good_f, np.array(c)) == _lib.E_ARG, c
        # the context still works
        r = ee_of(ctx, img, good_r, good_f)
        assert_allclose(r[:, :2], np.pi * good_r[None] ** 2 + 0 * r[:, :2], rtol=1e-13)
    finally:
        ctx.close()


# ---------------------------------------------------------------- 6. the SPARTA shell
def test_sparta_energy(psfrec):
    from muse_psfr_b200 import _fits
    tbl = config2_table()
    plain = psfrec.compute_psf_from_sparta_batch([tbl], lbda=LBDA6, verbose=False, field_positions=GRID3,
                                                 elliptical=True)[0]
    got = psfrec.compute_psf_from_sparta_batch([tbl], lbda=LBDA6, verbose=False, field_positions=GRID3, elliptical=True,
                                               ee_radii=EE_RADII, ee_fractions=FRACS)[0]
    names = ['PRIMARY', 'SPARTA_ATM_DATA', 'FIT_ROWS', 'FIT_MEAN', 'PSF_MEAN', 'FIT_FIELD', 'PSF_FIELD', 'SHAPE_MEAN',
             'SHAPE_FIELD']
    assert [h.name for h in got] == names + ['EE_MEAN', 'EE_FIELD']
    assert_same_result(_fits.HDUList(list(got)[:9]), plain)
    nl = LBDA6.size
    ref_mean = psfrec.encircled_energy(LBDA6, np.ascontiguousarray(got['PSF_MEAN'].data), EE_RADII, FRACS)
    ref_field = psfrec.encircled_energy(np.tile(LBDA6, 9), np.ascontiguousarray(got['PSF_FIELD'].data).reshape(-1, 40, 40),
                                        EE_RADII, FRACS)
    ref_mean = {k: ref_mean[k] for k in ref_mean.colnames}
    ref_field = {k: ref_field[k] for k in ref_field.colnames}
    ref_field['x'] = np.repeat(GRID3[0], nl)
    ref_field['y'] = np.repeat(GRID3[1], nl)

    def check(hdul):
        for name, ref in (('EE_MEAN', ref_mean), ('EE_FIELD', ref_field)):
            tab = hdul[name].data
            assert list(tab.dtype.names) == list(ref), name
            for col, v in ref.items():
                assert np.array_equal(tab[col], v), (name, col)
            for key in ('SEEING', 'GL', 'L0'):
                assert hdul[name].header[key] == got['FIT_MEAN'].header[key]
            assert hdul[name].header['EERAD4'] == EE_RADII[3] and hdul[name].header['EEFRAC3'] == FRACS[2]
    check(got)
    buf = io.BytesIO()
    got.writeto(buf)
    check(_fits.open(buf.getvalue()))
    one = psfrec.compute_psf_from_sparta(tbl, lbda=LBDA6, verbose=False, ee_radii=EE_RADII, ee_fractions=FRACS)
    assert [h.name for h in one] == names[:5] + ['EE_MEAN']
    assert_same_result(_fits.HDUList(list(one)[:5]), _fits.HDUList(list(plain)[:5]))
    for col, v in ref_mean.items():
        assert np.array_equal(one['EE_MEAN'].data[col], v), col

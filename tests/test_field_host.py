"""CPU tests of the field-resolved API: the checks ``compute_psf_field`` and the SPARTA shell make before
any device work, and the 4-D image extension (PSF_FIELD) through the FITS writer and reader."""
import io

import numpy as np
import pytest

from muse_psfr_b200 import _fits, psfrec

LBDA = np.array([500., 700.])


@pytest.mark.parametrize('positions, match', [
    (np.zeros((3, 2)), r'\[2, npos\]'),
    (np.zeros(2), r'\[2, npos\]'),
    (np.zeros((2, 2, 1)), r'\[2, npos\]'),
    (np.zeros((2, 0)), '1 to 256'),
    (np.zeros((2, 257)), '1 to 256'),
    ([[0., np.nan], [0., 0.]], 'finite'),
    ([[0., 1.], [np.inf, 0.]], 'finite'),
])
def test_compute_psf_field_refuses_positions(positions, match):
    with pytest.raises(ValueError, match=match):
        psfrec.compute_psf_field(LBDA, [1.0], [0.7], [25.], positions=positions)


def test_compute_psf_field_refuses_flags_and_draws():
    with pytest.raises(ValueError, match='one flag per draw'):
        psfrec.compute_psf_field(LBDA, [1.0, 0.9], [0.7, 0.6], [25., 20.], three_lgs_mode=[True])
    with pytest.raises(ValueError, match='one entry per draw'):
        psfrec.compute_psf_field(LBDA, [1.0, 0.9], [0.7], [25., 20.])


def test_compute_psf_field_empty():
    fit, cube = psfrec.compute_psf_field(LBDA, [], [], [], positions=[[0., 10.], [0., 5.]])
    assert fit.shape == (0, 2, 2, 16) and cube.shape == (0, 2, 2, 40, 40)
    fit, cube = psfrec.compute_psf_field([], [1.0], [0.7], [25.], want_cube=False)
    assert fit.shape == (1, 9, 0, 16) and cube is None


def test_sparta_refuses_bad_field_positions():
    tbl = psfrec.create_sparta_table(nlines=2)
    with pytest.raises(ValueError, match='finite'):
        psfrec.compute_psf_from_sparta(tbl, field_positions=[[0.], [np.nan]])
    with pytest.raises(ValueError, match=r'\[2, npos\]'):
        psfrec.compute_psf_from_sparta_batch([tbl], field_positions=[0., 1., 2.])


def test_four_dimensional_image_round_trip():
    rng = np.random.default_rng(0)
    psf = rng.random((3, 2, 40, 40))
    cols = {'lbda': np.tile(LBDA, 3), 'x': np.repeat([-30., 0., 12.5], 2), 'y': np.repeat([0., 30., -7.3], 2)}
    hdul = _fits.HDUList([_fits.PrimaryHDU(), _fits.table_to_hdu(cols, meta={'SEEING': 0.8}, name='FIT_FIELD'),
                          _fits.ImageHDU(data=psf, name='PSF_FIELD')])
    buf = io.BytesIO()
    hdul.writeto(buf)
    back = _fits.open(buf.getvalue())
    assert back['PSF_FIELD'].data.shape == (3, 2, 40, 40)
    assert np.array_equal(back['PSF_FIELD'].data, psf)
    for name, ref in cols.items():
        assert np.array_equal(back['FIT_FIELD'].data[name], ref)
    assert back['FIT_FIELD'].header['SEEING'] == 0.8
    try:
        ahdul = _fits.to_astropy(hdul)
    except ImportError:
        return
    assert ahdul['PSF_FIELD'].data.shape == (3, 2, 40, 40)
    assert np.array_equal(ahdul['PSF_FIELD'].data, psf)

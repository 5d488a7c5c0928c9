"""Sensor bands on the CPU: the SRF interpolation helper band_weights, and the numpy statement of the band definition
that the GPU band tests compare against (tests/band_ref.py)."""
import re
from pathlib import Path

import numpy as np
import pytest

import gort_b200
from band_ref import MODIS_EDGES, band_mean, band_scale, close_to_band_mean

ROOT = Path(__file__).resolve().parent.parent
GRID = np.arange(400.0, 2500.0 + 0.5, 1.0)


def test_modis_boxcars_on_the_full_grid():
    w = np.concatenate([gort_b200.band_weights(GRID, [lo, hi], [1.0, 1.0]) for lo, hi in MODIS_EDGES])
    assert w.shape == (7, 2101)
    assert set(np.unique(w)) == {0.0, 1.0}
    assert [int(r.sum()) for r in w] == [51, 36, 21, 21, 21, 25, 51]
    assert int(np.count_nonzero(w.sum(axis=0))) == 226            # the union of the 7 land bands
    lo, hi = MODIS_EDGES[0]
    assert np.array_equal(np.nonzero(w[0])[0], np.arange(int(lo) - 400, int(hi) - 400 + 1))


def test_several_bands_with_a_shared_table():
    x = np.linspace(600.0, 700.0, 11)
    resp = np.stack([np.exp(-0.5 * ((x - 650.0) / 10.0) ** 2), np.ones(11)])
    w = gort_b200.band_weights(GRID, x, resp)
    assert w.shape == (2, 2101)
    # grid points on table nodes take the table's values; the rest interpolate linearly; zero outside the table
    assert np.array_equal(w[0, 200:301:10], resp[0])
    assert w[0, 205] == pytest.approx(0.5 * (resp[0][0] + resp[0][1]), rel=1e-15)
    assert np.all(w[:, :200] == 0.0) and np.all(w[:, 301:] == 0.0)


def test_per_band_tables_and_a_coarse_grid():
    grid = np.arange(400.0, 2500.0 + 0.5, 10.0)
    w = gort_b200.band_weights(grid, [[500.0, 540.0], [800.0, 803.0]], [[1.0, 3.0], [2.0, 2.0]])
    assert np.allclose(w[0, 10:15], [1.0, 1.5, 2.0, 2.5, 3.0], rtol=0, atol=1e-15)
    assert np.count_nonzero(w[0]) == 5
    assert np.count_nonzero(w[1]) == 1 and w[1, 40] == 2.0     # a band narrower than the grid: one column


def test_band_weights_rejects_unordered_tables():
    with pytest.raises(ValueError):
        gort_b200.band_weights(GRID, [650.0, 620.0], [1.0, 1.0])
    with pytest.raises(ValueError):
        gort_b200.band_weights(GRID, [620.0, 650.0, 670.0], [1.0, 1.0])


def test_band_mean_is_the_definition():
    rng = np.random.Generator(np.random.PCG64(7))
    x = rng.uniform(0.0, 1.0, (3, 4, 50))
    w = np.zeros((4, 50))
    w[0, 5:15] = rng.uniform(0.1, 2.0, 10)
    w[1, 0] = 3.0                                       # single column, first column
    w[2, 31:50:2] = 1.0                                 # zero-weight columns inside the band, last column
    w[3, 10:40] = rng.uniform(0.0, 1.0, 30)
    w[3, 20] = 0.0
    got = band_mean(x, w)
    for b in range(4):
        s = [i for i in range(50) if w[b, i] > 0]
        ref = sum(w[b, i] * x[..., i] for i in s) / sum(w[b, i] for i in s)
        assert np.allclose(got[..., b], ref, rtol=1e-14, atol=0)
    assert np.allclose(got[..., 1], x[..., 0], rtol=1e-15, atol=0)
    # raw SRF values: the scale of a row does not matter
    assert np.allclose(band_mean(x, 7.5 * w), got, rtol=1e-14, atol=0)


def test_band_mean_nan_rules():
    x = np.ones((2, 10))
    w = np.zeros((2, 10))
    w[0, 2:6] = 1.0
    w[0, 3] = 0.0
    w[1, 6:9] = 1.0
    x[:, 3] = np.nan             # zero-weight column inside band 0: never read
    x[1, 7] = np.nan             # inside band 1: that band is NaN for that line only
    got = band_mean(x, w)
    assert np.array_equal(got[:, 0], [1.0, 1.0])
    assert got[0, 1] == 1.0 and np.isnan(got[1, 1])
    assert np.array_equal(band_scale(x, w), [[1.0, 1.0], [1.0, 1.0]])
    ok, _ = close_to_band_mean(got, x, w)
    assert ok
    bad = got.copy()
    bad[1, 1] = 1.0
    assert not close_to_band_mean(bad, x, w)[0]


def test_max_bands_matches_the_header():
    text = (ROOT / "include" / "gort_b200.h").read_text()
    assert int(re.search(r"#define GORT_MAX_BANDS (\d+)", text).group(1)) == gort_b200.MAX_BANDS == 64


@pytest.mark.parametrize("shape", [(7,), (7, 2100), (0, 2101), (65, 2101), (2, 7, 2101)])
def test_weights_of_the_wrong_shape_are_refused_before_the_library_reads_them(shape):
    """the library reads B x W doubles: weights built on another grid, or with no or too many bands, raise"""
    from gort_b200.api import _band_weights_arg
    with pytest.raises(ValueError):
        _band_weights_arg(np.ones(shape), 2101)
    w, B = _band_weights_arg(np.ones((7, 2101)), 2101)
    assert B == 7 and w.flags["C_CONTIGUOUS"]

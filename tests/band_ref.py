"""numpy statement of the band definition (include/gort_b200.h, gort_*_band_batch) and the tolerance the band tests use.

For band b with S_b = { i : weights[b][i] > 0 }:  value[b] = sum_{i in S_b} w_i x_i / sum_{i in S_b} w_i.
Columns outside S_b are never read."""
import numpy as np

MODIS_EDGES = [(620.0, 670.0), (841.0, 876.0), (459.0, 479.0), (545.0, 565.0), (1230.0, 1250.0), (1628.0, 1652.0),
               (2105.0, 2155.0)]


def band_mean(x, weights):
    """x [..., W], weights [B][W] -> [..., B]"""
    x = np.asarray(x, dtype=np.float64)
    w = np.asarray(weights, dtype=np.float64)
    out = np.empty(x.shape[:-1] + (w.shape[0],))
    for b in range(w.shape[0]):
        s = np.nonzero(w[b] > 0)[0]
        out[..., b] = (x[..., s] * w[b, s]).sum(axis=-1) / w[b, s].sum()
    return out


def band_scale(x, weights):
    """max_{i in S_b} |x_i| per band, NaN columns ignored -> [..., B]"""
    x = np.abs(np.asarray(x, dtype=np.float64))
    w = np.asarray(weights, dtype=np.float64)
    out = np.zeros(x.shape[:-1] + (w.shape[0],))
    for b in range(w.shape[0]):
        s = np.nonzero(w[b] > 0)[0]
        v = x[..., s]
        out[..., b] = np.max(np.where(np.isnan(v), 0.0, v), axis=-1)
    return out


def close_to_band_mean(got, x, weights, rel=1e-12):
    """(ok, worst ratio): NaN positions equal to those of the definition, |got - ref| <= rel * max_{S_b} |x_i| elsewhere"""
    ref = band_mean(x, weights)
    scale = band_scale(x, weights)
    got = np.asarray(got)
    if got.shape != ref.shape or not np.array_equal(np.isnan(got), np.isnan(ref)):
        return False, np.inf
    fin = ~np.isnan(ref)
    err = np.abs(got[fin] - ref[fin])
    lim = rel * scale[fin] + 1e-300
    worst = float(np.max(err / lim)) if err.size else 0.0
    return bool(np.all(err <= lim)), worst

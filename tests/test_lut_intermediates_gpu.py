"""GPU parity of the gap-probability intermediates the BRDF never reads (SURVEY.md 8f row 1): gortt_calc_vb, gortt_calc_fb,
gortt_calc_t_open, dk_open and k_open[h] (gortt_pn_kopen.c:925-1078, :351-375) against the restatement, which the CPU tests
pin to the compiled reference bit for bit.

fb = (1 - exp(-lv' vb)) / (1 - p_n0) is rounding noise wherever p_n0 rounds to 1 (the reference divides by DBL_MIN * 2 there,
:990) and wherever vb is itself a cancelled ~1e-16 (a sphere centred on the lowest layer touches the h1 plane): those entries
are compared for finiteness only (checkers.check_set).  Everything else: 1e-9, conditioning-aware like the LUT tests."""
import numpy as np
import pytest

from checkers import DEAD_KEYS as KEYS, check_set
from gort_b200 import workloads as wk

pytestmark = pytest.mark.gpu

def test_dead_intermediates_random_structures(gort, oracle):
    rng = np.random.Generator(np.random.PCG64(41))
    st = wk.random_structures(rng, 24)
    got = gort.lut_intermediates(st)
    worst = {k: 0.0 for k in KEYS}
    for m in range(st.shape[1]):
        wm = check_set({k: got[k][m] for k in KEYS}, st[:, m], oracle, "set %d %r" % (m, st[:, m]))
        worst = {k: max(worst[k], wm[k]) for k in KEYS}
    print("dead intermediates, worst rel err per output:", worst)
    # t_open is symmetric with a zero diagonal (:1033-1062)
    assert np.array_equal(got["t_open"], np.swapaxes(got["t_open"], 1, 2))
    assert np.all(np.diagonal(got["t_open"], axis1=1, axis2=2) == 0.0)
    # k_open[0] is the LUT record's openness factor
    lut = gort.lut(st)
    assert np.allclose(got["k_open"][:, 0], lut[:, 182], rtol=1e-13, atol=0)


def test_dead_intermediates_grouping_invariance_and_c5_points(gort, oracle):
    st = wk.c5_lut_grid()["structure"]
    blk = np.ascontiguousarray(st[:, 4096:4096 + 200])          # shares crown shapes: groups and sub-groups
    got = gort.lut_intermediates(blk)
    for k in (0, 7, 8, 63, 64, 65, 199):
        alone = gort.lut_intermediates(np.ascontiguousarray(blk[:, k:k + 1]))
        for q in KEYS:
            assert np.array_equal(alone[q][0], got[q][k], equal_nan=True), "%s of set %d differs when computed alone" % (q, k)
    for k in (0, 77, 199):
        check_set({q: got[q][k] for q in KEYS}, blk[:, k], oracle, "C5 point %d" % (4096 + k))

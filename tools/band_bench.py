"""Sensor-band paths against their per-wavelength counterparts, on one GPU: writes <out>/band_bench.json.

    python tools/band_bench.py <out_dir> [--scale 1.0]

  C4  10^5 members x 16 per-member geometries, 7 MODIS land bands as boxcars on the 1-nm grid (226 union columns):
      gort_forward_band_batch end to end (host arrays in and out), and the same chain of kernels on device tensors timed
      by CUDA events (LUT, spectra on the 226 columns, band kernels) -- against gort_forward_batch on the 226 columns end
      to end, and lut -> spectra -> brdf on the 226 columns -> a torch FP64 weighted reduction on the GPU.  Also the
      band kernels alone with 7, 13 and 36 bands over the same 226 columns.
  C2  the hemispherical sweep (11 664 lines, one set) on the full 2101-column grid: brdf_band_dev with the 7 bands
      against brdf_dev over all 2101 columns.
  C3  10^4 sets x 3 suns: energy_band_dev with the 7 bands on the 226 union columns against energy_dev on the same
      columns.
Every shape is warmed up; each timed window runs at least `--window` seconds.  Inputs are generated (gort_b200.workloads,
boxcar SRFs from the band edges): no SRF table is read.  Needs a CUDA device; there is no CPU path."""
import argparse
import json
import math
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

import torch  # noqa: E402

import gort_b200  # noqa: E402
from gort_b200 import workloads as wk  # noqa: E402
from band_ref import MODIS_EDGES  # noqa: E402

GRID = np.arange(400.0, 2500.5, 1.0)


def modis_weights(grid):
    return np.concatenate([gort_b200.band_weights(grid, [lo, hi], [1.0, 1.0]) for lo, hi in MODIS_EDGES])


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(torch.device("cuda:0"))


def timed(fn, window, stages=1):
    """mean ms per call of fn(ev) over a window of >= `window` s, by CUDA events; fn records ev[1..stages-1] itself
    between its stages -> [total, stage 1, ...]"""
    fn(None)
    fn(None)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn(None)
    torch.cuda.synchronize()
    reps = max(5, math.ceil(window / max(time.perf_counter() - t0, 1e-6)))
    sums = np.zeros(stages + 1)
    for _ in range(reps):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(stages + 1)]
        ev[0].record()
        fn(ev)
        ev[stages].record()
        ev[stages].synchronize()
        sums[0] += ev[0].elapsed_time(ev[stages])
        for k in range(stages):
            sums[1 + k] += ev[k].elapsed_time(ev[k + 1])
    return [float(v / reps) for v in sums] if stages > 1 else [float(sums[0] / reps)], reps


def wall(fn, window):
    """mean ms of a host call that returns synchronised"""
    fn()
    fn()
    t0 = time.perf_counter()
    fn()
    one = time.perf_counter() - t0
    reps = max(3, math.ceil(window / max(one, 1e-6)))
    t0 = time.perf_counter()
    for _ in range(reps):
        fn()
    return (time.perf_counter() - t0) * 1e3 / reps, reps


def device_info():
    info = {"torch_name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        info["nvidia_smi"] = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else q.stderr.strip()
    except (OSError, subprocess.TimeoutExpired) as e:
        info["nvidia_smi"] = "unavailable: %s" % e
    return info


def rates(ms, evals, bytes_written):
    return {"ms": ms, "represented_evals_per_s": evals / (ms * 1e-3), "bytes_written": int(bytes_written),
            "write_GB_per_s": bytes_written / (ms * 1e-3) / 1e9}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out")
    ap.add_argument("--scale", type=float, default=1.0, help="fraction of the C4 members and C3 sets (rehearsals)")
    ap.add_argument("--window", type=float, default=0.5, help="seconds per timed window")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("band_bench: no CUDA device (there is no CPU path)")
    out = Path(args.out)
    out.mkdir(parents=True, exist_ok=True)
    g = gort_b200.Gort(0)
    # every tensor, library call, reduction and event on one created stream (the legacy default stream's handle is 0,
    # which the library would read as "the context's own stream")
    stream = torch.cuda.Stream()
    s = lambda: stream.cuda_stream
    with torch.cuda.stream(stream):
        res = measure(g, args, s)
    g.close()
    text = json.dumps(res, indent=1)
    (out / "band_bench.json").write_text(text + "\n")
    print(text)


def measure(g, args, s):
    w_full = modis_weights(GRID)
    cols = np.nonzero(w_full.sum(axis=0) > 0)[0]
    U, B = len(cols), w_full.shape[0]
    wl_u, w_u = GRID[cols], np.ascontiguousarray(w_full[:, cols])
    support = int(np.count_nonzero(w_full > 0))             # sum_b |S_b|
    res = {"device": device_info(), "bands": "7 MODIS land bands, boxcars %s nm" % MODIS_EDGES,
           "union_columns": U, "sum_support_columns": support, "window_s": args.window}

    # ---- C4 --------------------------------------------------------------------------------------------------------
    M = max(1, int(round(100000 * args.scale)))
    x = wk.c4_enkf(n_members=M)
    st, leaf, soil, ang = x["structure"], x["leaf"], x["soil"], x["angles"]
    G = ang.shape[-1]
    c4 = {"members": M, "geometries": G}
    ms, reps = wall(lambda: g.forward_band(st, leaf, soil, GRID, w_full, ang), args.window)
    c4["forward_band_end_to_end"] = dict(rates(ms, M * G * support, M * G * B * 8), reps=reps,
                                         note="host arrays in and out, full 2101-column grid passed")
    rs_host = np.empty((M, G, U))
    ms, reps = wall(lambda: g.forward(st, leaf, soil, wl_u, ang, out=rs_host), args.window)
    c4["forward_union_end_to_end"] = dict(rates(ms, M * G * U, M * G * U * 8), reps=reps,
                                          note="gort_forward_batch on the 226 union columns into pageable host memory; "
                                               "no reduction")
    del rs_host
    d_st, d_leaf, d_soil, d_ang, d_wl, d_w = (dev(a) for a in (st, leaf, soil, ang, wl_u, w_u))
    d_wn = dev(w_u / w_u.sum(axis=1, keepdims=True))
    lut = torch.empty((M, gort_b200.LUT_STRIDE), dtype=torch.float64, device="cuda:0")
    sp = [torch.empty((M, U), dtype=torch.float64, device="cuda:0") for _ in range(3)]
    rb = torch.empty((M, G, B), dtype=torch.float64, device="cuda:0")

    def band_chain(ev):
        g.lut_dev(d_st, lut, stream=s())
        if ev: ev[1].record()
        g.spectra_dev(d_leaf, d_soil, d_wl, *sp, stream=s())
        if ev: ev[2].record()
        g.brdf_band_dev(d_st, lut, d_ang, *sp, d_w, rb, stream=s())

    (tot, t_lut, t_sp, t_band), reps = timed(band_chain, args.window, stages=3)
    c4["band_kernels"] = dict(rates(tot, M * G * support, M * G * B * 8), reps=reps, lut_ms=t_lut, spectra_ms=t_sp,
                              band_ms=t_band, lut_share=t_lut / tot)
    # the band kernels alone for more bands on the same 226 columns (13 and 36: as many as Sentinel-2 and MODIS have),
    # each band a contiguous share of the columns
    c4["band_kernel_vs_band_count"] = {}
    for nb in (B, 13, 36):
        wn = np.zeros((nb, U))
        for b, part in enumerate(np.array_split(np.arange(U), nb)):
            wn[b, part] = 1.0
        d_wnb = dev(wn)
        rbn = torch.empty((M, G, nb), dtype=torch.float64, device="cuda:0")
        (ms,), reps = timed(lambda ev: g.brdf_band_dev(d_st, lut, d_ang, *sp, d_wnb, rbn, stream=s()), args.window)
        c4["band_kernel_vs_band_count"][str(nb)] = dict(rates(ms, M * G * U, M * G * nb * 8), reps=reps,
                                                        note="geometry + band kernels; LUT and spectra not included")
        del rbn
    rsurf = torch.empty((M, G, U), dtype=torch.float64, device="cuda:0")

    def wl_chain(ev):
        g.lut_dev(d_st, lut, stream=s())
        if ev: ev[1].record()
        g.spectra_dev(d_leaf, d_soil, d_wl, *sp, stream=s())
        if ev: ev[2].record()
        g.brdf_dev(d_st, lut, d_ang, *sp, rsurf, stream=s())
        if ev: ev[3].record()
        torch.matmul(rsurf.view(M * G, U), d_wn.T, out=rb.view(M * G, B))

    (tot, t_lut, t_sp, t_brdf, t_red), reps = timed(wl_chain, args.window, stages=4)
    c4["per_wavelength_kernels_then_torch_reduction"] = dict(
        rates(tot, M * G * U, M * G * U * 8 + M * G * B * 8), reps=reps, lut_ms=t_lut, spectra_ms=t_sp, brdf_ms=t_brdf,
        reduction_ms=t_red)
    res["c4"] = c4
    del rsurf, lut, sp, rb
    torch.cuda.empty_cache()

    # ---- C2 --------------------------------------------------------------------------------------------------------
    x = wk.c2_hemisphere()
    st2 = x["structure"]
    lut2 = g.lut(st2)
    rl, tl, rsl = g.spectra(x["leaf"], x["soil"], GRID)
    L2 = x["angles"].shape[1]
    d2 = [dev(a) for a in (st2, lut2, x["angles"], rl[0], tl[0], rsl[0])]
    d_wf = dev(w_full)
    rb2 = torch.empty((1, L2, B), dtype=torch.float64, device="cuda:0")
    rs2 = torch.empty((1, L2, GRID.size), dtype=torch.float64, device="cuda:0")
    (ms,), reps = timed(lambda ev: g.brdf_band_dev(*d2, d_wf, rb2, stream=s()), args.window)
    c2 = {"lines": L2, "grid_columns": int(GRID.size)}
    c2["brdf_band_dev"] = dict(rates(ms, L2 * support, L2 * B * 8), reps=reps)
    (ms,), reps = timed(lambda ev: g.brdf_dev(*d2, rs2, stream=s()), args.window)
    c2["brdf_dev_all_columns"] = dict(rates(ms, L2 * GRID.size, L2 * GRID.size * 8), reps=reps)
    res["c2"] = c2
    del rs2

    # ---- C3 --------------------------------------------------------------------------------------------------------
    n3 = max(1, int(round(10000 * args.scale)))
    x = wk.c3_albedo(n_sets=n3)
    st3 = x["structure"]
    lut3 = g.lut(st3)
    sp3 = g.spectra(x["leaf"], x["soil"], wl_u)
    G3 = x["angles"].shape[1]
    d3 = [dev(a) for a in (st3, lut3, x["angles"])] + [dev(a) for a in sp3]
    eb = [torch.empty((n3, G3, B), dtype=torch.float64, device="cuda:0") for _ in range(3)]
    ew = [torch.empty((n3, G3, U), dtype=torch.float64, device="cuda:0") for _ in range(3)]
    c3 = {"sets": n3, "suns": G3}
    (ms,), reps = timed(lambda ev: g.energy_band_dev(*d3, d_w, *eb, stream=s()), args.window)
    c3["energy_band_dev"] = dict(rates(ms, n3 * G3 * support, 3 * n3 * G3 * B * 8), reps=reps)
    (ms,), reps = timed(lambda ev: g.energy_dev(*d3, *ew, stream=s()), args.window)
    c3["energy_dev_union_columns"] = dict(rates(ms, n3 * G3 * U, 3 * n3 * G3 * U * 8), reps=reps)
    res["c3"] = c3
    return res


if __name__ == "__main__":
    main()

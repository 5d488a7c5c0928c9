"""The exact favd / LAI tangent against the central-difference Jacobian, on one GPU: writes <out>/tangent_bench.json.

    python tools/tangent_bench.py <out_dir> [--scale 1.0] [--window 1.0]

  C4b  10^5 members, every parameter varying, 16 per-member geometries, 7 MODIS bands: wall time of
       gort_lai_tangent_batch(GORT_JAC_LAI) with rsurf against gort_jacobian_batch(GORT_JAC_LAI) with rsurf (host arrays
       in and out, both return synchronised), alternated after warm-up.
  C2   one forest, 11 664 lines x 2101 wavelengths on device tensors: brdf_tangent_dev against brdf_dev, whole calls by
       CUDA events, and per kernel (rsurf_tangent_kernel against rsurf_wide_kernel, and the geometry kernels) from
       torch.profiler in a separate pass.  Both per-wavelength kernels write 196 MB; their rates are given as fractions
       of the data-sheet 7.7 TB/s HBM bandwidth of a B200.
The GPU's name and power limit are recorded beside the numbers.  Needs a CUDA device; there is no CPU path."""
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

import torch  # noqa: E402

import gort_b200  # noqa: E402
from gort_b200 import workloads as wk  # noqa: E402

HBM_PEAK = 7.7e12      # B/s, data sheet, one B200


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(torch.device("cuda:0"))


def device_info():
    info = {"torch_name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        info["nvidia_smi"] = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else q.stderr.strip()
    except (OSError, subprocess.TimeoutExpired) as e:
        info["nvidia_smi"] = "unavailable: %s" % e
    return info


def alternated(fns, window):
    """mean and min ms of host calls that return synchronised, the calls of fns alternated -> {name: {...}}"""
    for f in fns.values():
        f()
        f()
    t0 = time.perf_counter()
    for f in fns.values():
        f()
    reps = max(3, math.ceil(window / max(time.perf_counter() - t0, 1e-6)))
    ts = {k: [] for k in fns}
    for _ in range(reps):
        for k, f in fns.items():
            t = time.perf_counter()
            f()
            ts[k].append((time.perf_counter() - t) * 1e3)
    return {k: {"mean_ms": float(np.mean(v)), "min_ms": float(np.min(v)), "reps": reps} for k, v in ts.items()}


def events(fn, window):
    """mean ms per call by CUDA events on the current stream"""
    fn()
    fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    reps = max(10, math.ceil(window / max(time.perf_counter() - t0, 1e-6)))
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps, reps


def kernel_ms(fn, reps=20):
    """mean device ms per call of every kernel fn launches, from torch.profiler"""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        if e.device_type is not None and "CUDA" in str(e.device_type) and e.count > 0:
            t = getattr(e, "device_time_total", None)
            if t is None:
                t = e.cuda_time_total
            out[e.key] = t / 1e3 / reps
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out")
    ap.add_argument("--scale", type=float, default=1.0, help="fraction of the C4b members (rehearsals)")
    ap.add_argument("--window", type=float, default=1.0, help="seconds per timed window")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("tangent_bench: no CUDA device (there is no CPU path)")
    out = Path(args.out)
    out.mkdir(parents=True, exist_ok=True)
    g = gort_b200.Gort(0)
    res = {"device": device_info()}

    # ---- C4b ----
    M = max(1, int(round(1e5 * args.scale)))
    w = wk.c4_enkf(n_members=M, seed=1002)
    a = (w["structure"], w["leaf"], w["soil"], w["wavelength"], w["angles"])
    LAI = gort_b200.JAC_LAI
    t = alternated({"lai_tangent": lambda: g.lai_tangent(*a, param=LAI, want_rsurf=True),
                    "jacobian_central_difference": lambda: g.jacobian(*a, param=LAI, want_rsurf=True)}, args.window)
    jt, rt = g.lai_tangent(*a, param=LAI, want_rsurf=True)
    jc, rc = g.jacobian(*a, param=LAI, want_rsurf=True)
    ok = np.isfinite(jc).all(axis=(1, 2)) & np.isfinite(jt).all(axis=(1, 2))
    scale = np.max(np.abs(jc[ok]), axis=(1, 2), keepdims=True)
    res["c4b"] = {"members": M, "geometries": int(w["angles"].shape[-1]), "bands": int(w["wavelength"].size), "wall": t,
                  "speedup_mean": t["jacobian_central_difference"]["mean_ms"] / t["lai_tangent"]["mean_ms"],
                  "rsurf_bit_identical": bool(np.array_equal(rt, rc, equal_nan=True)),
                  "max_abs_diff_over_member_max": float(np.max(np.abs(jc[ok] - jt[ok]) / scale)),
                  "finite_members": int(ok.sum())}

    # ---- C2 ----
    w = wk.c2_hemisphere()
    st, ang, wl = w["structure"], w["angles"], w["wavelength"]
    lut = torch.empty((1, gort_b200.LUT_STRIDE), dtype=torch.float64, device="cuda:0")
    dlut = torch.empty_like(lut)
    d_st = dev(st)
    g.lut_tangent_dev(d_st, lut, dlut)
    rl, tl, rs = g.spectra(w["leaf"], w["soil"], wl)
    ins = [dev(x) for x in (ang, rl[0], tl[0], rs[0])]
    G, W = ang.shape[1], wl.size
    X = torch.empty((1, G, W), dtype=torch.float64, device="cuda:0")
    T = torch.empty_like(X)
    g.synchronize()
    stream = torch.cuda.current_stream().cuda_stream
    fwd = lambda: g.brdf_dev(d_st, lut, *ins, X, stream=stream)
    tan = lambda: g.brdf_tangent_dev(d_st, lut, dlut, *ins, T, stream=stream)
    byt = G * W * 8
    calls = {}
    for name, f in (("brdf_dev", fwd), ("brdf_tangent_dev", tan)):
        ms, reps = events(f, args.window)
        calls[name] = {"ms": ms, "reps": reps}
    ks = {}
    for name, f in (("brdf_dev", fwd), ("brdf_tangent_dev", tan)):
        ks[name] = kernel_ms(f)
    per_wl = {}
    for name, key in (("rsurf_wide_kernel", "rsurf_wide_kernel"), ("rsurf_tangent_kernel", "rsurf_tangent_kernel")):
        src = ks["brdf_dev"] if key == "rsurf_wide_kernel" else ks["brdf_tangent_dev"]
        ms = sum(v for k, v in src.items() if key in k)
        per_wl[name] = {"ms": ms, "bytes_written": byt,
                        "fraction_of_hbm_datasheet": (byt / HBM_PEAK) / (ms * 1e-3) if ms > 0 else None}
    res["c2"] = {"lines": G, "wavelengths": W, "calls_by_events": calls, "kernels_by_profiler_ms": ks,
                 "per_wavelength_kernels": per_wl}
    g.close()
    text = json.dumps(res, indent=1)
    (out / "tangent_bench.json").write_text(text + "\n")
    print(text)


if __name__ == "__main__":
    main()

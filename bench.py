#!/usr/bin/env python3
"""bench.py -- BRDF evaluations/s of the GORT hot path on N B200s (BASELINE.json metric).

Workload (config.workload = "c2"): BASELINE.json configs[1], the hemispherical BRDF sweep --
18 view zeniths x 18 sun zeniths x 36 azimuths = 11 664 input lines x 2101 wavelengths
(400-2500 nm at 1 nm), one forest (LAI 4) per GPU = 24 506 064 evaluations per GPU per step.
One evaluation = one iteration of the reference's wavelength loop (gortt.c:460-567).  With N > 1 every
rank owns its own forest's sweep (weak scaling, no data-path collective: SURVEY.md 8e).

A step = one pass of the hot path (gort_brdf_batch: angle preparation, viewed proportions, hotspot,
per-wavelength loop) over the whole sweep.  The gap-probability LUT and the PROSPECT-D / Price spectra
are computed once on the GPU during set-up, exactly as the reference computes them once per run
(gortt.c:108-120, :224-227) and as the CPU baseline receives them.

    value     device-resident: inputs already in HBM, K back-to-back gort_brdf_batch_dev calls in the library's
              overlap mode (gort_set_overlap, include/gort_b200.h), CUDA events on the launching stream around
              the K steps, max over ranks.
    e2e       the same K steps through the host-pointer C ABI call gort_brdf_batch: pinned host buffers,
              H2D of all inputs and D2H of rsurf inside the timed region; next to it the rate of a plain pinned
              cudaMemcpyAsync of the same 196 MB measured in the same run (alone, and on all ranks at once): the
              ceiling of that leg.
    roofline  the dominant kernel (rsurf_wide_kernel), bound = hbm (8 B written per evaluation).  achieved / frac
              come from the KERNEL'S OWN duration: a second pass of the K steps with CUDA events around each kernel
              (gort_profile_begin/end; overlap and programmatic dependent launch off).  The repeated-call figure
              (bytes per step / time per step of the overlapped timed region, in which the geometry kernel hides
              under the previous step's stores) is reported next to it as achieved_repeated / frac_repeated.
    cpu_baseline  the unmodified reference compiled into oracle/_ref (kind "reference"; the oracle
              restatement, kind "port", if _ref did not travel), in-process, one process per host
              core, on a bounded sample of the same sweep.
    extras    N = 1: device times of the other kernels on C3 / C4 / C5 at full size, the sweep with shuffled lines and
              with component signatures, the C4 member update end to end through the host API, and the parity audit
              (tests/parity_audit.py: worst relative error per output and band against the compiled reference).
              N > 1: LUT generation for the C5 grid sharded over the ranks with its NCCL all-gather, and the sweep
              of ONE forest split by geometry blocks (strong scaling).

--impl reference times only the CPU arm, on all host cores, and prints the same JSON line shape.
Timed outputs are 196 MB per step (> the 126 MB L2), so every step streams to HBM; no explicit flush.

--dump-outputs DIR writes what the timed steps computed, so that two builds can be compared output for output on
identical inputs: DIR/rsurf.npy, the result rows of the last device-resident step, and DIR/rsurf_e2e.npy, those of
the last host-pointer step, each for the same fixed, seeded sample of 1536 of the 11 664 lines (all 2101 bands,
float64, 26 MB), and DIR/rsurf_lines.npy, the indices of those lines.  Rank 0's forest only.
"""
import argparse
import json
import os
import re
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

# the tree may be read-only and stays as the build left it: no __pycache__ from the project imports below
sys.dont_write_bytecode = True
ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

METRIC = "BRDF evals/sec (geom x lambda x member)"
UNIT = "evals/s"
F_LAMBDA = 92.0          # algorithmic FP64 ops per evaluation (SURVEY.md App. D)
F_GEOM = 350.0           # per (line, set)
F_LUT = 2.5e6            # per parameter set, outputs-only algorithm (SURVEY.md 8d)
DUMP_LINES = 1536        # lines of the sweep in --dump-outputs: 2 x 1536 x 2101 doubles = 52 MB, under 64 MB
DUMP_SEED = 2101


def load_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for k, nm in enumerate(names):
                if f[5 + k].lower().startswith("active"):
                    reasons.add(nm)
        sm_sorted = sorted(sm)
        # median of the upper half = clocks while the GPU was busy (idle samples drag a plain median down)
        busy = sm_sorted[len(sm_sorted) // 2:] if sm_sorted else []
        return {"sm_mhz": (busy[len(busy) // 2] if busy else None), "sm_max_mhz": (max(mx) if mx else None),
                "samples": len(sm), "reasons": sorted(reasons)}


def _cpus_from_list(text):
    cpus = set()
    for part in text.strip().split(","):
        if not part:
            continue
        lo, _, hi = part.partition("-")
        cpus.update(range(int(lo), int(hi or lo) + 1))
    return cpus


def bind_near_gpu(torch, local_rank):
    """Pin this process to the CPUs next to the GPU before any pinned host buffer is allocated: the e2e leg
    is PCIe-bound (196 MB of D2H per step) and a buffer on the far socket costs ~20 % of the link rate.
    The GPU's NUMA node from sysfs; where the box does not expose one (-1), the "CPU Affinity" column of
    `nvidia-smi topo -m`.  Best effort; returns a description for the JSON line."""
    info = {"gpu_node": None, "bound": False, "source": None}
    try:
        p = torch.cuda.get_device_properties(local_rank)
        bdf = "%04x:%02x:%02x.0" % (p.pci_domain_id, p.pci_bus_id, p.pci_device_id)
        cpus = set()
        try:
            node = int(Path("/sys/bus/pci/devices/%s/numa_node" % bdf).read_text().strip())
            info["gpu_node"] = node
            if node >= 0:
                cpus = _cpus_from_list(Path("/sys/devices/system/node/node%d/cpulist" % node).read_text())
                info["source"] = "sysfs numa_node"
        except OSError:
            pass
        if not cpus:
            out = subprocess.run(["nvidia-smi", "topo", "-m"], capture_output=True, text=True, timeout=20).stdout
            lines = [ln for ln in out.splitlines() if ln.strip()]
            head = next((ln for ln in lines if "CPU Affinity" in ln), None)
            row = next((ln for ln in lines if ln.split()[0] == "GPU%d" % local_rank), None)
            if head and row:
                # GPUi, then one link token per GPU / NIC column (X, NV#, SYS, NODE, PHB, PXB, PIX), then the CPU affinity
                toks = row.split()[1:]
                while toks and (toks[0] in ("X", "SYS", "NODE", "PHB", "PXB", "PIX") or toks[0].startswith("NV")):
                    toks = toks[1:]
                if toks and re.fullmatch(r"\d+(-\d+)?(,\d+(-\d+)?)*", toks[0]):
                    cpus = _cpus_from_list(toks[0])
                    info["source"] = "nvidia-smi topo -m"
        cpus &= os.sched_getaffinity(0)
        if len(cpus) >= 2:                       # never squeeze the process onto a single core
            os.sched_setaffinity(0, cpus)
            info["bound"] = True
            info["cpus"] = len(cpus)
    except Exception as e:                      # noqa: BLE001 -- placement is best effort, never the bench's failure
        info["error"] = str(e)[:80]
    return info


def probe_host_placement(gort_b200, torch, dev, ts, barrier, rank):
    """Which CPUs should this rank pin its host buffers from?  All ranks copy 64 MB device-to-host AT THE SAME TIME into
    buffers pinned from each of 8 groups of the allowed CPUs (a placement only shows its cost under that concurrency: see
    include/gort_b200.h); each rank keeps the group that gave it the best rate (ties: the lowest CPUs)."""
    cpus = sorted(os.sched_getaffinity(0))
    if len(cpus) < 4:
        return None, {"groups": 0, "note": "fewer than 4 cpus: nothing to choose"}
    ng = 8 if len(cpus) >= 16 else 4
    groups = [cpus[k * len(cpus) // ng:(k + 1) * len(cpus) // ng] for k in range(ng)]
    n = (64 << 20) // 8
    src = torch.empty(n, dtype=torch.float64, device=dev)
    rates = []
    with torch.cuda.stream(ts):
        for grp in groups:
            h = gort_b200.PinnedArray((n,), cpus=grp)
            ht = torch.from_numpy(h.array)
            best = 1e30
            for k in range(4):
                barrier()
                a = torch.cuda.Event(enable_timing=True); b = torch.cuda.Event(enable_timing=True)
                a.record(ts); ht.copy_(src, non_blocking=True); b.record(ts); b.synchronize()
                if k:
                    best = min(best, a.elapsed_time(b))
            rates.append(n * 8 / (best * 1e-3) / 1e9)
            del ht
            h.free()
    pick = 0
    for k in range(1, ng):
        if rates[k] > rates[pick] * 1.03:
            pick = k
    return groups[pick], {"groups": ng, "gbs_per_group_rank0": [round(r, 1) for r in rates] if rank == 0 else None,
                          "picked_cpus": "%d-%d" % (groups[pick][0], groups[pick][-1]),
                          "how": "all ranks copying 64 MB device-to-host at once into buffers pinned from each group"}


def dump_lines(G):
    """the fixed, seeded sample of sweep lines that --dump-outputs writes (sorted line indices)"""
    rng = np.random.Generator(np.random.PCG64(DUMP_SEED))
    return np.sort(rng.choice(G, size=min(G, DUMP_LINES), replace=False))


def dump_outputs(out_dir, arrays):
    """arrays {name: array} -> out_dir/<name>.npy, float64"""
    arrays = {k: np.ascontiguousarray(v, dtype=np.float64) for k, v in arrays.items()}
    assert sum(a.nbytes for a in arrays.values()) <= 64 << 20
    out_dir = Path(out_dir)
    out_dir.mkdir(parents=True, exist_ok=True)
    for name, a in arrays.items():
        np.save(out_dir / (name + ".npy"), a)


def sweep_inputs(rank):
    from gort_b200 import workloads as wk
    w = wk.c2_hemisphere(sets=1, lai0=4.0 + 0.25 * rank)
    return w


# ------------------------------------------------------------------------------------------------
# CPU arm (reference compiled into oracle/_ref, else the oracle port)
# ------------------------------------------------------------------------------------------------
def _cpu_worker(args):
    kind, st, lut, ang, rl, tl, rs, reps = args
    import checkers
    chk = checkers.ref() if kind == "reference" else checkers.ref_makefile_flags() if kind == "reference-g" else checkers.oracle()
    t0 = time.perf_counter()
    n = chk.brdf_repeat(st, lut, ang, rl, tl, rs, reps)
    return n, time.perf_counter() - t0


def cpu_arm_setup():
    import checkers
    kind = "reference" if checkers.ref() is not None else "port"
    chk = checkers.ref() if kind == "reference" else checkers.oracle()
    w = sweep_inputs(0)
    st = w["structure"][:, 0].copy()
    lut = chk.lut(st)
    rl, tl, rs = chk.spectra(w["leaf"][:, 0], w["soil"][:, 0], w["wavelength"])
    return kind, st, lut, w["angles"], rl, tl, rs


def cpu_arm_step(pool, cores, kind, st, lut, ang, rl, tl, rs, lines_per_core, reps=1):
    """One bounded sample: every core evaluates `lines_per_core` lines (a strided slice of the sweep,
    all 2101 bands) `reps` times.  Returns (evaluations, wall seconds)."""
    jobs = []
    G = ang.shape[1]
    for c in range(cores):
        idx = (np.arange(lines_per_core) * 37 + c * 101) % G       # spread over the whole hemisphere
        jobs.append((kind, st, lut, np.ascontiguousarray(ang[:, idx].T), rl, tl, rs, reps))
    t0 = time.perf_counter()
    res = pool.map(_cpu_worker, jobs)
    wall = time.perf_counter() - t0
    return sum(r[0] for r in res), wall


def run_reference_arm(args, rank, world):
    """--impl reference: the reference's own CPU implementation on all host cores."""
    if rank != 0:
        return
    import multiprocessing as mp
    cores = os.cpu_count() or 1
    kind, st, lut, ang, rl, tl, rs = cpu_arm_setup()
    lines = 96          # x 2101 bands = 2.0e5 evaluations per core per step, ~0.3-0.8 s of CPU work
    with mp.get_context("fork").Pool(cores) as pool:
        for _ in range(args.warmup):
            cpu_arm_step(pool, cores, kind, st, lut, ang, rl, tl, rs, lines)
        n_tot, t_tot = 0, 0.0
        for _ in range(args.steps):
            n, t = cpu_arm_step(pool, cores, kind, st, lut, ang, rl, tl, rs, lines)
            n_tot += n; t_tot += t
    v = n_tot / t_tot
    sample = "%d lines x 2101 bands per core per step (strided slice of the c2 sweep), %d cores" % (lines, cores)
    out = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * t_tot / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "c2", "lines": 11664, "wavelengths": 2101, "sets_per_gpu": 1,
                   "note": "CPU arm: bounded sample of the same sweep, LUT and spectra given"},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out), flush=True)


# ------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the C3 / C4 / C5 kernel measurements")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write a fixed sample of the last timed step's rsurf to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    import gort_b200

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the GORT path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    all_cpus = os.sched_getaffinity(0)
    numa = bind_near_gpu(torch, local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    g = gort_b200.Gort(local_rank)
    w = sweep_inputs(rank)
    st, ang, wl = w["structure"], w["angles"], w["wavelength"]
    G, W = ang.shape[1], wl.shape[0]
    evals_per_rank = G * W

    # ---- set-up on the GPU (not timed): LUT + spectra, as the reference does once per run ----
    lut = g.lut(st)
    rl, tl, rs = g.spectra(w["leaf"], w["soil"], wl)
    rl, tl, rs = rl[0].copy(), tl[0].copy(), rs[0].copy()

    T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    d_st, d_lut, d_ang, d_rl, d_tl, d_rs = T(st), T(lut), T(ang), T(rl), T(tl), T(rs)
    pitch = ((W + 15) // 16) * 16          # device rows padded to 128 B: every warp store is sector-aligned
    d_out = torch.empty((1, G, pitch), dtype=torch.float64, device=dev)
    # the launching stream: a torch stream whose handle is passed through the C ABI, so that the
    # torch CUDA events below are recorded on the very stream the kernels run on
    ts = torch.cuda.Stream(device=dev)
    stream = ts.cuda_stream
    assert stream != 0

    step_dev = g.brdf_dev_bind(d_st, d_lut, d_ang, d_rl, d_tl, d_rs, d_out, stream=stream)
    # the K timed steps are back-to-back calls of the same shape into the same buffer: the library's documented
    # overlap mode (include/gort_b200.h) lets the geometry kernel of step i+1 run under the stores of step i
    g.set_overlap(True)

    # ---- device-resident timing ----
    for _ in range(args.warmup):
        step_dev()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.25)
    l0 = g.launch_count()
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record(ts)
    h0 = time.perf_counter()
    for _ in range(args.steps):
        step_dev()
    host_enqueue_ms = (time.perf_counter() - h0) * 1e3 / args.steps
    e1.record(ts)
    barrier()
    ms_total = e0.elapsed_time(e1)
    launches = g.launch_count() - l0
    # the rows the last timed step stored, read before anything else writes d_out (the barrier above synchronised)
    lines = dump_lines(G)
    rsurf_dev = d_out[0].index_select(0, torch.from_numpy(lines).to(dev))[:, :W].cpu().numpy() if args.dump_outputs and rank == 0 else None
    # per-kernel durations: the same K steps again, this time with CUDA events recorded on the launching
    # stream around each kernel (gort_profile_begin/end).  Kept out of the timed region above because an
    # event between the two launches of a step would defeat their programmatic-dependent-launch overlap.
    g.profile_begin(args.steps)
    for _ in range(args.steps):
        step_dev()
    barrier()
    geom_ms, rsurf_ms, nprof = g.profile_end()
    # the same launch seen from inside: %globaltimer stamps of every CTA (a few isolated calls, stream order)
    g.kernel_stamps_enable(True)
    spans = []
    for _ in range(5):
        step_dev(); ts.synchronize()
        spans.append(g.kernel_stamps())
    g.kernel_stamps_enable(False)
    stamps = sorted(spans, key=lambda d: d["span_us"])[len(spans) // 2]
    for _ in range(3):          # re-establish the steady state of the overlap mode for anything that follows
        step_dev()
    ts.synchronize()

    # ---- end-to-end through the host-pointer C ABI (pinned host buffers, copies inside) ----
    g.set_overlap(False)
    near_cpus, placement = probe_host_placement(gort_b200, torch, dev, ts, barrier, rank)
    pin = lambda a: _pinned_copy(gort_b200, a, near_cpus)
    h_st, h_lut, h_ang, h_rl, h_tl, h_rs = pin(st), pin(lut), pin(ang), pin(rl), pin(tl), pin(rs)
    h_out = gort_b200.PinnedArray((1, G, W), cpus=near_cpus)      # pinned from the CPUs the probe picked
    for _ in range(args.warmup):
        g.brdf(h_st.array, h_lut.array, h_ang.array, h_rl.array, h_tl.array, h_rs.array, out=h_out.array)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        g.brdf(h_st.array, h_lut.array, h_ang.array, h_rl.array, h_tl.array, h_rs.array, out=h_out.array)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    barrier()
    clocks = sampler.stop() if rank == 0 else None       # sampled over both timed regions (device-resident and e2e)
    checksum = float(h_out.array[0, ::997, ::211].sum())
    rsurf_e2e = h_out.array[0].copy()                    # the result of the e2e leg (the copy test below reuses the buffer)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"rsurf": rsurf_dev, "rsurf_e2e": rsurf_e2e[lines], "rsurf_lines": lines})

    # ---- the ceiling of the e2e leg: a plain pinned D2H copy of the same 196 MB, all ranks at once ----
    d2h_ms = _plain_d2h_ms(torch, dev, ts, d_out, h_out.array, barrier)

    # ---- max over ranks ----
    tt = torch.tensor([ms_total, e2e_s * 1e3, rsurf_ms, geom_ms, d2h_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    ms_total, e2e_ms, rsurf_ms, geom_ms, d2h_ms = [float(x) for x in tt.tolist()]

    multi = multi_gpu_extras(g, torch, dist, dev, ts, rank, world, args) if world > 1 and not args.no_extras else None

    if rank == 0:
        ms_per_step = ms_total / args.steps
        value = world * evals_per_rank / (ms_per_step * 1e-3)
        e2e_step_ms = e2e_ms / args.steps
        e2e_value = world * evals_per_rank / (e2e_step_ms * 1e-3)
        hbm_peak, peak_src = load_peaks()
        alg_bytes = 8.0 * evals_per_rank                      # rsurf only; inputs amortise to < 0.1 B/eval
        # roofline of the dominant kernel from ITS OWN duration (events around each kernel, overlap off).  The repeated-call
        # figure divides by the step time of the overlapped timed region instead: there the geometry kernel of step
        # i+1 runs under the stores of step i and a launch's own duration is not separable.
        achieved = alg_bytes / (rsurf_ms * 1e-3) / 1e9
        achieved_rep = alg_bytes / (ms_per_step * 1e-3) / 1e9
        d2h_bytes = 8 * evals_per_rank
        d2h_gbs = d2h_bytes / (d2h_ms * 1e-3) / 1e9
        h2d = 8 * (st.size + lut.size + ang.size + rl.size + tl.size + rs.size)
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "c2", "lines": G, "wavelengths": W, "sets_per_gpu": 1,
                       "evals_per_gpu_per_step": evals_per_rank,
                       "device_row_pitch_doubles": pitch,
                       "line_order": "azimuth fastest: 36 consecutive lines share the sun (extras.c2_shuffled: every line a new sun)",
                       "mode": "gort_set_overlap(1): consecutive same-shape calls overlap on the GPU",
                       "l2": "outputs are 196 MB per step (> 126 MB L2); no explicit flush",
                       "setup_not_timed": "gap-probability LUT + PROSPECT-D/Price spectra, computed once on the GPU"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d),
                    "d2h_bytes_per_step": int(d2h_bytes), "ms_per_step": e2e_step_ms,
                    "plain_pinned_d2h_ms": d2h_ms, "plain_pinned_d2h_gbs_per_gpu": d2h_gbs,
                    "frac_of_d2h_peak": d2h_ms / e2e_step_ms,
                    "note": "ceiling = cudaMemcpyAsync of the same %d MB from HBM to pinned host memory, every rank at "
                            "once, same run; the kernels are %.1f %% of the step" % (d2h_bytes // 1000000, 100 * ms_per_step / e2e_step_ms)},
            "gpu_launches": int(launches), "host_enqueue_ms_per_step": host_enqueue_ms, "numa": numa,
            "host_buffer_placement": placement,
            "clocks": clocks,
            "roofline": {"bound": "hbm", "kernel": "rsurf_wide_kernel", "achieved": achieved, "peak": hbm_peak,
                         "unit": "GB/s", "frac": achieved / hbm_peak, "traffic": _ncu_traffic(),
                         "peak_source": peak_src, "kernel_ms": rsurf_ms, "geom_kernel_ms": geom_ms,
                         "how": "kernel_ms = mean CUDA-event time of the kernel's own launches (second pass of the K "
                                "steps, overlap and programmatic dependent launch off); achieved = algorithmic bytes / kernel_ms",
                         "achieved_repeated": achieved_rep, "frac_repeated": achieved_rep / hbm_peak,
                         "repeated_note": "algorithmic bytes / ms_per_step of the overlapped timed region (repeated-call throughput)",
                         "algorithmic_bytes_per_launch": alg_bytes,
                         "in_kernel": dict(stamps, achieved=alg_bytes / (stamps["span_us"] * 1e-6) / 1e9,
                                           frac=alg_bytes / (stamps["span_us"] * 1e-6) / 1e9 / hbm_peak,
                                           note="%globaltimer stamps of every CTA of an isolated launch (gort_kernel_stamps): span = first CTA's "
                                                "first instruction to last CTA's last completed store.  kernel_ms (CUDA events) additionally holds the "
                                                "launch and completion latency outside any CTA"),
                         "executed_work": _ncu_executed("rsurf_wide_kernel<4, 0, 2, 3, 0>")},
            "checksum": checksum,
        }
        if multi is not None:
            out["extras"] = multi
        if world == 1 and not args.no_extras:
            out["extras"] = extras(g, torch, dev, ts, near_cpus)
        if world == 1 and not args.no_cpu_baseline:
            os.sched_setaffinity(0, all_cpus)          # the CPU arm uses every host core
            out["cpu_baseline"] = cpu_baseline(rsurf_e2e, wl)
            out["max_rel_err"] = out["cpu_baseline"]["parity"]["max_rel_err"]
            if not args.no_extras:
                import parity_audit as pa
                rep = pa.audit(g, sizes=pa.BENCH_SIZES)
                out["extras"]["parity"] = {"pass": rep["pass"], "seconds": rep["seconds"], "tolerance": rep["tolerance"],
                                           "checker": rep["checker"],
                                           "columns": "per output: [max_rel_err, n_beyond_tol, n_excused, n_unexplained]",
                                           "sample": {c: v["what"] for c, v in rep["configs"].items()},
                                           "outputs": pa.headline(rep),
                                           "per_band": {c: {k: o.get("max_rel_err_per_band") or o.get("max_rel_err_per_100nm_from")
                                                            for k, o in v["outputs"].items() if k in ("rsurf", "albedo", "favegt", "fasoil")}
                                                        for c, v in rep["configs"].items()}}
                if not rep["pass"]:
                    print(json.dumps(out), flush=True)
                    raise SystemExit("bench.py: parity audit failed: %s" % "; ".join(pa.failures(rep)))
            if not out["cpu_baseline"]["parity"]["pass"]:
                print(json.dumps(out), flush=True)
                raise SystemExit("bench.py: parity check against the CPU arm failed")
        print(json.dumps(out), flush=True)

    g.close()
    if world > 1:
        dist.destroy_process_group()


def _plain_d2h_ms(torch, dev, ts, d_src, h_dst, barrier, reps=5):
    """best-of-reps CUDA-event time of one plain D2H copy into the (pinned, library-placed) host array h_dst, started on
    all ranks together"""
    h = torch.from_numpy(h_dst.reshape(-1))
    src = d_src.reshape(-1)[:h.numel()]
    best = 1e30
    with torch.cuda.stream(ts):
        for k in range(reps + 1):
            barrier()
            a = torch.cuda.Event(enable_timing=True); b = torch.cuda.Event(enable_timing=True)
            a.record(ts); h.copy_(src, non_blocking=True); b.record(ts); b.synchronize()
            if k:
                best = min(best, a.elapsed_time(b))
    return best


def multi_gpu_extras(g, torch, dist, dev, ts, rank, world, args):
    """N > 1 (every rank calls this; rank 0 reports).
    c5_lut_allgather: the C5 structural grid (131 072 LUTs) sharded by contiguous blocks of parameter sets, each rank's
        kernels, then ONE NCCL all-gather of the records (the only collective of the whole path, gortt.c:123-128 is the
        record), checked bit for bit against one GPU computing the whole grid.
    c2_strong: the sweep of ONE forest split by geometry blocks over the ranks (strong scaling, no collective)."""
    from gort_b200 import workloads as wk
    from gort_b200.api import LUT_STRIDE
    from gort_b200.parallel import shard_range
    stream = ts.cuda_stream
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    res = {}

    # ---- C5: sharded LUT generation + all-gather ----
    st = wk.c5_lut_grid()["structure"]
    M = st.shape[1]
    lo, hi = shard_range(M, rank, world)
    assert (hi - lo) * world == M, "the C5 grid divides evenly over 2 / 4 / 8 ranks"
    d_blk = T(st[:, lo:hi])                                  # H2D of the structure block: set-up, not timed
    d_loc = torch.empty((hi - lo, LUT_STRIDE), dtype=torch.float64, device=dev)
    d_all = torch.empty((M, LUT_STRIDE), dtype=torch.float64, device=dev)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    best = None
    with torch.cuda.stream(ts):
        for k in range(4):                                   # first pass: NCCL's lazily created communicator, module load
            dist.barrier(); torch.cuda.synchronize()
            ev[0].record(ts)
            g.lut_dev(d_blk, d_loc, stream=stream)
            ev[1].record(ts)
            dist.all_gather_into_tensor(d_all, d_loc)
            ev[2].record(ts)
            ev[2].synchronize()
            t = (ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2]), ev[0].elapsed_time(ev[2]))
            if k and (best is None or t[2] < best[2]):
                best = t
    tt = torch.tensor(best, dtype=torch.float64, device=dev)
    dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    kern_ms, gather_ms, total_ms = [float(x) for x in tt.tolist()]
    # the same with the all-gather hidden under the kernels: 4 super-blocks, each split over the ranks, the gather of
    # super-block j on a second stream while the kernels of super-block j+1 run (gort_b200/parallel.py)
    from gort_b200.parallel import lut_generate_pipelined
    n_sub = 4
    d_blocks, pipe_best, d_pipe = None, None, None
    with torch.cuda.stream(ts):
        for k in range(4):
            dist.barrier(); torch.cuda.synchronize()
            pa_, pb_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            pa_.record(ts)
            d_pipe, d_blocks = lut_generate_pipelined(st, g, rank, world, dev, n_sub=n_sub, compute_stream=ts, d_blocks=d_blocks)
            pb_.record(ts)
            pb_.synchronize()
            if k:
                pipe_best = pa_.elapsed_time(pb_) if pipe_best is None else min(pipe_best, pa_.elapsed_time(pb_))
    tp = torch.tensor([pipe_best], dtype=torch.float64, device=dev)
    dist.all_reduce(tp, op=dist.ReduceOp.MAX)
    pipe_ms = float(tp.item())
    # the same with NO collective: every rank's kernels store their rows into every rank's table while they compute
    # (gort_lut_batch_scatter_dev over symmetric memory: per-peer NVLink addresses, and the NVSwitch multicast address
    # when there is one), a device-side barrier of the ranks before and after, all inside the timed region
    from gort_b200.parallel import PeerLutTable, lut_generate_peer
    peer = {}
    try:
        tab = PeerLutTable(M, dev)
    except Exception as e:      # the platform refused symmetric memory (no fabric / fd handle exchange): say so, keep NCCL
        tab, peer = None, {"unavailable": "%s: %s" % (type(e).__name__, str(e).splitlines()[0] if str(e) else "")}
    d_peer = {}
    if tab is not None:
        modes = [("peer", False)] + ([("multicast", True)] if tab.multicast_ptr else [])
        for name, mc in modes:
            with torch.cuda.stream(ts):
                tab.table.zero_()
            dist.barrier(); torch.cuda.synchronize()
            bestp = None
            for k in range(4):
                dist.barrier(); torch.cuda.synchronize()
                pa_, pb_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                pa_.record(ts)
                lut_generate_peer(d_blk, tab, g, ts, multicast=mc)
                pb_.record(ts)
                pb_.synchronize()
                if k:
                    bestp = pa_.elapsed_time(pb_) if bestp is None else min(bestp, pa_.elapsed_time(pb_))
            tq = torch.tensor([bestp], dtype=torch.float64, device=dev)
            dist.all_reduce(tq, op=dist.ReduceOp.MAX)
            peer[name + "_total_ms"] = float(tq.item())
            dist.barrier(); torch.cuda.synchronize()
            d_peer[name] = tab.table.clone()
    # one GPU computing the whole grid: the reference bits and the 1-GPU kernel time
    d_full = T(st)
    d_one = torch.empty((M, LUT_STRIDE), dtype=torch.float64, device=dev)
    one_ms = _time_dev(torch, ts, lambda: g.lut_dev(d_full, d_one, stream=stream), reps=2)
    ts.synchronize()
    same = bool(torch.equal(torch.nan_to_num(d_all, nan=-7.0), torch.nan_to_num(d_one, nan=-7.0)) and
                torch.equal(torch.nan_to_num(d_pipe, nan=-7.0), torch.nan_to_num(d_one, nan=-7.0)))
    for name, t_ in d_peer.items():
        same = same and bool(torch.equal(torch.nan_to_num(t_, nan=-7.0), torch.nan_to_num(d_one, nan=-7.0)))
    flag = torch.tensor([1.0 if same else 0.0], dtype=torch.float64, device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if flag.item() != 1.0:
        raise SystemExit("bench: a multi-GPU assembly of the C5 grid differs from the bits one GPU computes")
    bytes_total = M * LUT_STRIDE * 8
    fused_ms = min([v for k_, v in peer.items() if k_.endswith("_total_ms")], default=None)
    best_ms = min(x for x in (total_ms, pipe_ms, fused_ms) if x is not None)
    res["c5_lut_allgather"] = {
        "luts": M, "luts_per_rank": hi - lo, "kernel_ms": kern_ms, "allgather_ms": gather_ms, "total_ms": total_ms,
        "pipelined_total_ms": pipe_ms, "pipelined_super_blocks": n_sub,
        "peer_stores": peer, "best_total_ms": best_ms,
        "luts_per_s": M / (best_ms * 1e-3), "one_gpu_kernel_ms": one_ms,
        "speedup_vs_one_gpu": one_ms / best_ms, "speedup_vs_one_gpu_allgather": one_ms / total_ms,
        "speedup_vs_one_gpu_pipelined": one_ms / pipe_ms,
        "allgather_bytes_total": bytes_total, "allgather_bytes_received_per_rank": bytes_total * (world - 1) // world,
        "allgather_gbs_per_rank": bytes_total * (world - 1) / world / (gather_ms * 1e-3) / 1e9,
        "assembled_equals_one_gpu_bits_on_every_rank": bool(flag.item() == 1.0),
        "timing": "CUDA events on the launching stream, best of 3 after a first pass, max over ranks; the structure blocks are "
                  "resident before the timed region.  kernel_ms / allgather_ms / total_ms: contiguous shards, kernels then ONE "
                  "all-gather; pipelined_total_ms: the grid in super-blocks, the gather of one under the kernels of the next; "
                  "peer_stores: no collective, the kernels that produce a row store it into every rank's table (per-peer "
                  "NVLink addresses / the NVSwitch multicast address), barriers of the ranks inside the timed region"}
    del d_pipe, d_blocks, d_peer, tab
    del d_full, d_one, d_all, d_loc

    # ---- C2 strong scaling: one forest, geometry blocks across ranks ----
    w = wk.c2_hemisphere()
    ang, wl = w["angles"], w["wavelength"]
    G, W = ang.shape[1], wl.shape[0]
    glo, ghi = shard_range(G, rank, world)
    lut = g.lut(w["structure"])
    rl, tl, rs = g.spectra(w["leaf"], w["soil"], wl)
    pitch = (W + 15) // 16 * 16
    d_in = [T(w["structure"]), T(lut), T(ang[:, glo:ghi]), T(rl[0]), T(tl[0]), T(rs[0])]
    d_o = torch.empty((1, ghi - glo, pitch), dtype=torch.float64, device=dev)
    call = g.brdf_dev_bind(*d_in, d_o, stream=stream)
    g.set_overlap(True)
    for _ in range(args.warmup):
        call()
    dist.barrier(); torch.cuda.synchronize()
    a = torch.cuda.Event(enable_timing=True); b = torch.cuda.Event(enable_timing=True)
    a.record(ts)
    for _ in range(args.steps):
        call()
    b.record(ts)
    dist.barrier(); torch.cuda.synchronize()
    g.set_overlap(False)
    tt = torch.tensor([a.elapsed_time(b)], dtype=torch.float64, device=dev)
    dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    ms = float(tt.item()) / args.steps
    res["c2_strong"] = {"lines_total": G, "lines_per_rank": ghi - glo, "wavelengths": W, "ms_per_step": ms,
                        "evals_per_s": G * W / (ms * 1e-3), "scaling": "strong",
                        "note": "one forest, contiguous geometry blocks per rank, no collective; device-resident, overlap mode"}
    return res


def _time_dev(torch, ts, fn, reps=3):
    """best-of-reps CUDA-event time (ms) of fn() enqueued on stream ts, after one warm-up"""
    fn()
    ts.synchronize()
    best = 1e30
    for _ in range(reps):
        a = torch.cuda.Event(enable_timing=True); b = torch.cuda.Event(enable_timing=True)
        a.record(ts); fn(); b.record(ts); b.synchronize()
        best = min(best, a.elapsed_time(b))
    return best


def extras(g, torch, dev, ts, near_cpus=None):
    """N = 1: device-resident timings of the other kernels on the BASELINE.json configs they serve (full sizes).
    FP64 figures: `algorithmic` uses the contract's per-unit flop counts (SURVEY.md App. D) -- for the BRDF and energy
    kernels that is the reference's work, most of which the regrouping removed, so it is labelled work avoided and is NOT a
    utilisation; `executed` is what ncu counted for the kernel (profiles/r2_ncu_summary.json, committed with the run it
    came from)."""
    from gort_b200 import workloads as wk
    from gort_b200.api import LUT_STRIDE
    import gort_b200
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    E = lambda *shape: torch.empty(shape, dtype=torch.float64, device=dev)
    stream = ts.cuda_stream
    res = {}
    hbm, _ = load_peaks()
    dfma_tflops = g.dfma_peak_tflops()
    res["dfma_microbench_tflops"] = dfma_tflops

    def alg(flops, ms, kernel, avoided):
        tf = flops / (ms * 1e-3) / 1e12
        d = {"algorithmic_flop": flops, "algorithmic_tflops": tf, "dfma_peak_tflops": dfma_tflops,
             "executed": _ncu_executed(kernel)}
        if avoided:
            d["note"] = "algorithmic = the reference's operation count; the regrouped kernel executes a fraction of it: work avoided, not a utilisation"
        else:
            d["frac_of_dfma_peak"] = tf / dfma_tflops
        return d

    # ---- C2 variants: shuffled line order, component signatures ----
    w = wk.c2_hemisphere()
    ang, wl = w["angles"], w["wavelength"]
    G, W = ang.shape[1], wl.shape[0]
    Wp = (W + 15) // 16 * 16
    d_st = T(w["structure"])
    d_lut = E(1, LUT_STRIDE); g.lut_dev(d_st, d_lut, stream=stream)
    d_rl, d_tl, d_rs = E(1, W), E(1, W), E(1, W)
    g.spectra_dev(T(w["leaf"]), T(w["soil"]), T(wl), d_rl, d_tl, d_rs, stream=stream)
    d_r = E(1, G, Wp)
    d_ang = T(ang)
    nat_ms = _time_dev(torch, ts, lambda: g.brdf_dev(d_st, d_lut, d_ang, d_rl[0], d_tl[0], d_rs[0], d_r, stream=stream))
    perm = np.random.Generator(np.random.PCG64(4)).permutation(G)
    d_angp = T(ang[:, perm])
    shf_ms = _time_dev(torch, ts, lambda: g.brdf_dev(d_st, d_lut, d_angp, d_rl[0], d_tl[0], d_rs[0], d_r, stream=stream))
    res["c2_shuffled"] = {"lines": G, "wavelengths": W, "isolated_call_ms_natural_order": nat_ms, "isolated_call_ms_shuffled": shf_ms,
                          "evals_per_s_shuffled": G * W / (shf_ms * 1e-3),
                          "hbm_frac_shuffled": 8.0 * G * W / (shf_ms * 1e-3) / 1e9 / hbm,
                          "note": "same sweep, lines permuted: every line starts a new run, so the (sun, lambda) terms "
                                  "(2 divisions + ~35 FP64 operations per wavelength) are rebuilt per line instead of once per "
                                  "36 lines and the kernel turns FP64-bound; callers that can should keep lines sharing a sun adjacent"}
    # back to back into ROTATING output buffers (a consumer that double-buffers): the output pointer is part of the
    # call's signature, so overlap mode does not engage and every call pays its geometry kernel and start-up
    d_r2 = E(1, G, Wp)
    binds = [g.brdf_dev_bind(d_st, d_lut, d_ang, d_rl[0], d_tl[0], d_rs[0], o, stream=stream) for o in (d_r, d_r2)]
    g.set_overlap(True)

    def rotate(n=40):
        for k in range(n):
            binds[k & 1]()
    rot_ms = _time_dev(torch, ts, rotate) / 40
    g.set_overlap(False)
    res["c2_rotated_outputs"] = {"calls": 40, "ms_per_call": rot_ms, "evals_per_s": G * W / (rot_ms * 1e-3),
                                 "hbm_frac": 8.0 * G * W / (rot_ms * 1e-3) / 1e9 / hbm,
                                 "note": "40 calls back to back alternating between two output buffers, overlap mode requested: "
                                         "it applies only to repeated calls into the same buffers, so this is plain stream order"}
    del d_r2, binds
    d_sc = E(1, G, Wp, 4)
    sc_ms = _time_dev(torch, ts, lambda: g.brdf_dev(d_st, d_lut, d_ang, d_rl[0], d_tl[0], d_rs[0], d_r, scomp=d_sc, stream=stream))
    res["c2_prnspec"] = {"lines": G, "wavelengths": W, "brdf_ms": sc_ms, "evals_per_s": G * W / (sc_ms * 1e-3),
                         "roofline": {"bound": "hbm", "achieved": 40.0 * G * W / (sc_ms * 1e-3) / 1e9, "peak": hbm, "unit": "GB/s",
                                      "frac": 40.0 * G * W / (sc_ms * 1e-3) / 1e9 / hbm,
                                      "note": "geometry kernel + per-wavelength kernel of one isolated call over the whole sweep, "
                                              "40 B per evaluation (rsurf + C, G, T, Z), 980 MB out"}}
    del d_r, d_sc

    # ---- C3: spectral albedo + fAPAR, 10^4 sets x 3 sun angles x 211 bands x 512 quadrature nodes ----
    w = wk.c3_albedo()
    M, W, S = w["structure"].shape[1], w["wavelength"].shape[0], w["angles"].shape[1]
    d_st, d_leaf, d_soil, d_wl, d_ang = T(w["structure"]), T(w["leaf"]), T(w["soil"]), T(w["wavelength"]), T(w["angles"])
    d_lut = E(M, LUT_STRIDE); d_rl, d_tl, d_rs = E(M, W), E(M, W), E(M, W)
    lut_ms = _time_dev(torch, ts, lambda: g.lut_dev(d_st, d_lut, stream=stream))
    sp_ms = _time_dev(torch, ts, lambda: g.spectra_dev(d_leaf, d_soil, d_wl, d_rl, d_tl, d_rs, stream=stream))
    # the same sets with the intermediates the reference also computes (vb, fb, t_open, dt_open, dk_open: ~90 % of its
    # LUT time, never read by the BRDF): "same work as the reference"
    d_int = [E(M, k) for k in (15, 15 * 91, 225, 225, 15, 15)]
    int_ms = _time_dev(torch, ts, lambda: g.lut_intermediates_dev(d_st, *d_int, stream=stream), reps=2)
    del d_int
    d_a, d_v, d_s = E(M, S, W), E(M, S, W), E(M, S, W)
    en_ms = _time_dev(torch, ts, lambda: g.energy_dev(d_st, d_lut, d_ang, d_rl, d_tl, d_rs, d_a, d_v, d_s, stream=stream))
    evals = M * S * 512 * W
    res["c3_albedo"] = {"sets": M, "sun_angles": S, "wavelengths": W, "quadrature_nodes": 512,
                        "energy_kernels_ms": en_ms, "evals_per_s": evals / (en_ms * 1e-3),
                        "energy_fp64": alg(M * S * 512 * (F_GEOM + W * (F_LAMBDA + 2.0)), en_ms, "energy_kernel", True),
                        "executed_per_sun_line": "16 zenith records + 512 azimuth passes + W spectral evaluations (the reference: 512 full "
                                                 "records + 512 W evaluations)",
                        "lut_kernels_ms": lut_ms, "luts_per_s": M / (lut_ms * 1e-3),
                        "lut_fp64": alg(M * F_LUT, lut_ms, "lut_tube_kernel", False),
                        "lut_intermediates_ms": int_ms,
                        "luts_per_s_same_work_as_reference": M / ((lut_ms + int_ms) * 1e-3),
                        "lut_same_work_note": "outputs (lut_kernels_ms) + the intermediates the reference computes on every run and the "
                                              "BRDF never reads (gort_lut_intermediates_batch: vb, fb, t_open, dt_open, dk_open)",
                        "spectra_kernel_ms": sp_ms, "spectra_fp64": alg(M * W * 130.0, sp_ms, "spectra_kernel", False),
                        "finite_fraction": float(torch.isfinite(d_a).double().mean())}
    del d_a, d_v, d_s

    # ---- C4: EnKF forward operator, 10^5 members x 16 geometries x 7 bands (all parameters varying) ----
    w = wk.c4_enkf()
    M, G, W = w["structure"].shape[1], w["angles"].shape[2], w["wavelength"].shape[0]
    d_st, d_leaf, d_soil, d_wl, d_ang = T(w["structure"]), T(w["leaf"]), T(w["soil"]), T(w["wavelength"]), T(w["angles"])
    d_lut = E(M, LUT_STRIDE); d_rl, d_tl, d_rs = E(M, W), E(M, W), E(M, W); d_out = E(M, G, W)
    lut_ms = _time_dev(torch, ts, lambda: g.lut_dev(d_st, d_lut, stream=stream), reps=2)
    sp_ms = _time_dev(torch, ts, lambda: g.spectra_dev(d_leaf, d_soil, d_wl, d_rl, d_tl, d_rs, stream=stream))
    br_ms = _time_dev(torch, ts, lambda: g.brdf_dev(d_st, d_lut, d_ang, d_rl, d_tl, d_rs, d_out, stream=stream))
    evals = M * G * W
    res["c4_enkf"] = {"members": M, "geometries": G, "bands": W, "brdf_ms": br_ms, "evals_per_s": evals / (br_ms * 1e-3),
                      "brdf_fp64": alg(M * G * (F_GEOM + W * F_LAMBDA), br_ms, "rsurf_flat_kernel", True),
                      "lut_kernels_ms": lut_ms, "luts_per_s": M / (lut_ms * 1e-3), "lut_fp64": alg(M * F_LUT, lut_ms, "lut_tube_kernel", False),
                      "spectra_kernel_ms": sp_ms,
                      "whole_member_update_ms": lut_ms + sp_ms + br_ms,
                      "evals_per_s_including_lut_and_spectra": evals / ((lut_ms + sp_ms + br_ms) * 1e-3),
                      "finite_fraction": float(torch.isfinite(d_out).double().mean())}
    # the same member update end to end through the host-pointer API: pinned host arrays in, rsurf out (the DA use case)
    hp = {k: _pinned_copy(gort_b200, np.ascontiguousarray(w[k]), near_cpus) for k in ("structure", "leaf", "soil", "angles")}
    h_out = gort_b200.PinnedArray((M, G, W), cpus=near_cpus)

    def member_update():
        lut_h = g.lut(hp["structure"].array)
        rl_h, tl_h, rs_h = g.spectra(hp["leaf"].array, hp["soil"].array, w["wavelength"])
        g.brdf(hp["structure"].array, lut_h, hp["angles"].array, rl_h, tl_h, rs_h, out=h_out.array)

    member_update()
    t_best = 1e30
    for _ in range(3):
        t0 = time.perf_counter(); member_update(); t_best = min(t_best, time.perf_counter() - t0)
    res["c4_enkf"]["e2e_three_calls_ms"] = t_best * 1e3
    res["c4_enkf"]["e2e_three_calls_note"] = ("gort_lut_batch + gort_spectra_batch + gort_brdf_batch with host arrays: LUTs and spectra "
                                              "travel through host memory between the calls")
    # ... and through the ensemble forward operator: one call, LUTs and spectra stay on the GPU, members in chunks on two
    # streams so that the copies of one chunk run under the kernels of the next
    fwd = lambda: g.forward(hp["structure"].array, hp["leaf"].array, hp["soil"].array, w["wavelength"], hp["angles"].array, out=h_out.array)
    fwd()
    t_fwd = 1e30
    for _ in range(3):
        t0 = time.perf_counter(); fwd(); t_fwd = min(t_fwd, time.perf_counter() - t0)
    res["c4_enkf"]["e2e_forward_batch_ms"] = t_fwd * 1e3
    res["c4_enkf"]["e2e_evals_per_s"] = evals / t_fwd
    res["c4_enkf"]["e2e_members_per_s"] = M / t_fwd
    res["c4_enkf"]["e2e_frac_of_kernel_time"] = (lut_ms + sp_ms + br_ms) / (t_fwd * 1e3)
    res["c4_enkf"]["e2e_note"] = ("gort_forward_batch with pinned host arrays: %d B in and %d B out per member; compute-bound: "
                                  "the ceiling is the kernels' own time (whole_member_update_ms)" % (8 * (6 + 7 + 4 + 4 * G), 8 * G * W))

    # C4a: the same ensemble with the crown structure shared and only LAI varying (favd): one crown-geometry phase
    # and one crown-count loop per LUT sub-group
    wa = wk.c4_enkf(vary_structure=False)
    d_sta = T(wa["structure"])
    luta_ms = _time_dev(torch, ts, lambda: g.lut_dev(d_sta, d_lut, stream=stream), reps=2)
    res["c4_enkf"]["lai_only_lut_kernels_ms"] = luta_ms
    res["c4_enkf"]["lai_only_luts_per_s"] = M / (luta_ms * 1e-3)

    # ---- C5: LUT generation over the structural grid (131 072 parameter sets), one GPU's share = all of it here ----
    st = wk.c5_lut_grid()["structure"]
    M = st.shape[1]
    d_st = T(st); d_lut = E(M, LUT_STRIDE)
    lut_ms = _time_dev(torch, ts, lambda: g.lut_dev(d_st, d_lut, stream=stream), reps=2)
    res["c5_lut_grid"] = {"luts": M, "lut_kernels_ms": lut_ms, "luts_per_s": M / (lut_ms * 1e-3),
                          "lut_fp64": dict(alg(M * F_LUT, lut_ms, "lut_crown_kernel<8>", True),
                                           note="algorithmic = the reference's per-set operation count; the grid shares crown shapes (64 sets "
                                                "per shape, sub-groups of 8 per stem density), so most of it is computed once per group: work "
                                                "avoided, not a utilisation"),
                          "bytes_out": M * LUT_STRIDE * 8, "nan_luts": int(torch.isnan(d_lut).any(dim=1).sum())}
    return res


def _pinned_copy(gort_b200, a, cpus=None):
    p = gort_b200.PinnedArray(a.shape, cpus=cpus)
    p.array[...] = a
    return p


def _ncu_traffic():
    """dram bytes per launch of the dominant kernel from the committed ncu --set full capture, if any."""
    p = ROOT / "profiles" / "rsurf_wide_dram_bytes.json"
    if p.exists():
        try:
            return json.loads(p.read_text())["dram_bytes_per_launch"]
        except Exception:
            return None
    return None


def _ncu_executed(kernel):
    """what ncu counted for `kernel` in the committed capture (profiles/r2_ncu_summary.json), or None"""
    p = ROOT / "profiles" / "r2_ncu_summary.json"
    if p.exists():
        try:
            return json.loads(p.read_text()).get(kernel)
        except Exception:
            return None
    return None


def _parity_per_band(kind, st, lut, ang, rl, tl, rs, lines, gpu_rsurf, wavelength):
    import checkers
    chk = checkers.ref() if kind == "reference" else checkers.oracle()
    idx = (np.arange(lines) * 37) % ang.shape[1]
    r_ref, _, _ = chk.brdf(st, lut, np.ascontiguousarray(ang[:, idx].T), rl, tl, rs, want_scomp=False)
    r_gpu = np.asarray(gpu_rsurf)[idx]
    nan_ok = bool(np.array_equal(np.isnan(r_gpu), np.isnan(r_ref)))
    with np.errstate(invalid="ignore"):
        rel = np.abs(r_gpu - r_ref) / np.maximum(np.abs(r_ref), 1e-12)
    per_band = np.nanmax(rel, axis=0)                                      # worst line, per wavelength
    wl = np.asarray(wavelength)
    bins = [(int(lo), float(per_band[(wl >= lo) & (wl < lo + 100)].max())) for lo in range(400, 2500, 100)]
    return {"against": kind, "what": "rsurf from GPU LUT + GPU spectra + GPU BRDF vs the CPU arm's own chain",
            "lines": lines, "bands": int(per_band.size), "tolerance": 1e-9,
            "max_rel_err": float(per_band.max()), "worst_band_nm": float(wl[int(per_band.argmax())]),
            "max_rel_err_per_100nm_from": bins, "nan_positions_coincide": nan_ok,
            "pass": bool(nan_ok and per_band.max() <= 1e-9)}


def cpu_baseline(gpu_rsurf=None, wavelength=None):
    """Bounded sample (~10-20 s of CPU work) of the same sweep on the host cores.  The leg's own outputs double as
    the parity check the metric asks for: the lines core 0 evaluates (reference LUT, reference spectra, reference
    BRDF) against the GPU path's result for the same lines, worst relative error per output band."""
    import multiprocessing as mp
    cores = os.cpu_count() or 1
    kind, st, lut, ang, rl, tl, rs = cpu_arm_setup()
    lines = 96
    parity = None
    if gpu_rsurf is not None:       # a parity leg that throws fails the bench: no except here
        parity = _parity_per_band(kind, st, lut, ang, rl, tl, rs, lines, gpu_rsurf, wavelength)
    with mp.get_context("fork").Pool(cores) as pool:
        cpu_arm_step(pool, cores, kind, st, lut, ang, rl, tl, rs, 8)                   # warm-up
        n1, t1 = cpu_arm_step(pool, cores, kind, st, lut, ang, rl, tl, rs, lines)
        reps = int(min(40, max(1, 12.0 / max(t1, 1e-3))))
        n, t = cpu_arm_step(pool, cores, kind, st, lut, ang, rl, tl, rs, lines, reps=reps)
        # the same sample through the build with the reference makefile's own flags (-g: no optimisation), SURVEY.md 8d
        import checkers
        slow = None
        if kind == "reference" and checkers.ref_makefile_flags() is not None:
            ng, tg = cpu_arm_step(pool, cores, "reference-g", st, lut, ang, rl, tl, rs, lines, reps=max(1, reps // 8))
            slow = {"value": ng / tg, "unit": UNIT, "cores": cores, "flags": "-Wall -g (the reference makefile's CFLAGS)",
                    "note": "same bits as the canonical -O2 -ffp-contract=off build (tests/test_oracle_cpu.py)"}
    out = {"value": n / t, "unit": UNIT, "cores": cores, "kind": kind,
           "sample": "%d lines x 2101 bands x %d reps per core (strided slice of the c2 sweep), in-process, "
                     "LUT and spectra given" % (lines, reps)}
    if slow is not None:
        out["makefile_flag_build"] = slow
    if parity is not None:
        out["parity"] = parity
    return out


if __name__ == "__main__":
    main()

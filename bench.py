#!/usr/bin/env python
"""bench.py -- RK4 grid-point.steps/s of the pseudospectral barotropic step on B200.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--grid G] [--impl xfb|reference] [--dump-outputs DIR]

One "step" is one RK4 step (4 tendency evaluations = 20 2-D FFTs in the reference).
  N = 1 : the elliptic vortex (reference generator makefield-elliptic-vortex.cpp) at 8192^2 -- the headline grid of
          BASELINE.json's north_star -- on one GPU ("scaling": "weak").
  N > 1 (launched by torchrun, one rank per GPU): BASELINE.json configs[4], the 16384^2 constant vortex SLAB-DECOMPOSED
          over the N GPUs with an NVLink all-to-all per 2-D transform ("scaling": "strong": the grid is fixed).  The
          same run verifies the slab result against the single-GPU path on that grid, measures the single-GPU time
          per step (T1) for parallel_efficiency = T1 / (N * T_N), and reports independent ensemble members (one
          8192^2 member per GPU, no communication) as the sub-record "ensemble".  `--ensemble` makes the ensemble the
          headline instead (the round-1 behaviour).

Output: ONE JSON line on rank 0 (keys documented in DESIGN.md "Measurement").
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "rk4_grid_point_steps_per_s"
UNIT = "grid-pt*steps/s"
ALGO_BYTES_PER_PT_STEP = 240.0      # SURVEY.md section 8(d): 4 stages x (40 B K-COL + 20 B K-ROW)
ALGO_BYTES_COL = 40.0               # per grid point per K-COL launch
ALGO_BYTES_ROW = 20.0               # per grid point per K-ROW launch


def dt_for(n: int) -> float:
    """RK4 advective limit for the elliptic vortex (|U|max = 83 m/s): 0.6 * 2.83/(k_max |U|), SURVEY 8(d)"""
    if n <= 1024:
        return 3.0
    kmax = 0.943 * np.pi * n / 600000.0
    return float(np.float32(0.6 * 2.83 / (kmax * 83.0)))


def measured_traffic(grid: int, which: str):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu --set full capture, or None"""
    p = os.path.join(ROOT, "profiles", "r02_traffic.json")
    try:
        d = json.load(open(p))
        return float(d[str(grid)][which]["dram_bytes_per_launch"]), d["source"]
    except Exception:
        return None, None


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """samples SM clock and throttle reasons with NVML every 100 ms while the timed region runs"""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop_evt.wait(0.1)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


def physical_gpu_index(local_rank: int) -> int:
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local_rank])
        except Exception:
            return local_rank
    return local_rank


# --------------------------------------------------------------------------------------------------
# CPU reference leg (oracle/_ref = the unmodified reference main.cpp built against the FFT shim)
# --------------------------------------------------------------------------------------------------

def run_reference_steps(n: int, dt: float, steps_a: int, steps_b: int, threads: int, field: str = "elliptic", budget_s: float = None):
    """Times the UNMODIFIED reference binary for two run lengths and differences them
    (start-up, table build and the step-0 record dump cancel).  Returns seconds per step.
    budget_s: the second run length is cut so that the whole measurement stays within about that many seconds
    (estimated from the first run); the run lengths actually used are returned in the note."""
    from oracle import build_oracle
    import fields
    exe = build_oracle.build_reference(n, programs=("main",)).get("main")
    if exe is None:
        return None, "no prebuilt reference binary for this grid"
    v0 = fields.GENERATORS[field](n)
    times = []
    with tempfile.TemporaryDirectory() as d:
        os.makedirs(os.path.join(d, "input"))
        os.makedirs(os.path.join(d, "output"))
        v0.tofile(os.path.join(d, "input", "initial_vorticity.bin"))
        for k, steps in enumerate((steps_a, steps_b)):
            if k == 1 and budget_s is not None:
                # T(steps_a) = start-up + steps_a steps >= steps_a steps: a safe (over-)estimate of the step time
                est = max(times[0] / max(1, steps_a), 1e-3)
                steps = steps_b = max(steps_a + 2, min(steps_b, steps_a + int(budget_s / est)))
            env = dict(os.environ, XFB_SHIM_THREADS=str(threads), XFB_DT=repr(float(dt)),
                       XFB_TOTAL_STEPS=str(steps), XFB_RECORD_STEP=str(10 ** 9))
            t0 = time.perf_counter()
            subprocess.run([exe], cwd=d, check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL, env=env)
            times.append(time.perf_counter() - t0)
    per_step = (times[1] - times[0]) / (steps_b - steps_a)
    if per_step <= 0:          # tiny samples: start-up noise larger than the steps themselves; fall back to the long run alone
        per_step = times[1] / steps_b
    return per_step, f"(T({steps_b} steps) - T({steps_a} steps)) / {steps_b - steps_a}"


def single_thread_figure(n: int = 1024, nsteps: int = 4):
    """the reference exactly as shipped (FFTW_ESTIMATE, no threads: main.cpp:126-135) -- one host thread, small grid"""
    sec, how = run_reference_steps(n, dt_for(n), 1, 1 + nsteps, 1)
    if sec is None or sec <= 0:
        return None
    return {"value": n * n / sec, "unit": UNIT, "cores": 1, "sample": f"elliptic {n}^2, 1 thread (as the reference ships), {how}"}


def cpu_baseline(sample_n: int, nsteps: int):
    threads = os.cpu_count() or 1
    sec, how = run_reference_steps(sample_n, dt_for(sample_n), 1, 1 + nsteps, threads, budget_s=25.0)
    if sec is None or sec <= 0:
        return {"value": None, "unit": UNIT, "cores": threads, "kind": "reference", "sample": how or "failed"}
    return {
        "value": sample_n * sample_n / sec, "unit": UNIT, "cores": threads, "kind": "reference",
        "sample": (f"unmodified reference main.cpp + fftw3f-equivalent shim (FFT rows/columns on {threads} OpenMP "
                   f"threads, pointwise loops single-threaded as in the reference), elliptic {sample_n}^2, {how}"),
        "single_thread": single_thread_figure(),
    }


def reference_arm(args):
    """--impl reference: the reference's own CPU implementation of the path (unmodified main.cpp + FFT shim) on this box's
    host cores, ON THE PRODUCT ARM'S CONFIG: elliptic 8192^2 at N = 1, constant vortex 16384^2 at N > 1 (the reference has
    no parallel path: the same single process whatever N).  Run-length differencing (BASELINE.md section 3); the second
    run length is bounded so the arm ends within a few minutes whatever K is."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    slab = args.gpus > 1 and not args.ensemble
    field = "const" if slab else "elliptic"
    grid = args.ref_grid or args.grid
    threads = os.cpu_count() or 1
    import psutil
    need = 26 * 4 * grid * grid            # 8 real + 11 complex arrays + 3 tables (main.cpp:103-123, fftwfop.cpp:5-79)
    note = ""
    while grid > 1024 and psutil.virtual_memory().available < 1.5 * need:
        grid //= 2
        need //= 4
        note = f" (host memory too small for {args.grid}^2: sample at {grid}^2)"
    dt = 3.0 if field == "const" else dt_for(grid)
    wa = 1
    sec, how = run_reference_steps(grid, dt, wa, wa + args.steps, threads, field=field, budget_s=args.ref_budget)
    if sec is None and grid != 2048:
        grid, note = 2048, f" (no reference binary for {args.grid}^2 here: sample at 2048^2)"
        sec, how = run_reference_steps(grid, dt_for(grid) if field != "const" else 3.0, wa, wa + args.steps, threads, field=field,
                                       budget_s=args.ref_budget)
    if sec is None:
        print(json.dumps({"impl": "reference", "unavailable": how}))
        return
    val = grid * grid / sec
    sample = (f"unmodified reference main.cpp (oracle/_ref) + fftw3f-equivalent shim, {threads} OpenMP threads in the FFTs "
              f"(pointwise loops single-threaded as in the reference), one RK4 step of the {field} vortex at {grid}^2{note}, {how}")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "strong" if slab else "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{field} vortex {args.grid}^2 RK4 step" + (f", reference arm sample {grid}^2" if grid != args.grid else ""),
                   "grid": grid, "same_grid_as_product_arm": grid == args.grid},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": "reference", "sample": sample,
                         "single_thread": single_thread_figure()},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# --------------------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------------------

DUMP_BYTES = 60 * 10 ** 6         # field data; with the .npy headers the files stay under 64 MB
DUMP_FIELDS = ("vort", "psi", "u", "v")


def dump_outputs(b, n: int, members: int, out_dir: str) -> None:
    """--dump-outputs: the fields a caller reads back after the timed steps (xfb_get_field: vort, psi, u, v of every
    member) as <out_dir>/<field>[_m<member>].npy, float32.  Within DUMP_BYTES in all: where a full field does not fit,
    the same rows are kept in every file, chosen by a fixed seed, so two builds can be compared file by file."""
    import xlab_fftbarotropic_b200 as xfb
    rows_fit = max(1, DUMP_BYTES // (len(DUMP_FIELDS) * members * 4 * n))
    rows = np.arange(n) if rows_fit >= n else np.sort(np.random.default_rng(0).choice(n, rows_fit, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    for m in range(members):
        for name in DUMP_FIELDS:
            f = b.get_field(getattr(xfb.capi, name.upper()), member=m)
            np.save(os.path.join(out_dir, name + (f"_m{m}" if m else "") + ".npy"), np.ascontiguousarray(f[rows]))


def gpu_arm(args):
    import torch
    import fields
    import xlab_fftbarotropic_b200 as xfb

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    n = args.grid
    dt = dt_for(n)
    G = n * n
    b = xfb.Backend(n, batch=args.members, device=local_rank)
    stream = torch.cuda.ExternalStream(b.stream, device=local_rank)

    # synthetic input, resident in HBM before the timed region
    v0 = fields.elliptic(n)
    host_in = torch.from_numpy(v0).pin_memory()
    host_out = torch.empty((n, n), dtype=torch.float32).pin_memory()
    dev_in = host_in.to(f"cuda:{local_rank}")
    torch.cuda.synchronize()
    for m in range(args.members):
        b.set_vorticity(int(dev_in.data_ptr()), member=m)
    b.sync()

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident throughput ("value") ----------------------------------------------------
    b.step(args.warmup, dt)
    b.sync()
    sampler = ClockSampler(physical_gpu_index(local_rank))
    l0 = b.launch_count
    b.profile(True)                  # brackets every stepper launch with CUDA events on the library's stream
    barrier()
    sampler.start()
    e0 = torch.cuda.Event(enable_timing=True)
    e1 = torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(stream):
        e0.record(stream)
        b.step(args.steps, dt)
        e1.record(stream)
    barrier()
    clocks = sampler.stop()
    ms = e0.elapsed_time(e1)
    prof = b.profile_read()
    b.profile(False)
    launches = b.launch_count - l0
    # the same K steps without the per-kernel events: the library replays the step's CUDA graph (its default path).
    # THIS region is `value`; on small grids, where a launch is 15-25 us, the bracketing events cost a third of the step
    barrier()
    with torch.cuda.stream(stream):
        b.step(2, dt)
        e0.record(stream)
        b.step(args.steps, dt)
        e1.record(stream)
    barrier()
    ms_graph = e0.elapsed_time(e1)
    # `value` is the product's default path (graph replay); the bracketed pass only feeds the per-kernel roofline
    ms_bracketed = ms
    ms = ms_graph
    if args.dump_outputs and rank == 0:
        dump_outputs(b, n, args.members, args.dump_outputs)
    if dist is not None:
        t = torch.tensor([ms, ms_bracketed], device=f"cuda:{local_rank}")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, ms_bracketed = float(t[0].item()), float(t[1].item())
    units = float(G) * args.members * world * args.steps
    value = units / (ms * 1e-3)

    # sanity: the state must still be finite (a CFL blow-up would make the number meaningless)
    z = b.get_spectrum(0)
    finite = bool(np.isfinite(z.view(np.float32)).all())

    # ---- end to end through the C ABI with host buffers ("e2e") ---------------------------------
    # Every step uploads its input from pinned host memory (xfb_set_vorticity), advances one RK4 step and reads the
    # result back (xfb_get_field -> pinned host memory).  Two figures:
    #   serial    : one request at a time on one handle (copy, compute, copy strictly one after the other);
    #   pipelined : K independent requests in flight (K handles, K host threads, each making the same three
    #               synchronous calls per step), so one request's PCIe copies overlap the others' kernels.  This is
    #               how a service keeps the GPU busy behind a 55 GB/s link, and it is the `value` reported.
    e2e_steps = max(3, min(args.steps, args.e2e_steps))
    hin, hout = int(host_in.data_ptr()), int(host_out.data_ptr())

    def request_loop(be, hi, ho, nsteps):
        for _ in range(nsteps):
            for m in range(args.members):
                be.set_vorticity(hi, member=m)            # H2D of this step's input (pinned)
            be.step(1, dt)
            for m in range(args.members):
                be._ck(be._L.xfb_get_field(be._h, m, xfb.capi.VORT, ho))   # D2H of the step's result

    def timed(fn):
        barrier()
        t0 = torch.cuda.Event(enable_timing=True)
        t1 = torch.cuda.Event(enable_timing=True)
        t0.record()
        fn()
        torch.cuda.synchronize()
        t1.record()
        t1.synchronize()
        ms_ = t0.elapsed_time(t1)
        if dist is not None:
            tt = torch.tensor([ms_], device=f"cuda:{local_rank}")
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            ms_ = float(tt.item())
        return ms_

    request_loop(b, hin, hout, 2)
    ms_serial = timed(lambda: request_loop(b, hin, hout, e2e_steps))
    e2e_serial = float(G) * args.members * world * e2e_steps / (ms_serial * 1e-3)

    K = max(2, args.e2e_inflight)
    extra = []
    for _ in range(K - 1):
        bb = xfb.Backend(n, batch=args.members, device=local_rank)
        hi_t = host_in.clone().pin_memory()
        ho_t = torch.empty_like(host_out).pin_memory()
        request_loop(bb, int(hi_t.data_ptr()), int(ho_t.data_ptr()), 1)
        extra.append((bb, hi_t, ho_t))

    def in_flight():
        th = [threading.Thread(target=request_loop, args=(b, hin, hout, e2e_steps))]
        th += [threading.Thread(target=request_loop, args=(bb, int(hi_t.data_ptr()), int(ho_t.data_ptr()), e2e_steps))
               for bb, hi_t, ho_t in extra]
        for x in th:
            x.start()
        for x in th:
            x.join()

    ms_e2e = timed(in_flight)
    e2e_value = float(G) * args.members * world * (K * e2e_steps) / (ms_e2e * 1e-3)
    e2e_ms_per_step = ms_e2e / (K * e2e_steps)
    same = all(bool(np.array_equal(host_out.numpy(), ho_t.numpy())) for _, _, ho_t in extra)
    for bb, _, _ in extra:
        bb.close()

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel ---------------------------------------------------------
    peak, peak_src = measured_peaks()
    col_avg = prof["col_ms"] / max(1, prof["col_launches"])
    row_avg = prof["row_ms"] / max(1, prof["row_launches"])
    pts = float(G) * args.members
    col_gbs = ALGO_BYTES_COL * pts / (col_avg * 1e-3) / 1e9 if col_avg > 0 else 0.0
    row_gbs = ALGO_BYTES_ROW * pts / (row_avg * 1e-3) / 1e9 if row_avg > 0 else 0.0
    dominant = "col" if prof["col_ms"] >= prof["row_ms"] else "row"
    achieved = col_gbs if dominant == "col" else row_gbs
    step_gbs = ALGO_BYTES_PER_PT_STEP * value / world / 1e9
    traffic, traffic_src = measured_traffic(n, "col_step" if dominant == "col" else "row_jac") if args.members == 1 else (None, None)
    names = {"col": "colt_kernel<COL_STEP>" if n <= 8192 else "col2l_kernel<COL_STEP>",
             "row": ("rowpair_jac_tmem_kernel" if n >= 4096 else "rowpair_kernel<ROW_JAC>") if n <= 8192 else "rowpair2l_jac_kernel"}
    roofline = {
        "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
        "traffic": traffic, "traffic_source": traffic_src, "kernel": names[dominant],
        "algo_bytes_per_launch": (ALGO_BYTES_COL if dominant == "col" else ALGO_BYTES_ROW) * pts,
        "peak_source": peak_src,
        "kernels": {
            "col_step": {"avg_ms": col_avg, "launches": prof["col_launches"], "algo_bytes_per_pt": ALGO_BYTES_COL,
                         "gbs": col_gbs, "frac": col_gbs / peak},
            "row_jac": {"avg_ms": row_avg, "launches": prof["row_launches"], "algo_bytes_per_pt": ALGO_BYTES_ROW,
                        "gbs": row_gbs, "frac": row_gbs / peak},
        },
        "whole_step": {"algo_bytes_per_pt_step": ALGO_BYTES_PER_PT_STEP, "gbs": step_gbs, "frac": step_gbs / peak},
    }

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        cpu = cpu_baseline(args.cpu_grid, args.cpu_steps)

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {
            "workload": f"elliptic vortex {n}^2 RK4 step, dt={dt:g}s, {args.members} member(s) per GPU"
                        + (f", {world} GPUs x independent members (ensemble sharding)" if world > 1 else ""),
            "grid": n, "members_per_gpu": args.members, "dt": dt,
            "l2": "working set (8 spectral arrays, %.1f GB) is larger than the 126 MB L2" % (8 * 8 * (n // 2 + 4) * n * args.members / 1e9),
            "state_finite": finite,
        },
        "clocks": clocks,
        "gpu_launches": int(launches),
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": 4 * G * args.members,
                "d2h_bytes_per_step": 4 * G * args.members, "steps": K * e2e_steps, "ms_per_step": e2e_ms_per_step,
                "requests_in_flight": K, "results_identical": same,
                "serial": {"value": e2e_serial, "ms_per_step": ms_serial / e2e_steps, "steps": e2e_steps, "requests_in_flight": 1}},
        "roofline": roofline,
        "timing": {"value_region": "K steps of xfb_step on its default path (the 8 launches of a step replayed from a CUDA graph)",
                   "bracketed_region_ms_per_step": ms_bracketed / args.steps,
                   "bracketed_region": "the same K steps with every launch bracketed by CUDA events (eager launches); source of "
                                       "roofline.kernels[*].avg_ms"},
    }
    if cpu is not None:
        line["cpu_baseline"] = cpu
    print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


def slab_arm(args):
    """N > 1 (or --slab): ONE grid slab-decomposed over the GPUs (one rank per GPU, NVLink all-to-all per 2-D transform);
    strong scaling.  Same JSON contract; the work is tools/slab_bench.py."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import slab_bench
    a = argparse.Namespace(grid=args.grid, steps=args.steps, warmup=args.warmup, chunks=args.chunks, no_check=args.no_slab_check,
                           no_ensemble=args.no_ensemble_record, field="const" if args.grid >= 16384 else "elliptic",
                           e2e_steps=max(1, min(args.e2e_steps, 3)))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    sampler = ClockSampler(physical_gpu_index(local_rank))
    sampler.start()
    r = slab_bench.run(a)
    clocks = sampler.stop()
    if r is None:
        return
    peak, peak_src = measured_peaks()
    world = r["n_gpus"]
    line = {
        "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": f"{r['field']} vortex {args.grid}^2 RK4 step slab-decomposed over {world} GPU(s), dt={r['dt']:g}s, "
                               f"{args.chunks} chunks, transport {r['transport']}",
                   "grid": args.grid, "l2": "per-rank working set is larger than the 126 MB L2", "state_finite": r["state_finite"],
                   "check_vs_single_gpu": r.get("check"), "limiter": r["limiter"]},
        "clocks": clocks, "gpu_launches": r["gpu_launches_per_rank"] * world,
        "e2e": {k: r["e2e"][k] for k in ("value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step", "steps", "ms_per_step")},
        "roofline": {"bound": "hbm", "achieved": ALGO_BYTES_PER_PT_STEP * r["value"] / world / 1e9, "peak": peak, "unit": "GB/s",
                     "frac": ALGO_BYTES_PER_PT_STEP * r["value"] / world / 1e9 / peak, "traffic": None,
                     "kernel": "whole step per rank (K-ROW + K-COL + exchange)", "peak_source": peak_src,
                     "kernels": r["kernels"]},
        "nvlink": {"bytes_per_gpu_per_step": r["a2a"]["nvlink_bytes_per_gpu_per_step"],
                   "comm_stream_bytes_per_gpu_per_step": r["a2a"]["comm_stream_bytes_per_gpu_per_step"],
                   "a2a_ms_per_step_on_comm_stream": r["a2a"]["ms_per_step_on_comm_stream"],
                   "comm_stream_gbs_per_direction": r["a2a"]["comm_stream_gbs_per_direction"],
                   "whole_step_gbs_per_direction": r["a2a"]["whole_step_gbs_per_direction"],
                   "peak_gbs": 770.0, "peak_source": "B200_PROFILING.md measured peer copy",
                   "frac_of_peak_whole_step": (r["a2a"]["whole_step_gbs_per_direction"] or 0.0) / 770.0},
        "t1": r.get("t1"), "parallel_efficiency": r.get("parallel_efficiency"),
        "ensemble": r.get("ensemble"),
    }
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="xfb", choices=["xfb", "reference"])
    ap.add_argument("--grid", type=int, default=None, help="default 8192 at N = 1, 16384 (slab-decomposed) at N > 1")
    ap.add_argument("--members", type=int, default=1, help="ensemble members per GPU")
    ap.add_argument("--e2e-steps", type=int, default=10)
    ap.add_argument("--e2e-inflight", type=int, default=4, help="independent requests in flight in the end-to-end measurement")
    ap.add_argument("--ref-grid", type=int, default=0, help="grid of the CPU arm (default: the product arm's grid; the "
                                                            "cpu_baseline leg inside the N = 1 product run uses --cpu-grid)")
    ap.add_argument("--ref-budget", type=float, default=150.0, help="--impl reference: seconds the timed run may take")
    ap.add_argument("--cpu-grid", type=int, default=4096, help="grid of the bounded cpu_baseline sample inside the product run")
    ap.add_argument("--cpu-steps", type=int, default=8)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--slab", action="store_true", help="force the slab-decomposed arm (the default for N > 1)")
    ap.add_argument("--ensemble", action="store_true", help="N > 1: independent members, one per GPU, as the headline")
    ap.add_argument("--chunks", type=int, default=8, help="slab arm: chunks of the compute/exchange overlap")
    ap.add_argument("--no-slab-check", action="store_true", help="slab arm: skip the in-run check against the single-GPU path and T1")
    ap.add_argument("--no-ensemble-record", action="store_true", help="slab arm: skip the ensemble sub-record")
    ap.add_argument("--dump-outputs", metavar="DIR", help="single-GPU arm: after the timed steps, write the fields they "
                                                          "computed to DIR/<field>.npy (float32, at most 64 MB in all), "
                                                          "e.g. bench_outputs")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    # ONE JSON line on stdout: libraries write there too (NCCL prints "NCCL version ..." when NCCL_DEBUG is set), so the
    # process-level stdout goes to stderr while the bench runs and the JSON line is written to the real stdout at the end
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(real_stdout, "w")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    slab = args.slab or ((world > 1 or args.gpus > 1) and not args.ensemble)
    if args.grid is None:
        args.grid = 16384 if slab else 8192
    if args.dump_outputs and (slab or args.impl == "reference"):
        ap.error("--dump-outputs is supported by the single-GPU product arm only")
    if args.impl == "reference":
        reference_arm(args)
    elif slab:
        slab_arm(args)
    else:
        gpu_arm(args)


if __name__ == "__main__":
    main()

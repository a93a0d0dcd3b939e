#!/usr/bin/env python
"""slab_bench.py -- one large grid slab-decomposed over the GPUs of a node (one process per GPU, NVLink all-to-all).

This is what `bench.py --gpus N` runs for N > 1 (BASELINE.json configs[4]: 16384^2 constant vortex on 1/2/4/8 B200,
strong scaling); it can also be launched directly:

  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
      tools/slab_bench.py --grid 16384 --steps 10 --warmup 3

In one run, in this order:
  1. CHECK on the benchmark grid itself (same kernel family): an analytic elliptical Gaussian vortex (strongly nonlinear,
     |U| ~ 70 m/s) is advanced 2 RK4 steps by the single-GPU path on rank 0 and by the slab path on all ranks; the
     gathered slab rows must agree with the single-GPU field (relative L2 reported; both sides are this repo's kernels --
     the comparison with the CPU oracle lives in tests/test_headline_parity.py).
  2. T1: the single-GPU time per step at this grid, measured on rank 0 right after the check (CUDA events), so that
     parallel_efficiency = T1 / (N * T_N) is computed from numbers of the same run on the same box.
  3. the timed slab run (W warm-up steps, exactly K timed steps, barrier + synchronise on both sides, max over ranks).
  4. end-to-end through the C ABI with HOST buffers (every step uploads this rank's rows and reads them back).
  5. an ensemble sub-record: one independent 8192^2 member per GPU, no communication (BASELINE.json configs[3]-style
     sharding), a few steps -- context for the slab number, not the headline.
Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

LX = 600000.0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--grid", type=int, default=16384)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--chunks", type=int, default=8)
    ap.add_argument("--no-check", action="store_true")
    ap.add_argument("--no-ensemble", action="store_true")
    ap.add_argument("--field", default="const", choices=["const", "elliptic"])
    ap.add_argument("--e2e-steps", type=int, default=3)
    args = ap.parse_args()
    res = run(args)
    if res is not None:
        print(json.dumps(res))


def analytic_vortex_rows(torch, n, r0, r1, dev):
    """rows [r0, r1) of zeta = 5e-3 exp(-((x-x0)/a)^2 - ((y-y0)/b)^2), a = 40 km, b = 25 km, float32, on `dev`"""
    x = (torch.arange(r0, r1, device=dev, dtype=torch.float32) * (LX / n))[:, None]
    y = (torch.arange(0, n, device=dev, dtype=torch.float32) * (LX / n))[None, :]
    return (5e-3 * torch.exp(-((x - 0.5 * LX) / 40000.0) ** 2 - ((y - 0.45 * LX) / 25000.0) ** 2)).contiguous()


def run(args):
    """-> result dict on rank 0, None elsewhere (called by bench.py for N > 1)"""
    import torch
    import torch.distributed as dist
    import fields
    import xlab_fftbarotropic_b200 as xfb

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1 and not dist.is_initialized():
        dist.init_process_group("nccl", device_id=dev)

    def new_id():
        t = torch.zeros(128, dtype=torch.uint8, device=dev)
        if rank == 0:
            t.copy_(torch.frombuffer(bytearray(xfb.nccl_unique_id()), dtype=torch.uint8))
        if world > 1:
            dist.broadcast(t, 0)
        return bytes(t.cpu().numpy().tobytes())

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    n = args.grid
    G = float(n) * n
    rows = n // world
    r0 = rank * rows
    dt_strong = float(np.float32(0.6 * 2.83 / (0.943 * np.pi * n / LX * 83.0)))     # RK4 advective limit, SURVEY 8(d)
    result = {"n_gpus": world, "chunks": args.chunks}

    sb = xfb.SlabBackend(n, rank, world, new_id(), nchunks=args.chunks, device=local_rank)
    transport = sb.transport
    fused_rows = bool(sb.fused)
    stream = torch.cuda.ExternalStream(sb.stream, device=local_rank)

    # ---- 1 + 2: check against the single-GPU path on THIS grid, and T1 -----------------------------------------------
    if not args.no_check and world > 1:
        check_steps = 2
        mine = analytic_vortex_rows(torch, n, r0, r0 + rows, dev)
        sb.set_vorticity(int(mine.data_ptr()))
        sb.step(check_steps, dt_strong)
        out = torch.empty_like(mine)
        sb._ck(sb._L.xfb_get_field(sb._h, 0, xfb.capi.VORT, int(out.data_ptr())))
        sb.sync()
        del mine
        ref = None
        t1_ms = None
        if rank == 0:
            one = xfb.Backend(n, device=local_rank)
            full = analytic_vortex_rows(torch, n, 0, n, dev)
            one.set_vorticity(int(full.data_ptr()))
            one.step(check_steps, dt_strong)
            ref = torch.empty_like(full)
            one._ck(one._L.xfb_get_field(one._h, 0, xfb.capi.VORT, int(ref.data_ptr())))
            one.sync()
            del full
            # T1 on the same handle: 1 more warm-up step, then 3 timed steps (CUDA events on the library's stream)
            s1 = torch.cuda.ExternalStream(one.stream, device=local_rank)
            one.step(1, dt_strong)
            one.sync()
            a, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            with torch.cuda.stream(s1):
                a.record(s1)
                one.step(3, dt_strong)
                b_.record(s1)
            one.sync()
            t1_ms = a.elapsed_time(b_) / 3
            one.close()
        # gather the slab rows on rank 0 (device), compare there
        if rank == 0:
            parts = [torch.empty_like(out) for _ in range(world)]
            dist.gather(out, parts, dst=0)
            full_slab = torch.cat(parts, 0)
            del parts
            num = torch.linalg.vector_norm((full_slab.double() - ref.double()).flatten()).item()
            den = torch.linalg.vector_norm(ref.double().flatten()).item()
            finite = bool(torch.isfinite(full_slab).all().item())
            err = num / den
            result["check"] = {"grid": n, "field": "analytic elliptical Gaussian vortex, zeta0 = 5e-3 1/s", "steps": check_steps,
                               "dt": dt_strong, "rel_l2_slab_vs_single_gpu": err, "finite": finite,
                               "ok": bool(finite and err < 2e-6),
                               "kernels": "the same K-ROW / K-COL instances the timed run uses (line length %d)" % n}
            result["t1"] = {"ms_per_step": t1_ms, "grid": n, "steps": 3,
                            "note": "single-GPU path on rank 0 of this run, other ranks idle"}
            del full_slab, ref
        else:
            dist.gather(out, None, dst=0)
        del out
        torch.cuda.empty_cache()
        barrier()

    # ---- 3: the timed run -------------------------------------------------------------------------------------------
    gen = fields.const_vortex if args.field == "const" else fields.elliptic
    dt = 3.0 if args.field == "const" else dt_strong
    mine = torch.from_numpy(gen(n, rows=(r0, r0 + rows))).to(dev)           # every rank generates its own rows
    sb.set_vorticity(int(mine.data_ptr()))
    sb.step(args.warmup, dt)
    sb.sync()
    sb.profile(True)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = sb.launch_count
    with torch.cuda.stream(stream):
        e0.record(stream)
        h0 = time.perf_counter()
        sb.step(args.steps, dt)
        host_enqueue_ms = (time.perf_counter() - h0) * 1e3
        e1.record(stream)
    barrier()
    ms = e0.elapsed_time(e1)
    prof = sb.profile_read()
    a2a = sb.a2a_read() if world > 1 else {"a2a_ms": 0.0, "exchanges": 0}
    sb.profile(False)
    launches = sb.launch_count - l0
    if world > 1:
        t = torch.tensor([ms, a2a["a2a_ms"], prof["row_ms"], prof["col_ms"]], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, a2a_ms, row_ms, col_ms = (float(x) for x in t)
    else:
        a2a_ms, row_ms, col_ms = 0.0, prof["row_ms"], prof["col_ms"]
    out = sb.get_field(xfb.capi.VORT)
    finite = torch.tensor([1.0 if bool(np.isfinite(out).all()) else 0.0], device=dev)
    if world > 1:
        dist.all_reduce(finite, op=dist.ReduceOp.MIN)
    finite = bool(finite.item() > 0.5)

    # ---- 4: end to end with host buffers ----------------------------------------------------------------------------
    e2e_steps = max(1, getattr(args, "e2e_steps", 3))
    host_in = mine.cpu().pin_memory()
    host_out = torch.empty_like(host_in).pin_memory()
    hin, hout = int(host_in.data_ptr()), int(host_out.data_ptr())
    sb.set_vorticity(host_in.numpy())
    sb.step(1, dt)
    barrier()
    with torch.cuda.stream(stream):
        e0.record(stream)
        for _ in range(e2e_steps):
            sb._ck(sb._L.xfb_set_vorticity(sb._h, 0, hin))
            sb.step(1, dt)
            sb._ck(sb._L.xfb_get_field(sb._h, 0, xfb.capi.VORT, hout))
        e1.record(stream)
    barrier()
    ms_e2e = e0.elapsed_time(e1)
    if world > 1:
        t2 = torch.tensor([ms_e2e], device=dev)
        dist.all_reduce(t2, op=dist.ReduceOp.MAX)
        ms_e2e = float(t2[0])
    sb.close()
    del mine
    torch.cuda.empty_cache()

    # ---- 5: ensemble sub-record -----------------------------------------------------------------------------------------
    ens = None
    if not args.no_ensemble:
        ne, es = 8192, 5
        b = xfb.Backend(ne, device=local_rank)
        v = analytic_vortex_rows(torch, ne, 0, ne, dev)
        b.set_vorticity(int(v.data_ptr()))
        dte = float(np.float32(0.6 * 2.83 / (0.943 * np.pi * ne / LX * 83.0)))
        b.step(3, dte)
        b.sync()
        se = torch.cuda.ExternalStream(b.stream, device=local_rank)
        barrier()
        with torch.cuda.stream(se):
            e0.record(se)
            b.step(es, dte)
            e1.record(se)
        barrier()
        tm = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        b.close()
        ens = {"value": float(ne) * ne * world * es / (float(tm[0]) * 1e-3), "unit": "grid-pt*steps/s", "scaling": "weak",
               "workload": f"one independent {ne}^2 member per GPU, no communication", "steps": es,
               "ms_per_step": float(tm[0]) / es}

    if rank == 0:
        value = G * args.steps / (ms * 1e-3)
        per_step = ms / args.steps
        # SURVEY 8(e): 20 spectral arrays (~4 B per grid point each) cross per step; per GPU and direction
        nv_total = 20.0 * 4.0 * G / world * (world - 1) / world if world > 1 else 0.0
        # what the communication stream itself carries: the row->column array of each stage is stored into peer memory
        # by K-ROW (fused), so only the four column->row arrays per stage remain there
        nv_comm = nv_total * (16.0 + (0.0 if fused_rows else 4.0)) / 20.0
        a2a_step = a2a_ms / args.steps
        if world > 1:
            if a2a_step > 0.75 * per_step:
                limiter = (f"NVLink exchange: the communication stream is busy {a2a_step:.2f} of {per_step:.2f} ms per step "
                           f"({nv_comm / 1e9:.2f} GB per GPU and direction)")
            else:
                limiter = (f"per-rank kernels (K-ROW spans {row_ms / args.steps:.2f} ms + K-COL spans {col_ms / args.steps:.2f} ms per step "
                           f"incl. waits; exchange {a2a_step:.2f} ms on the communication stream)")
        else:
            limiter = "single-GPU kernels"
        result.update({
            "metric": "rk4_grid_point_steps_per_s", "value": value, "unit": "grid-pt*steps/s", "grid": n, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": per_step, "scaling": "strong", "field": args.field, "dt": dt,
            "state_finite": finite, "gpu_launches_per_rank": int(launches), "transport": transport,
            "host_enqueue_ms_per_step": host_enqueue_ms / args.steps, "limiter": limiter,
            "a2a": {"ms_per_step_on_comm_stream": a2a_step, "exchanges": a2a["exchanges"],
                    "nvlink_bytes_per_gpu_per_step": nv_total, "comm_stream_bytes_per_gpu_per_step": nv_comm,
                    "comm_stream_gbs_per_direction": (nv_comm / (a2a_step * 1e-3) / 1e9) if a2a_step > 0 else None,
                    "whole_step_gbs_per_direction": nv_total / (per_step * 1e-3) / 1e9 if world > 1 else None},
            "kernels": {"row_ms_per_step": row_ms / args.steps, "col_ms_per_step": col_ms / args.steps,
                        "note": "spans on the compute stream, including the wait for their exchanges"},
            "e2e": {"value": G * e2e_steps / (ms_e2e * 1e-3), "unit": "grid-pt*steps/s", "steps": e2e_steps,
                    "ms_per_step": ms_e2e / e2e_steps, "h2d_bytes_per_step": 4 * G, "d2h_bytes_per_step": 4 * G},
        })
        if "t1" in result and result["t1"]["ms_per_step"]:
            result["parallel_efficiency"] = result["t1"]["ms_per_step"] / (world * per_step)
        if ens is not None:
            result["ensemble"] = ens
    if world > 1:
        dist.destroy_process_group()
    return result if rank == 0 else None


if __name__ == "__main__":
    main()

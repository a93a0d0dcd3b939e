"""Slab decomposition (SURVEY.md 8e): host arithmetic and the exchange indexing on CPU, the real kernels on GPU.

CPU (`-m "not gpu"`):
  * xfb_slab_partition covers every row and column exactly once;
  * a numpy model of the panel / chunk layouts of csrc/xfb_dist.cu (row_off / col_off) run by TWO gloo ranks:
    local r2c along y -> all-to-all -> c2c along x must equal numpy's rfft2 of the full field, and back.
GPU (`-m gpu`): the loopback team (all ranks on one device, same kernels and indexing as the NCCL path) must
reproduce the single-GPU backend to float32 rounding (the same butterflies in the same order; the slab
instantiation of K-ROW is a different template instance, so the compiler's FMA contraction may differ).
"""
import os
import socket
import sys

import numpy as np
import pytest

import fields
from conftest import rel_l2

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("n,p,c", [(256, 2, 1), (512, 4, 2), (1024, 8, 4), (16384, 8, 4), (8192, 2, 4)])
def test_partition_covers_grid(n, p, c):
    import xlab_fftbarotropic_b200 as xfb
    parts = [xfb.slab_partition(n, n, p, c, r) for r in range(p)]
    assert sum(q["rows"] for q in parts) == n
    assert [q["row0"] for q in parts] == [r * (n // p) for r in range(p)]
    assert all(q["rows"] % (2 * c) == 0 for q in parts), "row pairs and row chunks stay on one rank"
    cw = parts[0]["chunk_cols"]
    assert cw % 4 == 0 and all(q["chunk_cols"] == cw and q["cols"] == c * cw for q in parts)
    assert [q["col0"] for q in parts] == [r * c * cw for r in range(p)]
    assert parts[0]["pitch_global"] == p * c * cw >= n // 2 + 1
    assert parts[0]["pitch_global"] - (n // 2 + 1) < 4 * p * c + 4, "padding stays small"


@pytest.mark.parametrize("nx,ny,p,c", [(512, 2048, 4, 2), (2048, 256, 2, 4), (256, 1024, 8, 1), (16384, 1024, 8, 4),
                                       (16384, 256, 8, 8), (256, 16384, 2, 16)])
def test_partition_covers_rectangular_grid(nx, ny, p, c):
    """rows come from nx, columns (of the ny / 2 + 1 wide half spectrum) from ny"""
    import xlab_fftbarotropic_b200 as xfb
    parts = [xfb.slab_partition(nx, ny, p, c, r) for r in range(p)]
    assert sum(q["rows"] for q in parts) == nx
    assert [q["row0"] for q in parts] == [r * (nx // p) for r in range(p)]
    assert all(q["rows"] % (2 * c) == 0 for q in parts)
    cw = parts[0]["chunk_cols"]
    assert cw % 4 == 0 and all(q["chunk_cols"] == cw and q["cols"] == c * cw for q in parts)
    assert [q["col0"] for q in parts] == [r * c * cw for r in range(p)]
    assert parts[0]["pitch_global"] == p * c * cw >= ny // 2 + 1
    assert parts[0]["pitch_global"] - (ny // 2 + 1) < 4 * p * c + 4
    # the transposed grid splits its own rows and columns
    t = xfb.slab_partition(ny, nx, p, c, 0)
    assert t["rows"] == ny // p and t["pitch_global"] >= nx // 2 + 1


def test_partition_rejects_bad_arguments():
    import xlab_fftbarotropic_b200 as xfb
    with pytest.raises(xfb.XfbError):
        xfb.slab_partition(256, 256, 3, 1, 0)          # 256 rows do not split into 3 x pairs
    with pytest.raises(xfb.XfbError):
        xfb.slab_partition(256, 256, 2, 1, 2)          # rank out of range


# ---- numpy model of the exchange, run by two gloo ranks ------------------------------------------------
def _row_off(q, c, r0, C, rows, cw):
    return ((q * C + c) * rows + r0) * cw


def _col_off(q, c, r0, C, rows, cw, nx):
    return (c * nx + q * rows + r0) * cw


def _slab_worker(rank, world, port, n, C, out):
    import torch
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    import xlab_fftbarotropic_b200 as xfb
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    part = xfb.slab_partition(n, n, world, C, rank)
    rows, cw, pg = part["rows"], part["chunk_cols"], part["pitch_global"]
    full = fields.elliptic(n).astype(np.float64)
    mine = full[part["row0"]:part["row0"] + rows]
    # K-ROW: y transform of the local rows, written into panels (q, c) = [rows][cw] (pair interleave is a
    # permutation inside a block and does not change which block an element is in)
    y = np.zeros((rows, pg), np.complex128)
    y[:, :n // 2 + 1] = np.fft.rfft(mine, axis=1)
    row_side = np.zeros(world * C * rows * cw, np.complex128)
    for q in range(world):
        for c in range(C):
            o = _row_off(q, c, 0, C, rows, cw)
            row_side[o:o + rows * cw] = y[:, (q * C + c) * cw:(q * C + c + 1) * cw].ravel()
    # all-to-all: block (q, c) goes to rank q and lands in chunk c, rows block `rank`
    col_side = np.zeros(C * n * cw, np.complex128)
    send = [torch.from_numpy(np.concatenate([row_side[_row_off(q, c, 0, C, rows, cw):_row_off(q, c, 0, C, rows, cw) + rows * cw]
                                             for c in range(C)]).view(np.float64).copy()) for q in range(world)]
    # grouped point-to-point like the ncclSend/ncclRecv group of xfb_dist.cu; the own block is a local copy
    recv = [torch.empty_like(send[0]) for _ in range(world)]
    recv[rank].copy_(send[rank])
    ops = []
    for q in range(world):
        if q != rank:
            ops.append(dist.P2POp(dist.isend, send[q], q))
            ops.append(dist.P2POp(dist.irecv, recv[q], q))
    for w in dist.batch_isend_irecv(ops):
        w.wait()
    for q in range(world):
        blk = recv[q].numpy().view(np.complex128)
        for c in range(C):
            o = _col_off(q, c, 0, C, rows, cw, n)
            col_side[o:o + rows * cw] = blk[c * rows * cw:(c + 1) * rows * cw]
    # K-COL: x transform of each chunk [n][cw]
    spec = np.concatenate([np.fft.fft(col_side[c * n * cw:(c + 1) * n * cw].reshape(n, cw), axis=0) for c in range(C)], axis=1)
    ref = np.zeros((n, pg), np.complex128)
    ref[:, :n // 2 + 1] = np.fft.rfft2(full)
    err = np.abs(spec - ref[:, part["col0"]:part["col0"] + C * cw]).max() / np.abs(ref).max()
    out.put((rank, float(err)))
    dist.destroy_process_group()


@pytest.mark.parametrize("n,P,C", [(64, 2, 1), (128, 4, 2), (256, 8, 4)])
def test_fused_panel_table_is_the_transpose(n, P, C):
    """Fused row -> column exchange (csrc/xfb_dist.cu build_panel_table, xfb_row.cuh out_addr): every rank stores
    output element (local row r, global column k) at  panel_base[k // cw] + r * cw + k % cw  with
    panel_base[q * C + c] = receive array of rank q + col_off(me, c, 0).  A numpy model of exactly that addressing
    must give every rank the x-transformable chunks [n][cw] of numpy's rfft2."""
    import xlab_fftbarotropic_b200 as xfb
    parts = [xfb.slab_partition(n, n, P, C, r) for r in range(P)]
    rows, cw, pg = parts[0]["rows"], parts[0]["chunk_cols"], parts[0]["pitch_global"]
    full = fields.elliptic(n).astype(np.float64)
    recv = [np.zeros(C * n * cw, np.complex128) for _ in range(P)]          # jint_recv of every rank
    for me in range(P):
        y = np.zeros((rows, pg), np.complex128)
        y[:, :n // 2 + 1] = np.fft.rfft(full[parts[me]["row0"]:parts[me]["row0"] + rows], axis=1)
        table = [(q, _col_off(me, c, 0, C, rows, cw, n)) for q in range(P) for c in range(C)]   # panel -> (rank, offset)
        for r in range(rows):
            for panel in range(P * C):
                q, base = table[panel]
                recv[q][base + r * cw:base + (r + 1) * cw] = y[r, panel * cw:(panel + 1) * cw]
    ref = np.zeros((n, pg), np.complex128)
    ref[:, :n // 2 + 1] = np.fft.rfft2(full)
    for q in range(P):
        spec = np.concatenate([np.fft.fft(recv[q][c * n * cw:(c + 1) * n * cw].reshape(n, cw), axis=0) for c in range(C)], axis=1)
        err = np.abs(spec - ref[:, parts[q]["col0"]:parts[q]["col0"] + C * cw]).max() / np.abs(ref).max()
        assert err < 1e-12, (q, err)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


@pytest.mark.parametrize("n,C", [(64, 1), (128, 2)])
def test_exchange_indexing_two_gloo_ranks(n, C):
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_slab_worker, args=(r, 2, port, n, C, out)) for r in range(2)]
    for p in procs:
        p.start()
    res = [out.get(timeout=120) for _ in procs]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for rank, err in res:
        assert err < 1e-12, f"rank {rank}: slab 2-D transform differs from rfft2 by {err}"


# ---- GPU: loopback team against the single-GPU backend ----------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n,p,c", [(256, 2, 1), (512, 4, 2), (1024, 2, 4), (512, 8, 1)])
def test_loopback_team_matches_single_gpu(n, p, c):
    import xlab_fftbarotropic_b200 as xfb
    v0 = fields.kuo2004(n) if hasattr(fields, "kuo2004") else fields.elliptic(n)
    rng = np.random.default_rng(n + p)
    src = (1e-9 * rng.standard_normal((n, n))).astype(np.float32)
    one = xfb.Backend(n)
    team = xfb.LoopbackTeam(n, p, c)
    one.set_vorticity(v0)
    team.set_vorticity(v0)
    one.set_source(src)
    team.set_source(src)
    one.step(3, 3.0)
    team.step(3, 3.0)
    for which in (xfb.capi.VORT, xfb.capi.PSI, xfb.capi.U, xfb.capi.V, xfb.capi.DEFORM):
        a, b = one.get_field(which), team.get_field(which)
        # the deformation factor is a ratio of differences of second derivatives, formed by the fused float32
        # multipliers on one GPU and by the operator tables on the slab path: north_star's 1e-5 instead of the 2e-6
        # asked of the state fields (pointwise it is a ratio of small numbers where the flow is at rest)
        tol = 1e-5 if which == xfb.capi.DEFORM else 2e-6
        assert rel_l2(b, a) < tol, f"field {which}: {rel_l2(b, a)}"
        if which != xfb.capi.DEFORM:
            assert np.abs(a - b).max() <= 10 * tol * np.abs(a).max(), f"field {which}"
    # stepping again after the record fields were taken (the prologue is redone)
    one.step(1, 3.0)
    team.step(1, 3.0)
    a, b = one.get_field(xfb.capi.VORT), team.get_field(xfb.capi.VORT)
    assert rel_l2(b, a) < 2e-6
    assert team.launch_count > 0
    one.close()
    team.close()


@pytest.mark.gpu
def test_loopback_diagnostics_and_keff_histograms():
    """slab handles: both strain diagnostics from one set of second derivatives, and the effective-diffusivity histograms
    binned per rank and summed over the ranks (the ncclAllReduce of the multi-process path is the shared accumulator of
    the loopback team), against the single-GPU results"""
    import xlab_fftbarotropic_b200 as xfb
    n, p, c = 512, 4, 2
    v0 = fields.elliptic(n)
    one = xfb.Backend(n)
    team = xfb.LoopbackTeam(n, p, c)
    one.set_vorticity(v0)
    team.set_vorticity(v0)
    one.step(2, 3.0)
    team.step(2, 3.0)
    t1, d1 = one.diagnostics()
    t2, d2 = team.diagnostics()
    assert rel_l2(d2, d1) < 1e-5
    clear = np.abs(d1) > 1e-4
    assert np.array_equal((t2 > 0)[clear], (t1 > 0)[clear])
    well = (d1 >= 0.05) & (t1 > 0) & (t2 > 0)
    assert well.mean() > 0.3 and rel_l2(t2[well], t1[well]) < 1e-5
    lo, hi = float(v0.min()) - 1e-6, float(v0.max()) * 1.01
    a1, g1 = one.keff_hist(64, lo, hi)
    a2, g2 = team.keff_hist(64, lo, hi)
    assert abs(a2.sum() - 600000.0 ** 2) < 1e-6 * 600000.0 ** 2
    assert rel_l2(np.cumsum(a2), np.cumsum(a1)) < 1e-5
    assert rel_l2(np.cumsum(g2), np.cumsum(g1)) < 1e-5
    # the state is untouched by the diagnostics
    one.step(1, 3.0)
    team.step(1, 3.0)
    assert rel_l2(team.get_field(xfb.capi.VORT), one.get_field(xfb.capi.VORT)) < 2e-6
    one.close()
    team.close()


@pytest.mark.gpu
def test_loopback_rejects_field_ids_outside_the_header():
    """xfb_loopback_get_field takes the field ids of include/xfb.h only (XFB_SRC is not a team field): XFB_E_ARG"""
    import xlab_fftbarotropic_b200 as xfb
    n = 256
    team = xfb.LoopbackTeam(n, 2)
    team.set_vorticity(fields.elliptic(n))
    for which in (-1, xfb.capi.SRC, 10, 11, 12, 13):
        with pytest.raises(xfb.XfbError, match="error -1: bad field id"):
            team.get_field(which)
    assert np.isfinite(team.get_field(xfb.capi.TFIL)).all()
    team.close()


@pytest.mark.gpu
def test_loopback_16384_two_level_kernels():
    """the slab path at the grid bench.py measures (BASELINE.json configs[4]): two-level K-ROW fed by one bulk copy per
    panel, two-level K-COL storing this rank's own row pairs straight into its receive arrays (no self-copy in the
    exchange) -- against the single-GPU path, bit for bit (same kernels, same arithmetic)"""
    import xlab_fftbarotropic_b200 as xfb
    n, p, c = 16384, 2, 4
    x = (np.arange(n, dtype=np.float32) / n)
    v0 = (5e-3 * np.exp(-((x[:, None] - 0.5) / 0.07) ** 2 - ((x[None, :] - 0.45) / 0.04) ** 2)).astype(np.float32)
    one = xfb.Backend(n)
    one.set_vorticity(v0)
    one.step(2, 0.25)
    ref = one.get_field(xfb.capi.VORT)
    one.close()
    team = xfb.LoopbackTeam(n, p, c)
    team.set_vorticity(v0)
    team.step(2, 0.25)
    got = team.get_field(xfb.capi.VORT)
    team.close()
    assert np.isfinite(got).all()
    assert rel_l2(got, ref) < 2e-6, rel_l2(got, ref)


@pytest.mark.gpu
@pytest.mark.parametrize("n,p,c", [(512, 2, 2), (1024, 4, 1)])
def test_loopback_passive_tracer(n, p, c):
    """the passive tracer on slab handles: its tendency and its two gradient products cross the ranks through three more
    receive arrays; (i) a tracer equal to the vorticity with kappa = nu stays bit-identical to the vorticity the same team
    computes, (ii) an independent tracer matches the single-GPU tracer"""
    import xlab_fftbarotropic_b200 as xfb
    v0 = fields.kuo2004(n)
    c0 = fields.gaussian(n)
    team = xfb.LoopbackTeam(n, p, c)
    team.set_vorticity(v0)
    team.set_tracer(v0, 6.5)
    team.step(3, 3.0)
    assert np.array_equal(team.get_field(xfb.capi.TRACER), team.get_field(xfb.capi.VORT))
    team.set_vorticity(v0)
    team.set_tracer(c0, 20.0)
    team.step(3, 3.0)
    got = team.get_field(xfb.capi.TRACER)
    team.close()
    one = xfb.Backend(n)
    one.set_vorticity(v0)
    one.set_tracer(c0, 20.0)
    one.step(3, 3.0)
    ref = one.get_field(xfb.capi.TRACER)
    one.close()
    assert rel_l2(got, ref) < 2e-6, rel_l2(got, ref)

"""Quadratic invariants and isotropic shell spectra of the state (xfb_get_energy_spectrum, DESIGN.md section 3).

CPU: the shell rule and the definitions, pinned on the oracle's spectrum against its physical fields (Parseval).
GPU (`-m gpu`): every state layout against a float64 numpy restatement of the definitions applied to get_spectrum(),
ensemble offsets, the tracer, the slab indexing on the loopback team, the absence of side effects, the argument checks
and main.out -E.  Sums over ~10^8 modes in float64 with atomics in any order: totals agree to 1e-10 relative.
"""
import ctypes as C
import math
import os
import subprocess
import tempfile

import numpy as np
import pytest

import fields

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "xlab_fftbarotropic_b200", "bin")
L0 = 600000.0


# ---- float64 numpy restatement of the definitions ----------------------------------------------------------------
def wavenumbers(nx, ny, lx, ly):
    """the handle's float32 tables (fftwfop.cpp:15-24 expressions)"""
    twopi = np.float32(np.float32(np.pi) * np.float32(2.0))
    kx = (twopi * np.arange(nx, dtype=np.float32)) / np.float32(lx)
    kx[nx // 2 + 1:] = -kx[1:nx - nx // 2][::-1]
    ky = (twopi * np.arange(ny // 2 + 1, dtype=np.float32)) / np.float32(ly)
    return kx.astype(np.float32), ky.astype(np.float32)


def shells(nx, ny, lx, ly):
    """shell index of every mode (i, j) of the half spectrum"""
    i = np.arange(nx, dtype=np.int64)
    ip = np.minimum(i, nx - i)
    j = np.arange(ny // 2 + 1, dtype=np.int64)
    lx, ly = float(np.float32(lx)), float(np.float32(ly))
    if lx == ly:
        m = ip[:, None] ** 2 + j[None, :] ** 2
        s = np.floor(np.sqrt(m.astype(np.float64))).astype(np.int64)
        s = np.where(s * s > m, s - 1, s)
        s = np.where((s + 1) * (s + 1) <= m, s + 1, s)
        return s + (m > s * s + s)
    big = max(lx, ly)
    a = ip.astype(np.float64) * (big / lx)
    b = j.astype(np.float64) * (big / ly)
    return np.floor(np.sqrt(a[:, None] * a[:, None] + b[None, :] * b[None, :]) + 0.5).astype(np.int64)


def reference(zh, kx, ky, lx, ly, nshells):
    """(totals [E, Z, P], e, z) of a half spectrum in the reference layout, float64"""
    nx, hy = zh.shape
    ny = 2 * (hy - 1)
    re = zh.real.astype(np.float64)
    im = zh.imag.astype(np.float64)
    w = np.full(hy, 2.0)
    w[0] = w[ny // 2] = 1.0
    zw = (re * re + im * im) * w[None, :]
    k2 = kx.astype(np.float64)[:, None] ** 2 + ky.astype(np.float64)[None, :hy] ** 2
    e = np.where(k2 > 0, zw / np.where(k2 > 0, k2, 1.0), 0.0)
    c = 1.0 / (2.0 * float(nx * ny) ** 2)
    totals = np.array([e.sum(), zw.sum(), (zw * k2).sum()]) * c
    s = shells(nx, ny, lx, ly).ravel()
    keep = s < nshells
    es = np.bincount(s[keep], e.ravel()[keep], minlength=nshells)[:nshells] * c
    zs = np.bincount(s[keep], zw.ravel()[keep], minlength=nshells)[:nshells] * c
    return totals, es, zs


def rel(a, b):
    return abs(a - b) / abs(b)


def physical_parts(zh, kx, ky):
    """E and P as the physical fields u, v, zeta_x, zeta_y of a real transform hold them.  The y-derivative of the
    Nyquist column j = ny/2 and the x-derivative of the two self-conjugate points (nx/2, 0), (nx/2, ny/2) are imaginary
    fields, which c2r drops.  The definitions count every mode; these sums leave out exactly what the fields cannot
    carry (-> Parseval against the fields)."""
    nx, hy = zh.shape
    ny = 2 * (hy - 1)
    w = np.full(hy, 2.0)
    w[0] = w[ny // 2] = 1.0
    zw = (zh.real.astype(np.float64) ** 2 + zh.imag.astype(np.float64) ** 2) * w[None, :]
    kx2 = kx.astype(np.float64)[:, None] ** 2 * np.ones((1, hy))
    ky2 = ky.astype(np.float64)[None, :hy] ** 2 * np.ones((nx, 1))
    kx2[nx // 2, 0] = kx2[nx // 2, ny // 2] = 0.0
    ky2[:, ny // 2] = 0.0
    k2 = kx.astype(np.float64)[:, None] ** 2 + ky.astype(np.float64)[None, :hy] ** 2
    c = 1.0 / (2.0 * float(nx * ny) ** 2)
    ek = np.where(k2 > 0, zw * (kx2 + ky2) / np.where(k2 > 0, k2 * k2, 1.0), 0.0)
    return ek.sum() * c, (zw * (kx2 + ky2)).sum() * c


# ---- CPU -----------------------------------------------------------------------------------------------------------
def test_integer_shell_rule_is_rounded_distance():
    n = 1024
    s = shells(n, n, L0, L0)
    i = np.arange(n)
    ip = np.minimum(i, n - i)
    j = np.arange(n // 2 + 1)
    assert np.array_equal(s, np.round(np.hypot(ip[:, None], j[None, :])).astype(np.int64))


@pytest.mark.parametrize("nx,ny,lx,ly,expect", [(256, 256, L0, L0, 182), (768, 768, L0, L0, 544), (8192, 8192, L0, L0, 5794),
                                                (16384, 16384, L0, L0, 11586), (1024, 768, 600e3, 450e3, None)])
def test_shells_all(nx, ny, lx, ly, expect):
    from xlab_fftbarotropic_b200 import capi
    got = capi.shells_all(nx, ny, lx, ly)
    assert got == shells(nx, ny, lx, ly).max() + 1
    if expect is not None:
        assert got == expect


@pytest.mark.parametrize("n,gen", [(64, "elliptic"), (64, "kuo2004"), (256, "elliptic"), (256, "kuo2004")])
def test_definitions_against_oracle_fields(n, gen):
    from oracle import oracle as orc
    o = orc.Oracle(n)
    o.set_vorticity(fields.GENERATORS[gen](n))
    o.step(3, 3.0)
    zh = o.get_spectrum().reshape(n, n // 2 + 1)
    kx, ky = wavenumbers(n, n, L0, L0)
    nsh = shells(n, n, L0, L0).max() + 1
    tot, e, z = reference(zh, kx, ky, L0, L0, nsh)
    u = o.get_field(orc.U).astype(np.float64)
    v = o.get_field(orc.V).astype(np.float64)
    vort = o.get_field(orc.VORT).astype(np.float64)
    e_phys, p_phys = physical_parts(zh, kx, ky)
    assert e_phys <= tot[0] and p_phys <= tot[2]
    assert rel(e_phys, 0.5 * np.mean(u * u + v * v)) < 1e-5
    assert rel(tot[1], 0.5 * np.mean(vort * vort)) < 1e-5
    z128 = zh.astype(np.complex128)
    zx = np.fft.irfft2(1j * kx.astype(np.float64)[:, None] * z128, s=(n, n))
    zy = np.fft.irfft2(1j * ky.astype(np.float64)[None, :] * z128, s=(n, n))
    assert rel(p_phys, 0.5 * np.mean(zx * zx + zy * zy)) < 1e-5
    # with the Nyquist lines zeroed the fields hold every mode's derivative: the definitions themselves, to 1e-12
    zh0 = zh.copy()
    zh0[n // 2, :] = 0
    zh0[:, n // 2] = 0
    t0 = reference(zh0, kx, ky, L0, L0, 0)[0]
    z0 = zh0.astype(np.complex128)
    ux = np.fft.irfft2(1j * ky.astype(np.float64)[None, :] * z0 / np.where(np.add.outer(kx.astype(np.float64) ** 2, ky.astype(np.float64) ** 2) > 0,
                                                                           np.add.outer(kx.astype(np.float64) ** 2, ky.astype(np.float64) ** 2), 1.0), s=(n, n))
    vx = np.fft.irfft2(1j * kx.astype(np.float64)[:, None] * z0 / np.where(np.add.outer(kx.astype(np.float64) ** 2, ky.astype(np.float64) ** 2) > 0,
                                                                           np.add.outer(kx.astype(np.float64) ** 2, ky.astype(np.float64) ** 2), 1.0), s=(n, n))
    assert rel(t0[0], 0.5 * np.mean(ux * ux + vx * vx)) < 1e-12
    assert rel(t0[1], 0.5 * np.mean(np.fft.irfft2(z0, s=(n, n)) ** 2)) < 1e-12
    assert rel(e.sum(), tot[0]) < 1e-12 and rel(z.sum(), tot[1]) < 1e-12


# ---- GPU -----------------------------------------------------------------------------------------------------------
def _check(got, want, nshells):
    tot, e, z = got
    rt, re_, rz = want
    for k in range(3):
        assert rel(tot[k], rt[k]) < 1e-10, (k, tot[k], rt[k])
    assert len(e) == nshells and len(z) == nshells
    assert np.abs(e - re_).max() <= 1e-10 * rt[0]
    assert np.abs(z - rz).max() <= 1e-10 * rt[1]


def _against_spectrum(b, nshells=None, member=0, which=None):
    import xlab_fftbarotropic_b200 as xfb
    which = xfb.capi.VORT if which is None else which
    got = b.energy_spectrum(nshells, which=which, member=member)
    zh = b.get_spectrum(member)
    kx, ky = b.table(xfb.capi.TAB_GRADX), b.table(xfb.capi.TAB_GRADY)
    n = len(got[1])
    _check(got, reference(zh, kx, ky, b.lx, b.ly, n), n)
    return got


@pytest.mark.gpu
@pytest.mark.parametrize("nx,ny,gen,lx,ly", [(256, 256, "elliptic", L0, L0), (512, 512, "kuo2004", L0, L0),
                                             (1024, 1024, "gaussian", L0, L0), (4096, 4096, "elliptic", L0, L0),
                                             (8192, 8192, "elliptic", L0, L0), (16384, 16384, "const", L0, L0),
                                             (768, 768, "elliptic", L0, L0), (1024, 768, "blob", 600e3, 450e3)])
def test_every_layout_against_float64_reference(nx, ny, gen, lx, ly):
    import xlab_fftbarotropic_b200 as xfb
    if nx == 16384:
        import psutil
        if psutil.virtual_memory().available < 24 * 2 ** 30:
            pytest.skip("the 16384^2 reference needs ~16 GiB of host memory")
    if gen == "blob":
        x = (np.arange(nx) / nx)[:, None]
        y = (np.arange(ny) / ny)[None, :]
        v0 = (1e-4 * np.exp(-((x - 0.45) ** 2 + (y - 0.55) ** 2) / 0.01) * (1 + 0.3 * np.cos(6 * np.pi * x))).astype(np.float32)
    else:
        v0 = fields.GENERATORS[gen](nx)
    b = xfb.Backend(nx, ny, lx=lx, ly=ly)
    b.set_vorticity(v0)
    b.step(2, 3.0 if nx <= 1024 else 0.5)
    full = _against_spectrum(b)
    assert len(full[1]) == xfb.capi.shells_all(nx, ny, lx, ly)
    part = _against_spectrum(b, 17)
    assert np.array_equal(part[0], full[0]) or max(rel(part[0][k], full[0][k]) for k in range(3)) < 1e-12
    b.close()


@pytest.mark.gpu
def test_ensemble_member_offsets():
    import xlab_fftbarotropic_b200 as xfb
    n = 512
    gens = [fields.elliptic(n), fields.kuo2004(n), fields.gaussian(n)]
    b = xfb.Backend(n, batch=3)
    for m, v in enumerate(gens):
        b.set_vorticity(v, member=m)
    b.step(2, 3.0)
    for m, v in enumerate(gens):
        one = xfb.Backend(n)
        one.set_vorticity(v)
        one.step(2, 3.0)
        got, want = b.energy_spectrum(member=m), one.energy_spectrum()
        _check(got, want, len(want[1]))
        _against_spectrum(b, member=m)
        one.close()
    b.close()


@pytest.mark.gpu
@pytest.mark.parametrize("n", [512, 4096])
def test_parseval_on_gpu_fields(n):
    import xlab_fftbarotropic_b200 as xfb
    b = xfb.Backend(n)
    b.set_vorticity(fields.elliptic(n))
    b.step(2, 1.0)
    tot, _, _ = b.energy_spectrum(0)
    e_phys, p_phys = physical_parts(b.get_spectrum(), b.table(xfb.capi.TAB_GRADX), b.table(xfb.capi.TAB_GRADY))
    assert rel(e_phys, tot[0]) < 1e-3 and rel(p_phys, tot[2]) < 1e-2          # the Nyquist lines hold little
    f = {w: b.get_field(w).astype(np.float64) for w in (xfb.capi.U, xfb.capi.V, xfb.capi.VORT, xfb.capi.DVORTDX, xfb.capi.DVORTDY)}
    assert rel(e_phys, 0.5 * np.mean(f[xfb.capi.U] ** 2 + f[xfb.capi.V] ** 2)) < 1e-5
    assert rel(tot[1], 0.5 * np.mean(f[xfb.capi.VORT] ** 2)) < 1e-5
    assert rel(p_phys, 0.5 * np.mean(f[xfb.capi.DVORTDX] ** 2 + f[xfb.capi.DVORTDY] ** 2)) < 1e-5
    b.close()


@pytest.mark.gpu
def test_time_series_against_oracle():
    import xlab_fftbarotropic_b200 as xfb
    from oracle import oracle as orc
    n, dt = 512, 3.0
    v0, src = fields.kuo2004(n), fields.wave_source(n)
    orc.set_threads(0)
    o = orc.Oracle(n)
    o.set_vorticity(v0)
    o.set_source(src)
    b = xfb.Backend(n)
    b.set_vorticity(v0)
    b.set_source(src)
    kx, ky = wavenumbers(n, n, L0, L0)
    for k in range(10):
        o.step(20, dt)
        b.step(20, dt)
        want = reference(o.get_spectrum().reshape(n, n // 2 + 1), kx, ky, L0, L0, 0)[0]
        got = b.energy_spectrum(0)[0]
        for q in range(3):
            assert rel(got[q], want[q]) < 1e-4, (20 * (k + 1), q, got[q], want[q])
    b.close()


def _blob(n, cx=0.42, cy=0.55, r=0.08):
    x = (np.arange(n) / n)[:, None]
    y = (np.arange(n) / n)[None, :]
    return np.exp(-((x - cx) ** 2 + (y - cy) ** 2) / r ** 2).astype(np.float32)


@pytest.mark.gpu
def test_tracer():
    import xlab_fftbarotropic_b200 as xfb
    n = 512
    v0 = fields.elliptic(n)
    b = xfb.Backend(n)
    b.set_vorticity(v0)
    with pytest.raises(xfb.XfbError, match="error -4"):
        b.energy_spectrum(which=xfb.capi.TRACER)
    b.set_tracer(v0, b.nu)
    b.step(5, 3.0)
    tv, ev, zv = b.energy_spectrum()
    tc, ec, zc = b.energy_spectrum(which=xfb.capi.TRACER)
    _check((tc, ec, zc), (tv, ev, zv), len(ev))
    b.close()
    b = xfb.Backend(n)
    b.set_vorticity(v0)
    b.set_tracer(_blob(n), 25.0)
    b.step(5, 3.0)
    c = b.get_field(xfb.capi.TRACER).astype(np.float64)
    assert rel(b.energy_spectrum(0, which=xfb.capi.TRACER)[0][1], 0.5 * np.mean(c * c)) < 1e-5
    b.close()


@pytest.mark.gpu
@pytest.mark.parametrize("n,p,c", [(512, 2, 2), (1024, 4, 1), (16384, 8, 4)])
def test_loopback_slab_indexing(n, p, c):
    """Every rank reduces its own column chunks (global padding columns at 1024 / 4 ranks and 16384 / 8 ranks).  The
    loopback's state equals the single handle's only to float32 rounding (test_slab.py pins it at 2e-6), so the
    totals and shells are compared at 1e-6; a chunk or column offset error moves whole columns and fails far above."""
    import xlab_fftbarotropic_b200 as xfb
    v0 = fields.elliptic(n)
    c0 = _blob(n)
    team = xfb.LoopbackTeam(n, p, c)
    one = xfb.Backend(n)
    team.set_vorticity(v0); one.set_vorticity(v0)
    team.set_tracer(c0, 25.0); one.set_tracer(c0, 25.0)
    for which in (xfb.capi.VORT, xfb.capi.TRACER):
        for nsh in (None, 17):
            tt, et, zt = team.energy_spectrum(nsh, which=which)
            to, eo, zo = one.energy_spectrum(nsh, which=which)
            assert len(et) == len(eo)
            for k in range(3):
                assert rel(tt[k], to[k]) < 1e-6, (which, k, tt[k], to[k])
            assert np.abs(et - eo).max() <= 1e-6 * to[0] and np.abs(zt - zo).max() <= 1e-6 * to[1]
    # the single handle against its own state at 1e-10 (same kernel, single-GPU layout of this size)
    if n <= 1024:
        _against_spectrum(one)
    l0 = team.launch_count
    team.energy_spectrum(0)
    assert team.launch_count - l0 == p                   # one launch per rank
    team.close(); one.close()


@pytest.mark.gpu
def test_no_side_effects_and_launch_count():
    import xlab_fftbarotropic_b200 as xfb
    n = 512
    v0, c0 = fields.kuo2004(n), _blob(n)
    a, b = xfb.Backend(n), xfb.Backend(n)
    for h in (a, b):
        h.set_vorticity(v0)
        h.set_tracer(c0, 25.0)
    for s in range(30):
        a.step(1, 3.0)
        b.step(1, 3.0)
        l0 = a.launch_count
        a.energy_spectrum()
        a.energy_spectrum(17)
        a.energy_spectrum(0, which=xfb.capi.TRACER)
        assert a.launch_count - l0 == 3                   # one launch per call
    assert np.array_equal(a.get_spectrum(), b.get_spectrum())
    assert np.array_equal(a.get_field(xfb.capi.TRACER), b.get_field(xfb.capi.TRACER))
    a.close(); b.close()


@pytest.mark.gpu
def test_argument_and_state_errors():
    import xlab_fftbarotropic_b200 as xfb
    from xlab_fftbarotropic_b200 import capi
    L = capi.load()
    n = 256
    b = xfb.Backend(n, batch=2)
    t = np.zeros(3)
    e = np.zeros(200)
    z = np.zeros(200)
    P = capi._ptr
    assert L.xfb_get_energy_spectrum(b._h, 0, capi.VORT, 0, P(t), None, None) == -4          # before set_vorticity
    b.set_vorticity(fields.elliptic(n))
    call = lambda m, w, k, tt, ee, zz: L.xfb_get_energy_spectrum(b._h, m, w, k, tt, ee, zz)
    assert call(0, capi.VORT, 0, P(t), None, None) == 0
    assert call(0, capi.VORT, 200, P(t), P(e), P(z)) == 0
    for args in [(-1, capi.VORT, 0, P(t), None, None), (2, capi.VORT, 0, P(t), None, None),
                 (0, capi.PSI, 0, P(t), None, None), (0, capi.U, 0, P(t), None, None),
                 (0, capi.VORT, -1, P(t), None, None), (0, capi.VORT, 65537, P(t), P(e), P(z)),
                 (0, capi.VORT, 0, None, None, None), (0, capi.VORT, 5, P(t), None, P(z)), (0, capi.VORT, 5, P(t), P(e), None)]:
        assert call(*args) == -1, args
    assert call(0, capi.TRACER, 0, P(t), None, None) == -4                                   # before set_tracer
    b.close()
    team = xfb.LoopbackTeam(512, 2, 1)
    LT = lambda w, k, tt, ee, zz: L.xfb_loopback_get_energy_spectrum(team._t, w, k, tt, ee, zz)
    assert LT(capi.VORT, 0, P(t), None, None) == -4
    team.set_vorticity(fields.elliptic(512))
    assert LT(capi.TRACER, 0, P(t), None, None) == -4
    assert LT(capi.PSI, 0, P(t), None, None) == -1
    assert LT(capi.VORT, 65537, P(t), P(e), P(z)) == -1
    assert LT(capi.VORT, 0, None, None, None) == -1
    assert LT(capi.VORT, 3, P(t), None, P(z)) == -1
    team.close()


def _run_main(d, n, extra, dt=None, steps=20, rec=5):
    cmd = [os.path.join(BIN, "main.out"), "-n", str(n), "-t", str(steps), "-r", str(rec), "-q", *extra]
    if dt is not None:
        cmd += ["-d", str(dt)]
    return subprocess.run(cmd, cwd=d, capture_output=True, text=True, timeout=600)


def _workdir(base, v0):
    os.makedirs(os.path.join(base, "input"))
    os.makedirs(os.path.join(base, "output"))
    v0.tofile(os.path.join(base, "input", "initial_vorticity.bin"))


@pytest.mark.gpu
def test_main_out_energy_flag():
    n = 256
    v0 = fields.elliptic(n)
    with tempfile.TemporaryDirectory() as d:
        plain, withE = os.path.join(d, "plain"), os.path.join(d, "E")
        _workdir(plain, v0)
        _workdir(withE, v0)
        r0 = _run_main(plain, n, [])
        r1 = _run_main(withE, n, ["-E"])
        assert r0.returncode == 0 and r1.returncode == 0, r1.stderr[-2000:]
        assert r0.stdout == r1.stdout
        log0, log1 = open(os.path.join(plain, "log")).read(), open(os.path.join(withE, "log")).read()
        assert log0 == log1
        for name in sorted(os.listdir(os.path.join(plain, "output"))):
            with open(os.path.join(plain, "output", name), "rb") as f0, open(os.path.join(withE, "output", name), "rb") as f1:
                assert f0.read() == f1.read(), name
        assert "integrals.txt" not in os.listdir(os.path.join(plain, "output"))
        rows = np.loadtxt(os.path.join(withE, "output", "integrals.txt"), ndmin=2)
        assert rows.shape == (4, 6)
        assert list(rows[:, 0]) == [0, 5, 10, 15] and (rows[:, 2] == 0).all()
        for step, _, _, E, Z, P in rows:
            step = int(step)
            vort = np.fromfile(os.path.join(withE, "output", f"vort_step_{step}.bin"), dtype="<f4").astype(np.float64)
            assert rel(Z, 0.5 * np.mean(vort * vort)) < 1e-5
            sp = np.loadtxt(os.path.join(withE, "output", f"spectrum_step_{step}.txt"), comments="#")
            from xlab_fftbarotropic_b200 import capi
            assert sp.shape == (capi.shells_all(n, n, L0), 4)
            assert rel(sp[:, 2].sum(), E) < 1e-12 and rel(sp[:, 3].sum(), Z) < 1e-12
        # dt = 300 s: the oracle goes non-finite within 3 steps at 256^2
        blow = os.path.join(d, "blow")
        _workdir(blow, v0)
        r = _run_main(blow, n, ["-E"], dt=300, steps=50, rec=5)
        assert r.returncode == 1
        assert "main.out: non-finite energy/enstrophy at step 5 (member 0)" in r.stderr
        assert os.path.exists(os.path.join(blow, "output", "vort_step_5.bin"))
        assert not os.path.exists(os.path.join(blow, "output", "vort_step_10.bin"))


def _gpu_count():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


@pytest.mark.gpu
def test_main_out_energy_flag_two_gpus():
    if _gpu_count() < 2:
        pytest.skip("needs two GPUs")
    n = 1024
    v0 = fields.kuo2004(n)
    rows = {}
    with tempfile.TemporaryDirectory() as d:
        for tag, extra in (("one", ["-E"]), ("slab", ["-E", "-S", "2"])):
            w = os.path.join(d, tag)
            _workdir(w, v0)
            r = _run_main(w, n, extra, steps=6, rec=3)
            assert r.returncode == 0, r.stderr[-2000:]
            rows[tag] = np.loadtxt(os.path.join(w, "output", "integrals.txt"), ndmin=2)
    assert rows["one"].shape == rows["slab"].shape == (2, 6)
    assert np.array_equal(rows["slab"][:, :3], rows["one"][:, :3])
    # the slab state equals the single-GPU state to float32 rounding (test_host_programs.py: fields at 2e-6)
    np.testing.assert_allclose(rows["slab"][:, 3:], rows["one"][:, 3:], rtol=1e-6, atol=0)

"""GPU checks at BASELINE.json's full sizes (4096^2, 8192^2) that complement the oracle comparisons of
tests/test_headline_parity.py: size-independent properties of the reference algorithm, and forced steps of the default
kernels against their variants and the oracle.

  * KAT-3 linear decay (SURVEY.md section 4): a single mode has zero Jacobian, so one RK4 step multiplies a mode
    inside the dealiasing circle by 1 + z + z^2/2 + z^3/6 + z^4/24, z = -nu |k|^2 dt, and leaves a mode outside
    the circle untouched (the mask is applied to the tendency only, main.cpp:296-312).
  * KAT-5 invariants: mode (0,0) is constant, enstrophy does not grow.
  * two forced RK4 steps at 1024^2 ... 16384^2: the default kernels must reproduce both park variants of K-ROW
    (XFB_ROW_TMEM=0/1, <= 8192) and, at 4096, the two-level K-COL of the 16384 grid (XFB_COL_2L=1) against colt_kernel
    to float32 rounding -- the knobs are read once per process, so each variant runs in its own interpreter -- and
    the oracle to north_star's one-step tolerance, 1e-5.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import rel_l2
import fields

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LX, NU = 600000.0, 6.5


def _rk4_factor(k2, dt):
    z = -NU * k2 * dt
    return 1 + z + z * z / 2 + z ** 3 / 6 + z ** 4 / 24


@pytest.mark.parametrize("n", [4096, 8192])
def test_linear_decay_and_frozen_modes(n):
    import xlab_fftbarotropic_b200 as xfb
    b = xfb.Backend(n)
    h = n // 2 + 1
    dt = 0.5
    kd = 2 * int(np.ceil(n / 3.0)) ** 2
    # (i, j, inside the mask?) -- one mode at a time so the Jacobian vanishes identically
    modes = [(3, 5), (n - 7, 11), (n // 4, n // 4), (n // 2, 3), (n // 2 - 1, n // 2), (5, n // 2)]
    for i, j in modes:
        z = np.zeros((n, h), np.complex64)
        z[i, j] = 1000.0 + 500.0j
        b.set_spectrum(z)
        b.step(1, dt)
        out = b.get_spectrum()
        ii = min(i, n - i)
        inside = ii * ii + j * j < kd
        kx = 2 * np.pi * (i if i <= n // 2 else i - n) / LX
        ky = 2 * np.pi * j / LX
        fac = _rk4_factor(kx * kx + ky * ky, dt) if inside else 1.0
        got = out[i, j] / z[i, j]
        assert abs(got - fac) < 2e-6 * max(1.0, abs(fac)), (n, i, j, inside, got, fac)
        out[i, j] = 0
        assert np.abs(out).max() < 1e-3 * 1e-3, f"mode ({i},{j}) leaked into others: {np.abs(out).max()}"
    b.close()


@pytest.mark.parametrize("n", [4096])
def test_invariants_full_size(n):
    import xlab_fftbarotropic_b200 as xfb
    b = xfb.Backend(n)
    v0 = fields.elliptic(n)
    b.set_vorticity(v0)
    s0 = b.get_spectrum()
    ens0 = float((v0.astype(np.float64) ** 2).sum())
    b.step(5, 1.0)
    s1 = b.get_spectrum()
    v1 = b.get_field(xfb.capi.VORT)
    assert np.isfinite(v1).all()
    assert abs(s1[0, 0] - s0[0, 0]) <= 1e-6 * abs(s0[0, 0]) + 1e-12          # KAT-5: mean vorticity untouched
    ens1 = float((v1.astype(np.float64) ** 2).sum())
    assert ens1 <= ens0 * (1 + 1e-6)                                           # enstrophy does not grow
    assert ens1 > 0.9 * ens0
    b.close()


def test_two_members_at_8192_match_single_runs():
    """ensemble indexing of the 8192 kernels (tensor-memory parks, TMA box ring): members of one handle reproduce
    single-member handles bit for bit"""
    import xlab_fftbarotropic_b200 as xfb
    n, dt = 8192, 0.5
    inits = [fields.elliptic(n), fields.gaussian(n)]
    b2 = xfb.Backend(n, batch=2)
    for m, v0 in enumerate(inits):
        b2.set_vorticity(v0, member=m)
    b2.step(3, dt)
    got = [b2.get_spectrum(member=m) for m in range(2)]
    b2.close()
    for m, v0 in enumerate(inits):
        b1 = xfb.Backend(n)
        b1.set_vorticity(v0)
        b1.step(3, dt)
        ref = b1.get_spectrum()
        b1.close()
        assert np.isfinite(ref.view(np.float32)).all()
        assert np.array_equal(got[m].view(np.float32), ref.view(np.float32)), m


_VARIANT = r"""
import sys, numpy as np
sys.path.insert(0, {root!r}); sys.path.insert(0, {root!r} + "/tests")
import fields, xlab_fftbarotropic_b200 as xfb
n = {n}
b = xfb.Backend(n)
b.set_vorticity(fields.elliptic(n))
b.set_source(fields.wave_source(n))   # the forcing path too
b.step(2, {dt})
np.save({out!r}, b.get_spectrum())
"""


def _run_variant(n, dt, env, out):
    e = dict(os.environ)
    e.update(env)
    code = _VARIANT.format(root=ROOT, n=n, dt=dt, out=out)
    subprocess.run([sys.executable, "-c", code], check=True, env=e, timeout=600)
    return np.load(out)


@pytest.mark.parametrize("n,dt", [(1024, 3.0), (4096, 1.0), (8192, 0.5), (16384, 0.25)])
def test_forced_steps_kernel_variants_and_oracle(n, dt, tmp_path):
    ref = _run_variant(n, dt, {}, str(tmp_path / "default.npy"))
    assert np.isfinite(ref.view(np.float32)).all()
    variants = []
    if n <= 8192:
        # K-ROW with tensor-memory parks is the default at >= 4096 only: force it on and off everywhere
        variants = [{"XFB_ROW_TMEM": "1"}, {"XFB_ROW_TMEM": "0"}]
    if n == 4096:
        variants.append({"XFB_COL_2L": "1"})          # the two-level K-COL of the 16384 grid, forced onto 4096-point columns
    for env in variants:
        got = _run_variant(n, dt, env, str(tmp_path / "variant.npy"))
        assert rel_l2(got, ref) < 2e-6, (env, rel_l2(got, ref))
    if n == 16384:
        import psutil
        if psutil.virtual_memory().available < 48 * 2 ** 30:
            pytest.skip("the 16384^2 oracle needs ~30 GiB of host memory")
    from oracle import oracle as orc
    orc.set_threads(0)        # the shim FFT's line loops on all host cores; results do not depend on the thread count
    o = orc.Oracle(n)
    o.set_vorticity(fields.elliptic(n))
    o.set_source(fields.wave_source(n))
    o.step(2, dt)
    assert rel_l2(ref, o.get_spectrum()) < 1e-5


def test_one_step_against_oracle_2048():
    import xlab_fftbarotropic_b200 as xfb
    from oracle import oracle as orc
    n = 2048
    v0 = fields.kuo2004(n)
    b = xfb.Backend(n)
    o = orc.Oracle(n)
    b.set_vorticity(v0)
    o.set_vorticity(v0)
    b.step(1, 1.5)
    o.step(1, 1.5)
    assert rel_l2(b.get_spectrum(), o.get_spectrum()) < 1e-5
    assert rel_l2(b.get_field(xfb.capi.U), o.get_field(orc.U)) < 1e-5
    b.close()

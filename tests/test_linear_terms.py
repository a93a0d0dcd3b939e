"""Linear terms of the vorticity equation (xfb_set_linear_terms, DESIGN.md section 3): beta-plane -beta v, linear drag
-mu zeta and hyperviscosity -nu_h (-lap)^p zeta, added per mode as L(k) Z_k inside the dealiasing mask.

CPU: a float64 restatement of one RK4 step with L(k), checked against the restatement of the reference equation and
against the Rossby-wave dispersion relation.  GPU: exact discrete solutions on one lattice shell (where the Jacobian
vanishes and every mode evolves by the RK4 polynomial), graph invalidation, nonlinear steps against the restatement,
the decomposed and ensemble handles, beta drift of a vortex, main.out -B -R -H -P and argument errors."""
import os
import subprocess
import sys
import tempfile

import numpy as np
import pytest

from conftest import rel_l2
import fields

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "xlab_fftbarotropic_b200", "bin")
LX = 600000.0
NU = 6.5
DT = 3.0


# ---- float64 restatement ---------------------------------------------------------------------------------------------
def _wavenumbers(nx, ny, lx, ly):
    kx = 2 * np.pi * np.where(np.arange(nx) <= nx // 2, np.arange(nx), np.arange(nx) - nx) / lx
    ky = 2 * np.pi * np.arange(ny // 2 + 1) / ly
    return kx[:, None], ky[None, :]


def lin_factor(nx, ny, lx, ly, beta, mu, nu_h, p):
    """L(k) = -mu - nu_h k^(2p) + i beta kx / k^2 on the half spectrum ((0,0): the beta term is 0, the drag applies)"""
    KX, KY = _wavenumbers(nx, ny, lx, ly)
    K2 = KX ** 2 + KY ** 2
    safe = np.where(K2 > 0, K2, 1.0)
    return -mu - nu_h * K2 ** p + 1j * beta * KX / safe


def numpy_step_lin(z, nx, ny, lx, ly, nu, dt, beta=0.0, mu=0.0, nu_h=0.0, p=1):
    """one RK4 step of main.cpp:146-317 on rfft2 conventions, with L(k) Z_k added to the tendency inside the mask"""
    KX, KY = _wavenumbers(nx, ny, lx, ly)
    K2 = KX ** 2 + KY ** 2
    inv = -K2.copy()
    inv[0, 0] = 1.0
    ii = np.minimum(np.arange(nx), nx - np.arange(nx))[:, None]
    jj = np.arange(ny // 2 + 1)[None, :]
    mask = (ii * ii + jj * jj < np.ceil(nx / 3.0) ** 2 + np.ceil(ny / 3.0) ** 2)
    L = lin_factor(nx, ny, lx, ly, beta, mu, nu_h, p)

    def c2r(a):
        return np.fft.irfft2(a, s=(nx, ny))

    def tend(Z):
        psi = Z / inv
        zx, zy = c2r(1j * KX * Z), c2r(1j * KY * Z)
        u, v = -c2r(1j * KY * psi), c2r(1j * KX * psi)
        return mask * (np.fft.rfft2(-u * zx - v * zy) + nu * (-K2) * Z + L * Z)

    r1 = tend(z)
    r2 = tend(z + r1 * dt / 2)
    r3 = tend(z + r2 * dt / 2)
    r4 = tend(z + r3 * dt)
    return z + (r1 + 2 * r2 + 2 * r3 + r4) * dt / 6


def rk4_poly(z):
    return 1 + z + z * z / 2 + z ** 3 / 6 + z ** 4 / 24


def test_restatement_with_zero_terms_is_the_reference_equation():
    from test_headline_parity import _numpy_step
    n = 64
    rng = np.random.default_rng(3)
    v0 = 1e-4 * rng.standard_normal((n, n))
    z = np.fft.rfft2(v0)
    a = numpy_step_lin(z, n, n, LX, LX, NU, DT)
    b = _numpy_step(z, n, n, LX, LX, NU, DT)
    assert rel_l2(a, b) < 1e-14
    assert rel_l2(numpy_step_lin(z, n, n, LX, LX, NU, DT, beta=1e-9, mu=1e-4, nu_h=1e-3, p=2), b) > 1e-6


def test_restatement_rossby_wave_propagates_westward():
    """a single mode under beta > 0: phase speed -beta / k^2 along x (the slow index), i.e. westward"""
    n, a, b = 64, 3, 2
    beta = 1.6e-11
    k0 = 2 * np.pi / LX
    kx, k2 = a * k0, (a * a + b * b) * k0 * k0
    z = np.zeros((n, n // 2 + 1), complex)
    z[a, b] = 1e-6 * n * n                              # zeta ~ 1e-6 / s
    steps, dt = 225, 20000.0                            # a quarter wavelength west in 52 days
    zz = z
    for _ in range(steps):
        zz = numpy_step_lin(zz, n, n, LX, LX, 0.0, dt, beta=beta)
    # the Jacobian of one mode vanishes: the mode alone evolves, by the RK4 polynomial of i omega dt
    assert np.abs(np.delete(zz.ravel(), a * (n // 2 + 1) + b)).max() < 1e-9 * abs(z[a, b])
    phase = np.angle(zz[a, b] / z[a, b])
    shift = -phase / kx                                 # zeta ~ cos(kx (x - c t) + ...): pattern displacement along x
    expect = -beta / k2 * steps * dt
    assert shift < 0
    assert abs(shift - expect) < 1e-3 * abs(expect)
    # omega = -beta kx / k^2 as exp(i (k.x - omega t))
    assert abs(phase / (steps * dt) - beta * kx / k2) < 1e-3 * beta * kx / k2
    # the physical field moves west: its cross-correlation with the start peaks at a negative x shift
    f0 = np.fft.irfft2(z, s=(n, n))[:, 0]
    f1 = np.fft.irfft2(zz, s=(n, n))[:, 0]
    xc = [np.dot(np.roll(f0, s), f1) for s in range(-n // (2 * a), n // (2 * a) + 1)]
    assert range(-n // (2 * a), n // (2 * a) + 1)[int(np.argmax(xc))] < 0


def test_main_out_rejects_bad_linear_terms():
    exe = os.path.join(BIN, "main.out")
    for args in (["-P", "0"], ["-P", "9"], ["-R", "-1"], ["-H", "-2e3"], ["-B", "nan"], ["-B", "1e-11x"], ["-H", "inf"]):
        with tempfile.TemporaryDirectory() as d:
            r = subprocess.run([exe, "-n", "256", "-t", "1", *args], cwd=d, capture_output=True, text=True, timeout=60)
            assert r.returncode == 1, (args, r.stdout, r.stderr)
            assert "-P <order>" in r.stderr, args


# ---- GPU helpers -----------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def xfb():
    import xlab_fftbarotropic_b200 as m
    m.load()
    return m


def shell_points(r2, nmax):
    """lattice points (a, b) with a^2 + b^2 = r2, b >= 0 (a > 0 when b == 0): one of each conjugate pair"""
    pts = []
    for b in range(0, nmax):
        a2 = r2 - b * b
        if a2 < 0:
            break
        a = int(round(np.sqrt(a2)))
        if a * a != a2:
            continue
        for s in ({a, -a} if a else {0}):
            if b == 0 and s <= 0:
                continue
            pts.append((s, b))
    return pts


def _mask_kd(nx, ny):
    return np.ceil(nx / 3.0) ** 2 + np.ceil(ny / 3.0) ** 2


def _dealias_mask(nx, ny):
    ii = np.minimum(np.arange(nx), nx - np.arange(nx))[:, None]
    jj = np.arange(ny // 2 + 1)[None, :]
    return ii * ii + jj * jj < _mask_kd(nx, ny)


def shell_for(nx, ny):
    """a shell r^2 = 5525 m^2 (a multiple of the 24-point shell 5525) at about 0.6 of the mask radius, below half the
    smaller dimension.  The Jacobian's float32 roundoff puts a little of every mode the mask keeps into the state, so the
    explicit RK4 has to be stable up to the mask's edge: a shell this far out lets the hyperviscosity move the shell by far
    more than the tolerance while the edge stays stable"""
    r_mask = np.sqrt(_mask_kd(nx, ny))
    target = min(0.6 * r_mask, 0.45 * min(nx, ny))
    m = max(1, int(round(target / np.sqrt(5525.0))))
    r2 = 5525 * m * m
    assert np.sqrt(r2) < min(nx, ny) / 2 and r2 < _mask_kd(nx, ny)
    return r2


def coefficients(nx, ny, r2, which, p):
    """(beta, mu, nu_h): beta dt / k_min = 1 (the largest |omega| dt of the grid, mode (1, 0)), mu dt = 0.01,
    nu_h k^(2p) dt = 0.02 on the shell unless that puts nu_h k_mask^(2p) dt above 2 (RK4 is stable on the negative real
    axis up to 2.78 and on the imaginary axis up to 2.83)"""
    k0 = 2 * np.pi / LX
    beta = k0 / DT if which in ("beta", "all") else 0.0
    mu = 0.01 / DT if which in ("mu", "all") else 0.0
    nu_h = min(0.02 / (DT * (r2 * k0 * k0) ** p), 2.0 / (DT * (_mask_kd(nx, ny) * k0 * k0) ** p))
    return beta, mu, (nu_h if which in ("hyper", "all") else 0.0)


CASES = [("beta", 4), ("mu", 4), ("hyper", 1), ("hyper", 4), ("all", 1), ("all", 4)]
STEPS = 50


def shell_spectrum(nx, ny, r2, seed):
    """half spectrum with random modes on the shell only (a real field: the j = 0 column is Hermitian)"""
    pts = shell_points(r2, ny // 2)
    rng = np.random.default_rng(seed)
    amp = 1e-4 * nx * ny / np.sqrt(2 * len(pts))
    z = np.zeros((nx, ny // 2 + 1), np.complex64)
    vals = amp * (rng.standard_normal(len(pts)) + 1j * rng.standard_normal(len(pts)))
    for (a, b), v in zip(pts, vals):
        z[a % nx, b] = v
        if b == 0:
            z[(-a) % nx, 0] = np.conj(v)
    return z, pts


def shell_error(got, z0, pts, nx, ny, beta, mu, nu_h, p, steps=STEPS):
    """rel-L2 of the state after `steps` steps against R(dt L)^steps Z0 (off-shell entries must stay zero)"""
    L = lin_factor(nx, ny, LX, LX, beta, mu, nu_h, p)
    k0 = 2 * np.pi / LX
    idx = [(a % nx, b) for a, b in pts] + [((-a) % nx, 0) for a, b in pts if b == 0]
    rows = np.array([i for i, _ in idx])
    cols = np.array([j for _, j in idx])
    k2 = ((np.where(rows <= nx // 2, rows, rows - nx) * k0) ** 2 + (cols * k0) ** 2)
    lam = L[rows, cols] - NU * k2
    exp = z0[rows, cols].astype(np.complex128) * rk4_poly(DT * lam) ** steps
    on = got[rows, cols].astype(np.complex128)
    got = got.copy()
    got[rows, cols] = 0
    off = float(np.linalg.norm(got.view(np.float32)))
    err = np.sqrt(np.sum(np.abs(on - exp) ** 2) + off * off) / np.linalg.norm(exp)
    moved = np.linalg.norm(exp - z0[rows, cols] * rk4_poly(-DT * NU * k2) ** steps) / np.linalg.norm(exp)
    return err, moved


def run_shell_cases(xfb, nx, ny, batch=1):
    r2 = shell_for(nx, ny)
    b = xfb.Backend(nx, ny, batch=batch)
    out = []
    for which, p in CASES:
        beta, mu, nu_h = coefficients(nx, ny, r2, which, p)
        z0s = []
        for m in range(batch):
            z0, pts = shell_spectrum(nx, ny, r2, seed=nx + ny + 7 * m + p)
            b.set_spectrum(z0, member=m)
            z0s.append(z0)
        b.set_linear_terms(beta, mu, nu_h, p)
        b.step(STEPS, DT)
        for m in range(batch):
            err, moved = shell_error(b.get_spectrum(member=m), z0s[m], pts, nx, ny, beta, mu, nu_h, p)
            out.append((which, p, m, err, moved))
        del z0s
    b.close()
    return out


def _check(results, label):
    for which, p, m, err, moved in results:
        assert err <= 1e-5, f"{label} {which} p={p} member {m}: rel-L2 {err:.3e}"
        assert moved > 1e-3, f"{label} {which} p={p}: the terms move the answer by only {moved:.3e}"


# ---- 1. exact discrete solution on one shell -------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("nx,ny", [(256, 256), (512, 512), (1024, 1024), (4096, 4096), (8192, 8192), (16384, 16384),
                                   (768, 768), (1024, 768)])
def test_exact_shell_solution(xfb, nx, ny):
    _check(run_shell_cases(xfb, nx, ny), f"{nx}x{ny}")


@pytest.mark.gpu
def test_exact_shell_solution_ensemble(xfb):
    _check(run_shell_cases(xfb, 256, 256, batch=4), "256^2 x 4 members")


@pytest.mark.gpu
def test_exact_shell_solution_two_level_4096():
    """the XFB_COL_2L=1 instance of the two-level K-COL at 4096 (the knob is read once per process)"""
    code = ("import sys; sys.path[:0] = [%r, %r]; import test_linear_terms as t, xlab_fftbarotropic_b200 as x; "
            "x.load(); t._check(t.run_shell_cases(x, 4096, 4096), '4096^2 two-level')") % (ROOT, os.path.join(ROOT, "tests"))
    env = dict(os.environ, XFB_COL_2L="1")
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]


@pytest.mark.gpu
@pytest.mark.parametrize("n,p,c", [(256, 2, 1), (512, 4, 2)])
def test_exact_shell_solution_loopback(xfb, n, p, c):
    r2 = shell_for(n, n)
    team = xfb.LoopbackTeam(n, p, c)
    for which, order in (("all", 1), ("all", 4), ("beta", 4)):
        beta, mu, nu_h = coefficients(n, n, r2, which, order)
        zs, pts = shell_spectrum(n, n, r2, seed=n + order)
        v0 = np.fft.irfft2(zs.astype(np.complex128), s=(n, n)).astype(np.float32)
        z0 = np.fft.rfft2(v0.astype(np.float64))
        team.set_vorticity(v0)
        team.set_linear_terms(beta, mu, nu_h, order)
        team.step(STEPS, DT)
        KX, KY = _wavenumbers(n, n, LX, LX)
        lam = lin_factor(n, n, LX, LX, beta, mu, nu_h, order) - NU * (KX ** 2 + KY ** 2)
        # the float32 field carries a little of every mode; those outside the dealiasing mask are never updated (their
        # RK4 factor would be far outside the stability region)
        exp = np.fft.irfft2(z0 * np.where(_dealias_mask(n, n), rk4_poly(DT * lam) ** STEPS, 1.0), s=(n, n))
        err = rel_l2(team.get_field(xfb.capi.VORT), exp)
        assert err <= 1e-5, (which, order, err)
    team.close()


# ---- 2. graph invalidation and switching off ---------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n", [256, 768])
def test_changed_terms_drop_the_captured_step(xfb, n):
    r2 = shell_for(n, n)
    b = xfb.Backend(n)
    z0, pts = shell_spectrum(n, n, r2, seed=11)
    c1 = coefficients(n, n, r2, "all", 2)
    c3 = coefficients(n, n, r2, "all", 3)
    c2 = (-0.5 * c3[0], 2 * c3[1], 0.5 * c3[2])
    b.set_spectrum(z0)
    b.set_linear_terms(*c1, 2)
    b.step(5, DT)
    b.set_linear_terms(*c2, 3)
    b.step(5, DT)
    got = b.get_spectrum()
    L1 = lin_factor(n, n, LX, LX, *c1, 2)
    L2 = lin_factor(n, n, LX, LX, *c2, 3)
    KX, KY = _wavenumbers(n, n, LX, LX)
    nuk = -NU * (KX ** 2 + KY ** 2)
    inside = _dealias_mask(n, n)          # z0 is zero outside the mask, where the factors would overflow
    f1 = np.where(inside, rk4_poly(DT * (L1 + nuk)), 1.0)
    f2 = np.where(inside, rk4_poly(DT * (L2 + nuk)), 1.0)
    exp = z0.astype(np.complex128) * f1 ** 5 * f2 ** 5
    assert rel_l2(got, exp) <= 1e-5
    # had the first graph been replayed, the answer would be the other one
    assert rel_l2(z0 * f1 ** 10, exp) > 1e-3
    # all zeros: bit-identical to a handle that never set terms
    v0 = fields.gaussian(n)
    b.set_linear_terms(0.0, 0.0, 0.0)
    b.set_vorticity(v0)
    b.step(5, DT)
    fresh = xfb.Backend(n)
    fresh.set_vorticity(v0)
    fresh.step(5, DT)
    assert np.array_equal(b.get_spectrum().view(np.float32), fresh.get_spectrum().view(np.float32))
    assert np.array_equal(b.get_field(xfb.capi.VORT), fresh.get_field(xfb.capi.VORT))
    b.close()
    fresh.close()


# ---- 3. nonlinear steps against the restatement ------------------------------------------------------------------------
def _nonlinear_coefficients(n):
    k0 = 2 * np.pi / LX
    kd = 2 * np.ceil(n / 3.0) ** 2
    return 0.5 * k0 / DT, 0.01 / DT, 1.0 / (DT * (kd * k0 * k0) ** 2), 2


@pytest.mark.gpu
@pytest.mark.parametrize("n,field", [(512, "gaussian"), (1024, "elliptic"), (768, "gaussian")])
def test_nonlinear_steps_against_restatement(xfb, n, field):
    v0 = getattr(fields, field)(n)
    beta, mu, nu_h, p = _nonlinear_coefficients(n)
    b = xfb.Backend(n)
    b.set_vorticity(v0)
    b.set_linear_terms(beta, mu, nu_h, p)
    z = np.fft.rfft2(v0.astype(np.float64))
    b.step(1, DT)
    z1 = numpy_step_lin(z, n, n, LX, LX, NU, DT, beta, mu, nu_h, p)
    assert rel_l2(b.get_spectrum(), z1) < 1e-5
    assert rel_l2(numpy_step_lin(z, n, n, LX, LX, NU, DT), z1) > 1e-4      # the terms matter at this tolerance
    b.step(19, DT)
    for _ in range(19):
        z1 = numpy_step_lin(z1, n, n, LX, LX, NU, DT, beta, mu, nu_h, p)
    assert rel_l2(b.get_spectrum(), z1) < 1e-4
    b.close()


# ---- 4. decomposition and ensembles --------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n,p,c", [(256, 2, 1), (512, 4, 2)])
def test_loopback_team_matches_single_gpu_with_terms(xfb, n, p, c):
    v0 = fields.kuo2004(n)
    beta, mu, nu_h, order = _nonlinear_coefficients(n)
    one = xfb.Backend(n)
    team = xfb.LoopbackTeam(n, p, c)
    for h in (one, team):
        h.set_vorticity(v0)
        h.set_linear_terms(beta, mu, nu_h, order)
        h.step(3, DT)
    for which in (xfb.capi.VORT, xfb.capi.PSI, xfb.capi.U, xfb.capi.V):
        assert rel_l2(team.get_field(which), one.get_field(which)) < 2e-6, which
    one.close()
    team.close()


@pytest.mark.gpu
def test_ensemble_members_match_single_member_handles(xfb):
    n, members = 256, 4
    beta, mu, nu_h, order = _nonlinear_coefficients(n)
    ens = xfb.Backend(n, batch=members)
    inits = [fields.gaussian_member(n, m) for m in range(members)]
    for m, v in enumerate(inits):
        ens.set_vorticity(v, member=m)
    ens.set_linear_terms(beta, mu, nu_h, order)
    ens.step(6, DT)
    for m, v in enumerate(inits):
        one = xfb.Backend(n)
        one.set_vorticity(v)
        one.set_linear_terms(beta, mu, nu_h, order)
        one.step(6, DT)
        assert np.array_equal(ens.get_spectrum(member=m).view(np.float32), one.get_spectrum().view(np.float32)), m
        one.close()
    ens.close()


# ---- 5. beta drift of a vortex ----------------------------------------------------------------------------------------------
def _centroid(f):
    sel = f > 0.5 * f.max()
    i, j = np.nonzero(sel)
    return i.mean(), j.mean()


@pytest.mark.gpu
def test_beta_drift_of_cyclone_and_anticyclone(xfb):
    """Chan & Williams (1987): on a beta plane a cyclone drifts west (-x) and poleward (+y), an anticyclone west and
    equatorward; the reference point is the same run with beta = 0.  The beta gyres take time to spin up and the
    displacement grows about quadratically at first (float64 restatement at 128^2, in 512^2 cells: 2 cells west after
    6 h, 6 after 12 h, 15 after 24 h), so the run lasts a day"""
    n, steps = 512, int(24 * 3600 / DT)
    v0 = fields.gaussian(n)
    for sign, dy_sign in ((1.0, 1.0), (-1.0, -1.0)):
        res = {}
        for beta in (0.0, 2.3e-11):
            b = xfb.Backend(n)
            b.set_vorticity((sign * v0).astype(np.float32))
            b.set_linear_terms(beta, 0.0, 0.0)
            b.step(steps, DT)
            res[beta] = _centroid(sign * b.get_field(xfb.capi.VORT))
            b.close()
        dx = res[2.3e-11][0] - res[0.0][0]
        dy = res[2.3e-11][1] - res[0.0][1]
        assert dx < -5, (sign, dx, dy)
        assert dy_sign * dy > 5, (sign, dx, dy)


# ---- 6. host program -----------------------------------------------------------------------------------------------------
def _gpu_count():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


def _run_main(v0, n, steps, rec, extra):
    with tempfile.TemporaryDirectory() as d:
        os.makedirs(os.path.join(d, "input"))
        os.makedirs(os.path.join(d, "output"))
        v0.tofile(os.path.join(d, "input", "initial_vorticity.bin"))
        r = subprocess.run([os.path.join(BIN, "main.out"), "-n", str(n), "-t", str(steps), "-r", str(rec), "-q", *extra], cwd=d,
                           capture_output=True, text=True, timeout=600)
        files = {}
        if r.returncode == 0:
            for k in ("vort", "psi", "u", "v"):
                files[k] = np.fromfile(os.path.join(d, "output", f"{k}_step_{rec}.bin"), dtype="<f4").reshape(n, n)
        return r, files


@pytest.mark.gpu
def test_main_out_linear_terms_match_backend(xfb):
    n, steps, rec = 256, 4, 3
    v0 = fields.elliptic(n)
    beta, mu, nu_h, order = _nonlinear_coefficients(n)
    args = ["-B", repr(float(np.float32(beta))), "-R", repr(float(np.float32(mu))), "-H", repr(float(np.float32(nu_h))),
            "-P", str(order)]
    r, files = _run_main(v0, n, steps, rec, args)
    assert r.returncode == 0, r.stderr[-2000:]
    b = xfb.Backend(n)
    b.set_vorticity(v0)
    b.set_linear_terms(beta, mu, nu_h, order)
    b.step(rec, DT)
    for k, which in (("vort", xfb.capi.VORT), ("psi", xfb.capi.PSI), ("u", xfb.capi.U), ("v", xfb.capi.V)):
        assert np.array_equal(files[k], b.get_field(which)), k
    b.close()
    # the flags change the answer; a hyperviscosity coefficient out of float range stops the run
    r0, plain = _run_main(v0, n, steps, rec, [])
    assert r0.returncode == 0 and not np.array_equal(plain["vort"], files["vort"])
    rbad, _ = _run_main(v0, n, steps, rec, ["-H", "1e-30", "-P", "8"])       # nu_h k_c^16 below the normal floats
    assert rbad.returncode == 1 and "out of float range" in rbad.stderr


@pytest.mark.gpu
def test_main_out_linear_terms_on_two_slab_ranks(xfb):
    if _gpu_count() < 2:
        pytest.skip("needs two GPUs")
    n, steps, rec = 512, 4, 3
    v0 = fields.kuo2004(n)
    args = ["-B", "1e-10", "-R", "1e-5", "-H", "1e3", "-P", "2"]
    r1, one = _run_main(v0, n, steps, rec, args)
    r2, slab = _run_main(v0, n, steps, rec, ["-S", "2", *args])
    assert r1.returncode == 0 and r2.returncode == 0, r2.stderr[-2000:]
    for k in ("vort", "psi"):
        assert rel_l2(slab[k], one[k]) < 2e-6, k


# ---- 7. argument errors ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_argument_errors(xfb):
    L = xfb.load()
    b = xfb.Backend(256)
    E_ARG = -1
    for args in ((0.0, 0.0, 1.0, 0), (0.0, 0.0, 1.0, 9), (0.0, -1e-5, 0.0, 4), (0.0, 0.0, -1.0, 4),
                 (float("nan"), 0.0, 0.0, 4), (0.0, float("nan"), 0.0, 4), (0.0, 0.0, float("inf"), 4),
                 (0.0, 0.0, 1e-30, 8)):
        assert L.xfb_set_linear_terms(b._h, *args) == E_ARG, args
    assert L.xfb_set_linear_terms(None, 0.0, 0.0, 0.0, 4) == E_ARG
    assert L.xfb_set_linear_terms(b._h, -1e-11, 0.0, 0.0, 4) == 0          # beta may be negative
    assert L.xfb_set_linear_terms(b._h, 0.0, 0.0, 0.0, 4) == 0
    b.close()

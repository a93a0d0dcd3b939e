"""Synthetic initial vortices: numpy restatements of the reference generators
(/root/reference/src/makefield-*.cpp, field_generator.cpp).  Used by tests and bench.py; the
float32/float64 promotion of each expression follows the C++ source."""
import numpy as np

L = np.float32(600000.0)


def _grid(n, rows=None):
    """rows = (r0, r1): only the grid rows i in [r0, r1) (a slab-decomposed rank generates its own rows)"""
    dx = np.float32(L / np.float32(n))
    x = (np.arange(n, dtype=np.float32) * dx).astype(np.float32)
    xs = x if rows is None else x[rows[0]:rows[1]]
    return xs[:, None], x[None, :]   # x = i*dx (slow), y = j*dy (fast)


def _radius(x, y, cx, cy):
    # sqrtf(pow(x-cx,2) + pow(y-cy,2)): float differences, squared and summed in double, narrowed, sqrtf
    dxx = (x - cx).astype(np.float32).astype(np.float64)
    dyy = (y - cy).astype(np.float32).astype(np.float64)
    return np.sqrt((dxx * dxx + dyy * dyy).astype(np.float32)).astype(np.float32)


def gaussian(n):
    """makefield-gaussian.cpp:14-31"""
    x, y = _grid(n)
    c = np.float32(L / 2.0)
    r = _radius(x, y, c, c)
    q = r.astype(np.float64) / 60000.0          # float / double literal -> double
    return (np.float64(np.float32(1e-3)) * np.exp(-(q * q))).astype(np.float32)


def _lcg(seed, k):
    """k-th output in [0, 1) of the 32-bit LCG x <- 1664525 x + 1013904223 started from `seed` (Numerical Recipes)"""
    x = seed & 0xFFFFFFFF
    for _ in range(k + 1):
        x = (1664525 * x + 1013904223) & 0xFFFFFFFF
    return x / 4294967296.0


def gaussian_member(n, member):
    """Member `member` of BASELINE.json's ensemble config (64 Gaussian vortices at 512^2).  The reference has no
    ensemble and no RNG anywhere; members are the makefield-gaussian vortex with its centre moved by up to +-5 % of L
    in x and y and its amplitude scaled by 1 +- 10 %, drawn from an LCG seeded with the member index (SURVEY.md 8d).
    Member 0 of a one-member ensemble is NOT special: use gaussian() for the reference generator's field."""
    x, y = _grid(n)
    cx = np.float32(L * np.float32(0.5 + 0.1 * (_lcg(member, 0) - 0.5)))
    cy = np.float32(L * np.float32(0.5 + 0.1 * (_lcg(member, 1) - 0.5)))
    amp = np.float32(1e-3 * (1.0 + 0.2 * (_lcg(member, 2) - 0.5)))
    r = _radius(x, y, cx, cy)
    q = r.astype(np.float64) / 60000.0
    return (np.float64(amp) * np.exp(-(q * q))).astype(np.float32)


def const_vortex(n, rows=None):
    """makefield-const-vortex.cpp:14-35"""
    x, y = _grid(n, rows)
    c = np.float32(L / 2.0)
    r = _radius(x, y, c, c)
    return np.where(r <= np.float32(6000.0), np.float32(2e-5), np.float32(0)).astype(np.float32)


def elliptic(n, rows=None):
    """makefield-elliptic-vortex.cpp:14-50"""
    x, y = _grid(n, rows)
    c = np.float32(L / 2.0)
    eps, lam, zeta0 = np.float32(0.7), np.float32(2.0), np.float32(0.005)
    r_i, r_o = np.float32(30000.0), np.float32(60000.0)
    r = _radius(x, y, c, c)
    with np.errstate(divide="ignore", invalid="ignore"):
        cs = np.where(r == 0, np.float32(0), ((y - c).astype(np.float32) / r).astype(np.float32)).astype(np.float32)
        e2 = np.float64(eps) * np.float64(eps)
        ec = (eps * cs).astype(np.float32).astype(np.float64)
        alpha = np.sqrt(((1.0 - e2) / (1.0 - ec * ec)).astype(np.float32)).astype(np.float32)
        ria = (r_i * alpha).astype(np.float32)
        roa = (r_o * alpha).astype(np.float32)
        rp = ((r - ria).astype(np.float32) / (roa - ria).astype(np.float32)).astype(np.float32)
        t1 = (-lam / rp).astype(np.float32).astype(np.float64)          # float / float
        t2 = 1.0 / (rp - np.float32(1)).astype(np.float32).astype(np.float64)
        with np.errstate(over="ignore"):
            skirt = (np.float64(zeta0) * (1.0 - np.exp(t1 * np.exp(t2)))).astype(np.float32)
    out = np.where(r <= ria, zeta0, np.where(r <= roa, skirt, np.float32(0)))
    return out.astype(np.float32)


def _cake(data, n, cx, cy, zeta0, scale_r):
    """field_generator.cpp:10-28"""
    x, y = _grid(n)
    dxx = (x - np.float32(cx)).astype(np.float32).astype(np.float64)
    dyy = (y - np.float32(cy)).astype(np.float32).astype(np.float64)
    r = (np.sqrt((dxx * dxx + dyy * dyy)).astype(np.float32) / np.float32(scale_r)).astype(np.float32)
    r64 = r.astype(np.float64)
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        add = np.float64(np.float32(zeta0)) * (1.0 - np.exp(-30.0 / r64 * np.exp(1.0 / (r64 - 1.0))))
    add = np.where(r < 1, add, 0.0)
    return np.where(r < 1, (data.astype(np.float64) + add).astype(np.float32), data)


def kuo2004(n):
    """makefield-Kuo2004.cpp:30-44 (the reference adds into an uninitialised malloc; zero pages in practice)"""
    data = np.zeros((n, n), np.float32)
    data = _cake(data, n, L / 2.0, L / 2.0, 1.5e-2, 10000.0)
    data = _cake(data, n, L / 2.0 + 50000.0, L / 2.0, 3e-3, 30000.0)
    return data.astype(np.float32)


def wave_source(n):
    """a smooth forcing term for the source path of the stepper: 2e-8 sin(2 pi 3 x) cos(2 pi 5 y), x, y in [0, 1)"""
    x = np.arange(n, dtype=np.float32) / n
    return (2e-8 * np.sin(2 * np.pi * 3 * x)[:, None] * np.cos(2 * np.pi * 5 * x)[None, :]).astype(np.float32)


GENERATORS = {"elliptic": elliptic, "const": const_vortex, "gaussian": gaussian, "kuo2004": kuo2004}

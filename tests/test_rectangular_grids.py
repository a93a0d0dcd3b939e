"""The fused kernels on rectangular power-of-two grids (nx != ny) and on lx != ly domains.

xfb_size_supported accepts every pair of powers of two from 256 to 16384, but a square grid hides a class of errors: the
Nyquist column and the padding columns enter the dealiasing mask once nx > 1.12 ny (the x-Nyquist row once ny > 1.12 nx),
the shorter direction reads the twiddle table with a stride, the persistent kernels get fewer items than SMs at 16384 x 256
and 256 x 16384, and nothing tells lx from ly.  Everything here is compared with a float64 numpy restatement of
main.cpp:146-317 plus the linear terms of DESIGN.md section 3 (`ref_step`), written without the kernels and without oracle/.

CPU (`-m "not gpu"`): the restatement itself -- against the CPU oracle on square grids, its tables bit for bit, its
sensitivity to an lx / ly swap, to a transposed input and to an error confined to the Nyquist column, and the mask census
that puts Nyquist-line modes inside the mask.

GPU: every off-diagonal pair with nx ny <= 2^24 (34 shapes) against ref_step; the 8 larger pairs with the closed forms and
the transforms; ensembles, the passive tracer, the diagnostics, the energy spectrum and the slab decomposition on
rectangular grids.  Tolerances are those of the square-grid tests: bit-exact for tables and pointwise operators, 5e-7 for
single transforms, 1e-5 for one and two RK4 steps, 2e-6 between the loopback team and the single-GPU handle.
"""
import numpy as np
import pytest
import scipy.fft as sfft

from conftest import rel_l2
import fields

POW = [256, 512, 1024, 2048, 4096, 8192, 16384]
SHAPES = [(a, b) for a in POW for b in POW if a != b and a * b <= 2 ** 24]            # 34: checked against ref_step
LARGE = [(a, b) for a in POW for b in POW if a != b and a * b > 2 ** 24]             # 8: closed forms and transforms
LX, LY = 600e3, 450e3
NU = 6.5


def domain(nx, ny):
    """lx != ly on every shape whose nx is an even power of two (19 of the 34, both orientations of several ratios)"""
    return (LX, LY) if (nx.bit_length() - 1) % 2 == 0 else (LX, LX)


def step_dt(nx, ny):
    """the time steps of test_large_grids.py by the longer side"""
    m = max(nx, ny)
    return 3.0 if m <= 1024 else (1.0 if m <= 4096 else 0.5)


def _fft(f):
    return sfft.rfft2(f, workers=-1)


def _ifft(z, nx, ny):
    # like FFTW's c2r, pocketfft's drops Im of the j = 0 and j = ny/2 columns after the x pass
    return sfft.irfft2(z, s=(nx, ny), workers=-1)


# ---- tables: the reference's float32 expressions (fftwfop.cpp:15-68, as create_body restates them) ------------------
TWOPI = np.float32(np.float32(np.pi) * np.float32(2.0))            # acosf(-1.0f) * 2.0f


def tables(nx, ny, lx, ly):
    """(gradx_coe[nx], grady_coe[ny/2+1], laplacian_coe, laplacian_coe_inverse, dealiasing_mask) as float32"""
    hy = ny // 2 + 1
    kx = np.empty(nx, np.float32)
    kx[:nx // 2 + 1] = (TWOPI * np.arange(nx // 2 + 1, dtype=np.float32)) / np.float32(lx)
    kx[nx // 2 + 1:] = -kx[1:nx - nx // 2][::-1]
    ky = (TWOPI * np.arange(hy, dtype=np.float32)) / np.float32(ly)
    lap = (-(kx.astype(np.float64)[:, None] ** 2 + ky.astype(np.float64)[None, :] ** 2)).astype(np.float32)
    lapinv = lap.copy()
    lapinv[0, 0] = 1.0
    mask = np.where(mask_index(nx, ny) >= mask_kd(nx, ny), np.float32(0), np.float32(1)).astype(np.float32)
    return kx, ky, lap, lapinv, mask


def mask_kd(nx, ny):
    """fftwfop.cpp:11-12,57: dk = (int)ceil(((float)N) / 3.0), kd = (float)(dkx^2 + dky^2)"""
    dkx = int(np.ceil(np.float64(np.float32(nx)) / 3.0))
    dky = int(np.ceil(np.float64(np.float32(ny)) / 3.0))
    return float(np.float32(float(dkx) * dkx + float(dky) * dky))


def mask_index(nx, ny):
    """ii^2 + jj^2 of every half-spectrum entry (ii = min(i, nx - i))"""
    ii = np.minimum(np.arange(nx), nx - np.arange(nx)).astype(np.int64)[:, None]
    jj = np.arange(ny // 2 + 1, dtype=np.int64)[None, :]
    return ii * ii + jj * jj


def lin_factor(nx, ny, lx, ly, beta, mu, nu_h, p):
    """L(k) = -mu - c_h (k^2 / k_c^2)^p + i beta kx / k^2 with c_h, 1 / k_c^2 formed as xfb_set_linear_terms forms them"""
    kx, ky = tables(nx, ny, lx, ly)[:2]
    kxc, kyc = float(kx[nx // 2]), float(ky[ny // 2])
    kc2 = kxc * kxc + kyc * kyc
    ch = float(np.float32(float(np.float32(nu_h)) * kc2 ** p))
    inv_kc2 = float(np.float32(1.0 / kc2))
    KX, KY = kx.astype(np.float64)[:, None], ky.astype(np.float64)[None, :]
    K2 = KX * KX + KY * KY
    beta, mu = float(np.float32(beta)), float(np.float32(mu))
    return -mu - ch * (K2 * inv_kc2) ** p + 1j * beta * KX / np.where(K2 > 0, K2, 1.0)


def ref_step(Z, nx, ny, lx, ly, nu, dt, src=None, beta=0.0, mu=0.0, nu_h=0.0, p=1, C=None, kappa=0.0):
    """One RK4 step of main.cpp:146-317 in float64 on rfft2 conventions, with the source of main.cpp:225-227, the linear
    terms L(k) Z_k of DESIGN.md section 3 inside the mask, and optionally a passive tracer C advected by the same stage
    velocity (dc/dt = -u.grad c + kappa lap c).  Returns Z1, or (Z1, C1) with a tracer."""
    kx, ky, lap, lapinv, mask = tables(nx, ny, lx, ly)
    KX, KY = kx.astype(np.float64)[:, None], ky.astype(np.float64)[None, :]
    lap, lapinv, mask = lap.astype(np.float64), lapinv.astype(np.float64), mask.astype(np.float64)
    nu, dt, kappa = float(np.float32(nu)), float(np.float32(dt)), float(np.float32(kappa))
    lin = nu * lap
    if beta or mu or nu_h:
        lin = lin + lin_factor(nx, ny, lx, ly, beta, mu, nu_h, p)
    s = 0.0 if src is None else np.asarray(src, np.float64)

    def tend(z, c):
        zx, zy = _ifft(1j * KX * z, nx, ny), _ifft(1j * KY * z, nx, ny)
        psi = z / lapinv
        u, v = -_ifft(1j * KY * psi, nx, ny), _ifft(1j * KX * psi, nx, ny)
        rz = mask * (_fft(-u * zx - v * zy + s) + lin * z)
        if c is None:
            return rz, None
        cx, cy = _ifft(1j * KX * c, nx, ny), _ifft(1j * KY * c, nx, ny)
        return rz, mask * (_fft(-u * cx - v * cy) + kappa * lap * c)

    Z = np.asarray(Z, np.complex128)
    C = None if C is None else np.asarray(C, np.complex128)
    r1, q1 = tend(Z, C)
    r2, q2 = tend(Z + r1 * (dt / 2), None if C is None else C + q1 * (dt / 2))
    r3, q3 = tend(Z + r2 * (dt / 2), None if C is None else C + q2 * (dt / 2))
    r4, q4 = tend(Z + r3 * dt, None if C is None else C + q3 * dt)
    Z1 = Z + (r1 + 2 * r2 + 2 * r3 + r4) * (dt / 6)
    if C is None:
        return Z1
    return Z1, C + (q1 + 2 * q2 + 2 * q3 + q4) * (dt / 6)


def ref_fields(Z, nx, ny, lx, ly):
    """record fields of a state as main.cpp writes them: VORT, PSI, U, V, DVORTDX, DVORTDY"""
    kx, ky, _, lapinv, _ = tables(nx, ny, lx, ly)
    KX, KY = kx.astype(np.float64)[:, None], ky.astype(np.float64)[None, :]
    psi = Z / lapinv.astype(np.float64)
    return {"vort": _ifft(Z, nx, ny), "psi": _ifft(psi, nx, ny), "u": -_ifft(1j * KY * psi, nx, ny),
            "v": _ifft(1j * KX * psi, nx, ny), "dvortdx": _ifft(1j * KX * Z, nx, ny), "dvortdy": _ifft(1j * KY * Z, nx, ny)}


def rk4_poly(z):
    return 1 + z + z * z / 2 + z ** 3 / 6 + z ** 4 / 24


# ---- inputs that reach the edges ---------------------------------------------------------------------------------------
def edge_regions(nx, ny):
    """boolean half-spectrum masks: the Nyquist column j = ny/2, the x-Nyquist row i = nx/2, and the modes within two
    lattice spacings of the dealiasing mask's edge on either side, |sqrt(ii^2 + jj^2) - sqrt(kd)| <= 2"""
    h = ny // 2 + 1
    col = np.zeros((nx, h), bool)
    col[:, ny // 2] = True
    row = np.zeros((nx, h), bool)
    row[nx // 2, :] = True
    band = np.abs(np.sqrt(mask_index(nx, ny).astype(np.float64)) - np.sqrt(mask_kd(nx, ny))) <= 2
    return {"nyquist_col": col, "nyquist_row": row, "mask_edge": band}


def edge_errors(got, want, nx, ny):
    """rel-L2 of a half spectrum over each edge region"""
    got = np.asarray(got)
    return {k: rel_l2(got[m], want[m]) for k, m in edge_regions(nx, ny).items()}


def rough_field(nx, ny, lx, ly, seed, umax=10.0):
    """random real field with a k^-1 amplitude spectrum, plus a band seeded on the Nyquist row, on the Nyquist column and
    around the mask edge that holds 5 % of the norm in each of the three regions (a smooth field has almost nothing there,
    so a wrong update of those modes would barely move the global rel-L2); scaled to max |u|, |v| = umax m/s.
    -> float32 field, its exact float64 spectrum"""
    rng = np.random.default_rng(seed)
    h = ny // 2 + 1
    k = np.sqrt(mask_index(nx, ny).astype(np.float64))
    amp = 1.0 / np.maximum(k, 1.0)
    amp[0, 0] = 0.0
    base = np.sqrt(np.sum(amp * amp))
    for m in edge_regions(nx, ny).values():
        amp[m] = 0.05 * base / np.sqrt(m.sum())
    z = amp * (rng.standard_normal((nx, h)) + 1j * rng.standard_normal((nx, h)))
    f = _ifft(z, nx, ny)                                 # Hermitian projection of the j = 0 and j = ny/2 columns
    fl = ref_fields(_fft(f), nx, ny, lx, ly)
    f *= umax / max(np.abs(fl["u"]).max(), np.abs(fl["v"]).max())
    f32 = f.astype(np.float32)
    return f32, _fft(f32.astype(np.float64))


def smooth_source(nx, ny, seed, scale):
    """forcing with a steep spectrum (no edge band), rms = scale"""
    rng = np.random.default_rng(seed)
    h = ny // 2 + 1
    k = np.sqrt(mask_index(nx, ny).astype(np.float64))
    z = (rng.standard_normal((nx, h)) + 1j * rng.standard_normal((nx, h))) / np.maximum(k, 1.0) ** 2
    s = _ifft(z, nx, ny)
    return (s * (scale / np.sqrt(np.mean(s * s)))).astype(np.float32)


def host_bytes_needed(nx, ny, ref=True):
    """host memory of one case: ~40 float64 full-size arrays for a reference step, ~12 for transforms alone"""
    return (320 if ref else 96) * nx * ny + 2 * 2 ** 30


def need_host_memory(nx, ny, ref=True):
    import psutil
    need = host_bytes_needed(nx, ny, ref)
    if psutil.virtual_memory().available < need:
        pytest.skip(f"{nx}x{ny} needs ~{need / 2 ** 30:.0f} GiB of free host memory")


# ---- CPU: the restatement itself -----------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,gen", [(64, "elliptic"), (64, "kuo2004"), (256, "elliptic"), (256, "kuo2004")])
def test_ref_step_matches_oracle_on_square_grids(n, gen):
    from oracle import oracle as orc
    v0 = fields.GENERATORS[gen](n)
    o = orc.Oracle(n)
    o.set_vorticity(v0)
    o.step(1, 3.0)
    got = ref_step(np.fft.rfft2(v0.astype(np.float64)), n, n, 600000.0, 600000.0, NU, 3.0)
    assert rel_l2(o.get_spectrum(), got) <= 1e-6, rel_l2(o.get_spectrum(), got)
    # c2r of a spectrum that is not Hermitian in the j = 0 and j = n/2 columns: the convention ref_step relies on
    rng = np.random.default_rng(n)
    z = (rng.standard_normal((n, n // 2 + 1)) + 1j * rng.standard_normal((n, n // 2 + 1))).astype(np.complex64)
    assert rel_l2(o.c2r(z), _ifft(z.astype(np.complex128), n, n) * (n * n)) < 5e-7


def test_table_restatement_matches_oracle_bit_for_bit():
    from oracle import oracle as orc
    n = 256
    o = orc.Oracle(n)
    for which, t in enumerate(tables(n, n, 600000.0, 600000.0)):
        assert np.array_equal(t.view(np.uint32), o.table(which).view(np.uint32)), which


def test_reference_sees_lx_ly_swap_and_transpose():
    nx, ny = 256, 128
    v0, z0 = rough_field(nx, ny, LX, LY, seed=1)
    a = ref_step(z0, nx, ny, LX, LY, NU, 3.0)
    assert rel_l2(ref_step(z0, nx, ny, LY, LX, NU, 3.0), a) > 1e-3
    # the mirror image (transposed, and negated: the vorticity is a pseudo-scalar) on the transposed grid with the same
    # lengths, mirrored back, is not the same answer either
    zt = _fft(-v0.T.astype(np.float64))
    bt = -_ifft(ref_step(zt, ny, nx, LX, LY, NU, 3.0), ny, nx).T
    assert rel_l2(bt, _ifft(a, nx, ny)) > 1e-3
    # the linear terms see the swap too (k_c and beta kx / k^2)
    kw = dict(beta=1e-10, mu=1e-5, nu_h=1e3, p=2)
    assert rel_l2(ref_step(z0, nx, ny, LY, LX, NU, 3.0, **kw), ref_step(z0, nx, ny, LX, LY, NU, 3.0, **kw)) > 1e-3


@pytest.mark.parametrize("nx,ny,line", [(512, 128, "nyquist_col"), (128, 512, "nyquist_row")])
def test_mask_census_includes_nyquist_lines(nx, ny, line):
    mask = tables(nx, ny, LX, LY)[4] > 0
    reg = edge_regions(nx, ny)
    assert int((mask & reg[line]).sum()) > 0, line
    other = "nyquist_row" if line == "nyquist_col" else "nyquist_col"
    assert int((mask & reg[other]).sum()) == 0
    # on a square grid neither Nyquist line is ever inside
    sq = tables(256, 256, LX, LX)[4] > 0
    assert not (sq & (edge_regions(256, 256)["nyquist_col"] | edge_regions(256, 256)["nyquist_row"])).any()
    # the inputs put energy there: the seeded band is not a rounding-level signal
    _, z0 = rough_field(nx, ny, LX, LY, seed=2)
    m = mask & reg[line]
    assert np.linalg.norm(z0[m]) > 1e-3 * np.linalg.norm(z0)


def test_edge_metrics_see_an_error_confined_to_the_nyquist_column():
    """an error confined to the update of one edge region, 5e-5 of that region's state, stays well below the global 1e-5
    bound but not below the per-region one"""
    nx, ny = 512, 128
    _, z0 = rough_field(nx, ny, LX, LY, seed=3)
    z1 = ref_step(z0, nx, ny, LX, LY, NU, 3.0)
    for name, m in edge_regions(nx, ny).items():
        inside = m & (tables(nx, ny, LX, LY)[4] > 0)          # modes the step updates (none on the x-Nyquist row here)
        if not inside.any():
            continue
        d = z1[inside] - z0[inside]
        bad = z1.copy()
        bad[inside] += d * (5e-5 * np.linalg.norm(z1[m]) / np.linalg.norm(d))
        assert rel_l2(bad, z1) < 3e-6, name
        assert edge_errors(bad, z1, nx, ny)[name] > 3e-5, name


def test_single_mode_decays_by_the_rk4_polynomial_in_ref_step():
    """the closed form of the GPU tests is ref_step's answer: a single mode has no Jacobian, and a mode with its lattice
    indices swapped decays at another rate on an lx != ly domain"""
    nx, ny = 256, 128
    dt = 3.0
    beta, mu, nu_h, p = closed_form_coefficients(nx, ny, LX, LY, dt, 2)
    lam = lin_factor(nx, ny, LX, LY, beta, mu, nu_h, p) + NU * tables(nx, ny, LX, LY)[2].astype(np.float64)
    facs = []
    for i, j in ((12, 7), (7, 12)):
        z = np.zeros((nx, ny // 2 + 1), complex)
        z[i, j] = 1e3 * (0.8 + 0.6j)
        z1 = ref_step(z, nx, ny, LX, LY, NU, dt, beta=beta, mu=mu, nu_h=nu_h, p=p)
        f = rk4_poly(dt * lam[i, j])
        assert abs(z1[i, j] / z[i, j] - f) < 1e-12
        z1[i, j] = 0
        assert np.abs(z1).max() < 1e-12 * 1e3
        facs.append(f)
    assert abs(facs[0] - facs[1]) > 1e-3 * abs(facs[0])


def test_size_supported_for_every_rectangular_pair():
    import xlab_fftbarotropic_b200 as xfb
    L = xfb.load()
    for nx, ny in SHAPES + LARGE:
        assert L.xfb_size_supported(nx, ny) == 1, (nx, ny)


# ---- GPU -----------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def xfb():
    import xlab_fftbarotropic_b200 as m
    m.load()
    return m


def _ids(shapes):
    return [f"{a}x{b}" for a, b in shapes]


def _random_spectrum(rng, nx, ny):
    h = ny // 2 + 1
    return (rng.standard_normal((nx, h)) + 1j * rng.standard_normal((nx, h))).astype(np.complex64)


@pytest.mark.gpu
@pytest.mark.parametrize("nx,ny", SHAPES + LARGE, ids=_ids(SHAPES + LARGE))
def test_tables_operators_and_transforms(xfb, nx, ny):
    need_host_memory(nx, ny, ref=False)
    lx, ly = domain(nx, ny)
    b = xfb.Backend(nx, ny, lx=lx, ly=ly)
    tab = tables(nx, ny, lx, ly)
    for which, t in enumerate(tab):
        assert np.array_equal(b.table(which).view(np.uint32), t.view(np.uint32)), f"table {which}"
    kx, ky, lap, lapinv, mask = tab
    rng = np.random.default_rng(nx + 3 * ny)
    z = _random_spectrum(rng, nx, ny)
    zr, zi = z.real, z.imag
    exp = {"gradx": (-(zi * kx[:, None]), zr * kx[:, None]), "grady": (-(zi * ky[None, :]), zr * ky[None, :]),
           "laplacian": (zr * lap, zi * lap), "invertLaplacian": (zr / lapinv, zi / lapinv), "dealiase": (zr * mask, zi * mask)}
    for name, (er, ei) in exp.items():
        got = getattr(b, name)(z)
        assert np.array_equal(got.real, er) and np.array_equal(got.imag, ei), name
    del exp, zr, zi
    f = rng.standard_normal((nx, ny)).astype(np.float32)
    F = b.r2c(f)
    assert rel_l2(F, _fft(f.astype(np.float64))) < 5e-7
    g = b.c2r(z)                                      # not Hermitian in the j = 0 and j = ny/2 columns
    assert rel_l2(g, _ifft(z.astype(np.complex128), nx, ny) * (nx * ny)) < 5e-7
    back = b.c2r(F) / np.float32(nx * ny)
    assert rel_l2(back, f) < 1e-6
    b.close()


@pytest.mark.gpu
@pytest.mark.parametrize("nx,ny", SHAPES, ids=_ids(SHAPES))
def test_two_forced_steps_against_ref_step(xfb, nx, ny):
    need_host_memory(nx, ny)
    lx, ly = domain(nx, ny)
    dt = step_dt(nx, ny)
    v0, z0 = rough_field(nx, ny, lx, ly, seed=nx + 7 * ny)
    src = smooth_source(nx, ny, seed=nx + 5 * ny, scale=1e-3 * float(np.sqrt(np.mean(v0.astype(np.float64) ** 2))) / dt)
    z0 = z0.astype(np.complex64)
    b = xfb.Backend(nx, ny, lx=lx, ly=ly)
    b.set_spectrum(z0)
    b.set_source(src)
    b.step(2, dt)
    got = b.get_spectrum()
    gfields = {k: b.get_field(w) for k, w in (("vort", xfb.capi.VORT), ("psi", xfb.capi.PSI), ("u", xfb.capi.U),
                                               ("v", xfb.capi.V), ("dvortdx", xfb.capi.DVORTDX), ("dvortdy", xfb.capi.DVORTDY))}
    b.close()
    want = z0.astype(np.complex128)
    for _ in range(2):
        want = ref_step(want, nx, ny, lx, ly, NU, dt, src=src)
    err = rel_l2(got, want)
    edges = edge_errors(got, want, nx, ny)
    print(f"{nx}x{ny} lx={lx:g} ly={ly:g}: spectrum {err:.2e}, " + ", ".join(f"{k} {v:.2e}" for k, v in edges.items()))
    assert err < 1e-5, err
    for k, e in edges.items():
        assert e < 1e-5, (k, e)
    wf = ref_fields(want, nx, ny, lx, ly)
    for k, g in gfields.items():
        assert rel_l2(g, wf[k]) < 1e-5, (k, rel_l2(g, wf[k]))


# ---- closed forms: a single mode has no Jacobian -------------------------------------------------------------------------
CLOSED_STEPS = 10


def closed_form_coefficients(nx, ny, lx, ly, dt, p, kref2=None):
    """beta dt / k_0 = 1 for the longest wave, mu dt = 0.01, nu_h k^(2p) dt = 0.02 at |k|^2 = kref2 unless that puts
    nu_h k^(2p) dt above 1 somewhere inside the mask (float32 roundoff of the Jacobian seeds every mode the mask keeps)"""
    kx, ky, lap, _, mask = tables(nx, ny, lx, ly)
    k2 = -lap.astype(np.float64)
    kedge2 = float(k2[mask > 0].max())
    kref2 = kedge2 / 16 if kref2 is None else kref2
    beta = 2 * np.pi / max(lx, ly) / dt
    nu_h = min(0.02 / (dt * kref2 ** p), 1.0 / (dt * kedge2 ** p))
    return beta, 0.01 / dt, nu_h, p


def closed_form_modes(nx, ny):
    """(i, j): a mode and its swapped-index twin, a negative kx, a Nyquist-line mode inside the mask, one outside it"""
    r = max(4, min(nx, ny) // 8)
    modes = [(r, r // 2 + 1), (r // 2 + 1, r), (nx - 7, 11)]
    kd = mask_kd(nx, ny)
    if 9 + (ny // 2) ** 2 < kd:
        modes.append((3, ny // 2))
    if (nx // 2) ** 2 + 9 < kd:
        modes.append((nx // 2, 3))
    modes.append((nx // 2 - 1, ny // 2))
    return modes


@pytest.mark.gpu
@pytest.mark.parametrize("nx,ny", SHAPES + LARGE, ids=_ids(SHAPES + LARGE))
def test_single_modes_follow_the_rk4_polynomial(xfb, nx, ny):
    need_host_memory(nx, ny, ref=False)
    lx, ly = LX, LY
    dt = step_dt(nx, ny)
    h = ny // 2 + 1
    modes = closed_form_modes(nx, ny)
    assert any(j == ny // 2 or i == nx // 2 for i, j in modes[3:-1]), "a Nyquist-line mode inside the mask"
    lap = tables(nx, ny, lx, ly)[2].astype(np.float64)
    inside = tables(nx, ny, lx, ly)[4] > 0
    amp = np.complex64(5e-5 * nx * ny * (0.8 + 0.6j))          # vorticity ~ 1e-4 / s: the Jacobian's roundoff stays tiny
    i0, j0 = modes[0]
    b = xfb.Backend(nx, ny, lx=lx, ly=ly)
    worst = 0.0
    for p in (1, 4):
        beta, mu, nu_h, _ = closed_form_coefficients(nx, ny, lx, ly, dt, p, kref2=-lap[i0, j0])
        b.set_linear_terms(beta, mu, nu_h, p)
        lam = lin_factor(nx, ny, lx, ly, beta, mu, nu_h, p) + NU * lap
        facs = {}
        for i, j in modes:
            z = np.zeros((nx, h), np.complex64)
            z[i, j] = amp
            b.set_spectrum(z)
            b.step(CLOSED_STEPS, dt)
            out = b.get_spectrum()
            got = complex(out[i, j])
            if inside[i, j]:
                exp = complex(amp) * rk4_poly(dt * lam[i, j]) ** CLOSED_STEPS
                e = abs(got - exp) / abs(exp)
                worst = max(worst, e)
                assert e < 1e-5, (p, i, j, got, exp, e)
                plain = complex(amp) * rk4_poly(dt * NU * lap[i, j]) ** CLOSED_STEPS
                assert abs(exp - plain) > 1e-3 * abs(exp), (p, i, j, "the linear terms must move the mode")
                facs[(i, j)] = exp
            else:
                assert got == complex(amp), (p, i, j, "outside the mask a mode is frozen")
            out[i, j] = 0
            leak = float(np.abs(out).max())
            assert leak <= 1e-8 * abs(amp), (p, i, j, leak)
            del out
        # the swapped pair: different rates on an lx != ly domain, each one as ref_step has it
        a, s = facs[modes[0]], facs[modes[1]]
        assert abs(a - s) > 1e-3 * abs(a)
    b.close()
    print(f"{nx}x{ny}: closed forms within {worst:.2e}")


# ---- ensembles ---------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("nx,ny", [(512, 2048), (2048, 256)], ids=_ids([(512, 2048), (2048, 256)]))
def test_ensemble_members_match_single_member_handles(xfb, nx, ny):
    lx, ly = LX, LY
    dt = step_dt(nx, ny)
    inits = [rough_field(nx, ny, lx, ly, seed=100 + m)[0] for m in range(3)]
    srcs = [smooth_source(nx, ny, seed=200 + m, scale=1e-9) for m in range(3)]
    ens = xfb.Backend(nx, ny, lx=lx, ly=ly, batch=3)
    for m in range(3):
        ens.set_vorticity(inits[m], member=m)
        ens.set_source(srcs[m], member=m)
    ens.step(3, dt)
    for m in range(3):
        one = xfb.Backend(nx, ny, lx=lx, ly=ly)
        one.set_vorticity(inits[m])
        one.set_source(srcs[m])
        one.step(3, dt)
        ref = one.get_spectrum()
        assert np.isfinite(ref.view(np.float32)).all()
        assert np.array_equal(ens.get_spectrum(member=m).view(np.float32), ref.view(np.float32)), m
        assert np.array_equal(ens.get_field(xfb.capi.U, member=m), one.get_field(xfb.capi.U)), m
        one.close()
    ens.close()


# ---- passive tracer ----------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("nx,ny", [(1024, 256), (256, 1024)], ids=_ids([(1024, 256), (256, 1024)]))
def test_tracer_on_rectangular_grids(xfb, nx, ny):
    lx, ly = LX, LY
    dt = step_dt(nx, ny)
    v0, _ = rough_field(nx, ny, lx, ly, seed=nx + ny)
    b = xfb.Backend(nx, ny, lx=lx, ly=ly)
    b.set_vorticity(v0)
    b.set_tracer(v0, NU)
    b.step(3, dt)
    assert np.array_equal(b.get_field(xfb.capi.TRACER), b.get_field(xfb.capi.VORT))
    c0 = rough_field(nx, ny, lx, ly, seed=nx + ny + 1)[0] * np.float32(50.0)
    b.set_vorticity(v0)
    b.set_tracer(c0, 20.0)
    b.step(1, dt)
    zv, zc = ref_step(_fft(v0.astype(np.float64)), nx, ny, lx, ly, NU, dt, C=_fft(c0.astype(np.float64)), kappa=20.0)
    got_c = b.get_field(xfb.capi.TRACER)
    assert rel_l2(got_c, _ifft(zc, nx, ny)) < 1e-5, rel_l2(got_c, _ifft(zc, nx, ny))
    assert rel_l2(b.get_field(xfb.capi.VORT), _ifft(zv, nx, ny)) < 1e-5
    b.close()


# ---- diagnostics and invariants --------------------------------------------------------------------------------------
def smooth_vortex(nx, ny):
    """an elliptical vortex with a wave on it: smooth, so the filamentation time is well conditioned on most of the grid"""
    x = (np.arange(nx) / nx)[:, None]
    y = (np.arange(ny) / ny)[None, :]
    return (1e-4 * np.exp(-((x - 0.45) ** 2 / 0.02 + (y - 0.55) ** 2 / 0.008)) * (1 + 0.3 * np.cos(6 * np.pi * x))
            + 2e-5 * np.sin(2 * np.pi * 3 * x) * np.cos(2 * np.pi * 2 * y)).astype(np.float32)


def ref_diagnostics(Z, nx, ny, lx, ly):
    """the definitions of oracle/barotropic_oracle.c orc_diagnostics in float64"""
    kx, ky, _, lapinv, _ = tables(nx, ny, lx, ly)
    KX, KY = kx.astype(np.float64)[:, None], ky.astype(np.float64)[None, :]
    psi = Z / lapinv.astype(np.float64)
    pxy = _ifft(-KX * KY * psi, nx, ny)
    pxx = _ifft(-KX * KX * psi, nx, ny)
    pyy = _ifft(-KY * KY * psi, nx, ny)
    s1, s2, z = -2 * pxy, pxx - pyy, pxx + pyy
    ss, zz = s1 * s1 + s2 * s2, z * z
    q, den = ss - zz, ss + zz
    tfil = np.where(q > 0, 2 / np.sqrt(np.where(q > 0, q, 1.0)), 0.0)
    deform = np.where(den > 0, q / np.where(den > 0, den, 1.0), 0.0)
    return tfil, deform


def shells(nx, ny, lx, ly):
    """shell index of every half-spectrum mode (DESIGN.md section 3; test_energy_spectrum.py's restatement)"""
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


def energy_reference(zh, nx, ny, lx, ly, nshells):
    """(totals [E, Z, P], e, z) of a half spectrum in float64 (test_energy_spectrum.py's restatement)"""
    kx, ky = tables(nx, ny, lx, ly)[:2]
    hy = ny // 2 + 1
    re = zh.real.astype(np.float64)
    im = zh.imag.astype(np.float64)
    w = np.full(hy, 2.0)
    w[0] = w[ny // 2] = 1.0
    zw = (re * re + im * im) * w[None, :]
    k2 = kx.astype(np.float64)[:, None] ** 2 + ky.astype(np.float64)[None, :] ** 2
    e = np.where(k2 > 0, zw / np.where(k2 > 0, k2, 1.0), 0.0)
    c = 1.0 / (2.0 * float(nx * ny) ** 2)
    totals = np.array([e.sum(), zw.sum(), (zw * k2).sum()]) * c
    s = shells(nx, ny, lx, ly).ravel()
    keep = s < nshells
    es = np.bincount(s[keep], e.ravel()[keep], minlength=nshells)[:nshells] * c
    zs = np.bincount(s[keep], zw.ravel()[keep], minlength=nshells)[:nshells] * c
    return totals, es, zs


@pytest.mark.gpu
@pytest.mark.parametrize("nx,ny", [(2048, 512), (512, 2048)], ids=_ids([(2048, 512), (512, 2048)]))
def test_diagnostics_histograms_and_energy_spectrum(xfb, nx, ny):
    lx, ly = LX, LY
    v0 = smooth_vortex(nx, ny)
    b = xfb.Backend(nx, ny, lx=lx, ly=ly)
    b.set_vorticity(v0)
    b.step(2, step_dt(nx, ny))
    zh = b.get_spectrum()
    Z = zh.astype(np.complex128)
    tfil, deform = ref_diagnostics(Z, nx, ny, lx, ly)
    gt, gd = b.diagnostics()
    assert rel_l2(gd, deform) < 1e-4, rel_l2(gd, deform)
    assert rel_l2(b.get_field(xfb.capi.DEFORM), deform) < 1e-4
    both = (tfil > 0) & (gt > 0) & (tfil < 1e6)
    assert both.mean() > 0.3
    assert rel_l2(gt[both], tfil[both]) < 1e-3, rel_l2(gt[both], tfil[both])
    gt2 = b.get_field(xfb.capi.TFIL)
    both2 = (tfil > 0) & (gt2 > 0) & (tfil < 1e6)
    assert rel_l2(gt2[both2], tfil[both2]) < 1e-3
    # effective-diffusivity histograms: the area element is (lx / nx)(ly / ny)
    lo, hi = float(v0.min()) - 1e-6, float(v0.max()) * 1.01
    area, g2 = b.keff_hist(64, lo, hi)
    assert abs(area.sum() - lx * ly) < 1e-6 * lx * ly, area.sum()
    kx, ky = tables(nx, ny, lx, ly)[:2]
    vort = _ifft(Z, nx, ny).astype(np.float32)
    grad2 = (_ifft(1j * kx.astype(np.float64)[:, None] * Z, nx, ny) ** 2 + _ifft(1j * ky.astype(np.float64)[None, :] * Z, nx, ny) ** 2)
    bins = np.clip(np.floor((vort - np.float32(lo)) * np.float32(64 / (np.float32(hi) - np.float32(lo)))).astype(np.int64), 0, 63)
    da = (lx / nx) * (ly / ny)
    a_ref = np.bincount(bins.ravel(), minlength=64) * da
    g_ref = np.bincount(bins.ravel(), grad2.ravel(), minlength=64) * da
    assert rel_l2(np.cumsum(area), np.cumsum(a_ref)) < 1e-3
    assert rel_l2(np.cumsum(g2), np.cumsum(g_ref)) < 1e-3
    # energy, enstrophy, palinstrophy and shell spectra on the fused layout
    tot, e, z = b.energy_spectrum()
    assert len(e) == xfb.capi.shells_all(nx, ny, lx, ly) == shells(nx, ny, lx, ly).max() + 1
    rt, re_, rz = energy_reference(zh, nx, ny, lx, ly, len(e))
    for k in range(3):
        assert abs(tot[k] - rt[k]) < 1e-10 * abs(rt[k]), (k, tot[k], rt[k])
    assert np.abs(e - re_).max() <= 1e-10 * rt[0]
    assert np.abs(z - rz).max() <= 1e-10 * rt[1]
    b.close()


# ---- slab decomposition ------------------------------------------------------------------------------------------------
LOOPBACK = [(512, 2048, 4, 2), (2048, 256, 2, 4), (256, 1024, 8, 1), (16384, 1024, 8, 4)]


@pytest.mark.gpu
@pytest.mark.parametrize("nx,ny,p,c", LOOPBACK, ids=[f"{a}x{b}-{p}ranks-{c}chunks" for a, b, p, c in LOOPBACK])
def test_loopback_team_matches_single_gpu(xfb, nx, ny, p, c):
    lx, ly = domain(nx, ny)
    dt = step_dt(nx, ny)
    v0, _ = rough_field(nx, ny, lx, ly, seed=nx + ny + p)
    src = smooth_source(nx, ny, seed=p * c, scale=1e-9)
    one = xfb.Backend(nx, ny, lx=lx, ly=ly)
    team = xfb.LoopbackTeam(nx, p, c, lx=lx, ny=ny, ly=ly)
    for hnd in (one, team):
        hnd.set_vorticity(v0)
        hnd.set_source(src)
        hnd.step(3, dt)
    for which in (xfb.capi.VORT, xfb.capi.PSI, xfb.capi.U, xfb.capi.V):
        a, b = one.get_field(which), team.get_field(which)
        assert rel_l2(b, a) < 2e-6, (which, rel_l2(b, a))
        assert np.abs(a - b).max() <= 2e-5 * np.abs(a).max(), which
    one.step(1, dt)
    team.step(1, dt)
    assert rel_l2(team.get_field(xfb.capi.VORT), one.get_field(xfb.capi.VORT)) < 2e-6
    one.close()
    team.close()

"""GPU parity of the generic mixed-radix path (csrc/xfb_generic.cu): grids the fused power-of-two kernels do not
serve, first of all the reference's own default NPTS = 768 = 3 * 256 (src/configuration.hpp:18).
Same tolerances as tests/test_gpu_parity.py."""
import numpy as np
import pytest

from conftest import rel_l2
import fields

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def xfb():
    import xlab_fftbarotropic_b200 as pkg
    return pkg


@pytest.fixture(scope="module")
def orc():
    from oracle import oracle
    return oracle


@pytest.mark.parametrize("n", [96, 768])
def test_tables_and_operators_bit_exact(xfb, orc, n):
    assert xfb.load().xfb_size_supported(n, n) == 2
    b, o = xfb.Backend(n), orc.Oracle(n)
    for which in range(5):
        assert np.array_equal(b.table(which), o.table(which)), f"table {which}"
    rng = np.random.default_rng(n)
    h = n // 2 + 1
    z = (rng.standard_normal((n, h)) + 1j * rng.standard_normal((n, h))).astype(np.complex64)
    for g, r in (("gradx", "gradx"), ("grady", "grady"), ("laplacian", "laplacian"), ("invertLaplacian", "invert_laplacian"),
                 ("dealiase", "dealias")):
        assert np.array_equal(getattr(b, g)(z).view(np.float32), getattr(o, r)(z).view(np.float32)), g
    b.close()


@pytest.mark.parametrize("n", [96, 360, 768])
def test_transforms(xfb, orc, n):
    rng = np.random.default_rng(n + 1)
    f = rng.standard_normal((n, n)).astype(np.float32)
    b, o = xfb.Backend(n), orc.Oracle(n)
    F = b.r2c(f)
    assert rel_l2(F, o.r2c(f)) < 5e-7
    assert rel_l2(F, np.fft.rfft2(f.astype(np.float64))) < 5e-7
    h = n // 2 + 1
    z = (rng.standard_normal((n, h)) + 1j * rng.standard_normal((n, h))).astype(np.complex64)
    assert rel_l2(b.c2r(z), o.c2r(z)) < 5e-7                     # non-Hermitian input: Im of DC / Nyquist dropped
    assert rel_l2(b.c2r(F) / np.float32(n * n), f) < 1e-6
    b.close()


@pytest.mark.parametrize("n,gen,steps", [(768, "elliptic", 1), (768, "kuo2004", 20), (96, "gaussian", 100)])
def test_step_parity_reference_default_grid(xfb, orc, n, gen, steps):
    v0 = fields.GENERATORS[gen](n)
    b, o = xfb.Backend(n), orc.Oracle(n)
    b.set_vorticity(v0)
    o.set_vorticity(v0)
    b.step(steps, 3.0)
    o.step(steps, 3.0)
    tol = 1e-5 if steps == 1 else 1e-4
    assert rel_l2(b.get_spectrum(), o.get_spectrum()) < tol
    for which in (xfb.capi.VORT, xfb.capi.PSI, xfb.capi.U, xfb.capi.V):
        assert rel_l2(b.get_field(which), o.get_field(which)) < tol, which
    b.close()


def test_source_and_pressure_on_768(xfb, orc):
    n = 768
    rng = np.random.default_rng(3)
    v0 = fields.elliptic(n)
    src = (1e-9 * rng.standard_normal((n, n))).astype(np.float32)
    b, o = xfb.Backend(n), orc.Oracle(n)
    for x in (b, o):
        x.set_vorticity(v0)
        x.set_source(src)
        x.step(2, 3.0)
    assert rel_l2(b.get_field(xfb.capi.VORT), o.get_field(orc.VORT)) < 1e-5
    psi = o.get_field(orc.PSI)
    pb = b.invert_pres(psi, 3, 5, 1.0, 1e-5)
    po = o.invert_pres(psi, 3, 5, 1.0, 1e-5)
    assert rel_l2(pb, po) < 1e-4
    b.close()


def test_field_ids_outside_the_header_are_rejected(xfb):
    """xfb_get_field / xfb_get_field_async take the field ids of include/xfb.h only: any other id fails with "bad field
    id" on the unfused record path (generic grids), whatever chains the library keeps for its own use.  Both entry points
    report a failure of the field computation as XFB_E_CUDA, the code they have always returned for it."""
    import ctypes as C
    n = 96
    b = xfb.Backend(n)
    b.set_vorticity(fields.elliptic(n))
    L = b._L
    out = np.empty((n, n), np.float32)
    p = C.c_void_p()
    assert L.xfb_host_alloc(C.byref(p), n * n) == 0
    t = C.c_int()
    for which in (-1, 10, 11, 12, 13, 42):
        assert L.xfb_get_field(b._h, 0, which, out.ctypes.data_as(C.c_void_p)) == -3, which
        assert b"bad field id" in L.xfb_last_error()
        assert L.xfb_get_field_async(b._h, 0, which, p, C.byref(t)) == -3, which
        assert b"bad field id" in L.xfb_last_error()
    assert np.isfinite(b.get_field(xfb.capi.DEFORM)).all()          # the handle is still usable
    L.xfb_host_free(p)
    b.close()

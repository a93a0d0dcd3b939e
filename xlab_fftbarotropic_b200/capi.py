"""ctypes binding of the C ABI (include/xfb.h) -- the same calls a cgo/JNI/C++ host would make.

The product path has no CPU fallback: if libxfb.so is missing this module raises, and if no CUDA
device is present xfb_create fails with XFB_E_CUDA.
"""
from __future__ import annotations

import ctypes as C
import math
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("XFB_LIB") or os.path.join(HERE, "libxfb.so")   # XFB_LIB: A/B builds of the same ABI

VORT, PSI, U, V, SRC, TFIL, DEFORM, DVORTDX, DVORTDY, TRACER = range(10)
TAB_GRADX, TAB_GRADY, TAB_LAP, TAB_LAPINV, TAB_MASK = range(5)

SYMBOLS = [
    "xfb_last_error", "xfb_create", "xfb_destroy", "xfb_sync", "xfb_gradx", "xfb_grady", "xfb_laplacian",
    "xfb_invert_laplacian", "xfb_dealias", "xfb_get_table", "xfb_r2c", "xfb_c2r", "xfb_set_vorticity",
    "xfb_set_spectrum", "xfb_get_spectrum", "xfb_set_source", "xfb_step", "xfb_get_field", "xfb_get_keff_hist", "xfb_get_diagnostics",
    "xfb_set_tracer", "xfb_get_tracer_keff_hist",
    "xfb_host_alloc", "xfb_host_free", "xfb_get_field_async", "xfb_wait_field",
    "xfb_invert_pres", "xfb_launch_count", "xfb_stream", "xfb_size_supported", "xfb_profile", "xfb_profile_read",
    "xfb_slab_partition", "xfb_nccl_unique_id", "xfb_create_dist", "xfb_profile_read_a2a", "xfb_slab_transport", "xfb_slab_fused",
    "xfb_loopback_create", "xfb_loopback_destroy", "xfb_loopback_set_vorticity", "xfb_loopback_set_source",
    "xfb_loopback_step", "xfb_loopback_get_field", "xfb_loopback_launch_count", "xfb_loopback_get_diagnostics",
    "xfb_loopback_get_keff_hist", "xfb_loopback_set_tracer",
    "xfb_get_energy_spectrum", "xfb_loopback_get_energy_spectrum",
    "xfb_set_linear_terms", "xfb_loopback_set_linear_terms",
]

_lib = None


class XfbError(RuntimeError):
    pass


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise XfbError(f"{LIB_PATH} is missing: build it with `python -m xlab_fftbarotropic_b200.build` "
                       "(there is no CPU fallback)")
    L = C.CDLL(LIB_PATH)
    vp, ci, cf = C.c_void_p, C.c_int, C.c_float
    L.xfb_last_error.restype = C.c_char_p
    L.xfb_create.argtypes = [C.POINTER(vp), ci, ci, cf, cf, cf, ci, ci]
    L.xfb_destroy.argtypes = [vp]
    L.xfb_sync.argtypes = [vp]
    for n in ("xfb_gradx", "xfb_grady", "xfb_laplacian", "xfb_invert_laplacian", "xfb_dealias", "xfb_r2c", "xfb_c2r"):
        getattr(L, n).argtypes = [vp, vp, vp]
    L.xfb_get_table.argtypes = [vp, ci, vp]
    L.xfb_set_vorticity.argtypes = [vp, ci, vp]
    L.xfb_set_spectrum.argtypes = [vp, ci, vp]
    L.xfb_get_spectrum.argtypes = [vp, ci, vp]
    L.xfb_set_source.argtypes = [vp, ci, vp]
    L.xfb_step.argtypes = [vp, ci, cf]
    L.xfb_get_field.argtypes = [vp, ci, ci, vp]
    L.xfb_get_diagnostics.argtypes = [vp, ci, vp, vp]
    L.xfb_host_alloc.argtypes = [C.POINTER(vp), C.c_size_t]
    L.xfb_host_free.argtypes = [vp]
    L.xfb_get_field_async.argtypes = [vp, ci, ci, vp, C.POINTER(ci)]
    L.xfb_wait_field.argtypes = [vp, ci]
    L.xfb_get_keff_hist.argtypes = [vp, ci, ci, cf, cf, vp, vp]
    L.xfb_get_tracer_keff_hist.argtypes = [vp, ci, ci, cf, cf, vp, vp]
    L.xfb_get_energy_spectrum.argtypes = [vp, ci, ci, ci, vp, vp, vp]
    L.xfb_loopback_get_energy_spectrum.argtypes = [vp, ci, ci, vp, vp, vp]
    L.xfb_set_tracer.argtypes = [vp, ci, vp, cf]
    L.xfb_set_linear_terms.argtypes = [vp, cf, cf, cf, ci]
    L.xfb_loopback_set_linear_terms.argtypes = [vp, cf, cf, cf, ci]
    L.xfb_invert_pres.argtypes = [vp, vp, vp, C.c_size_t, C.c_size_t, cf, cf]
    L.xfb_launch_count.restype = C.c_longlong
    L.xfb_launch_count.argtypes = [vp]
    L.xfb_stream.restype = vp
    L.xfb_stream.argtypes = [vp]
    L.xfb_size_supported.argtypes = [ci, ci]
    L.xfb_profile.argtypes = [vp, ci]
    L.xfb_profile_read.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(C.c_longlong), C.POINTER(C.c_double),
                                   C.POINTER(C.c_longlong)]
    ip = C.POINTER(ci)
    L.xfb_slab_partition.argtypes = [ci, ci, ci, ci, ci, ip, ip, ip, ip, ip, ip]
    L.xfb_nccl_unique_id.argtypes = [C.c_char_p]
    L.xfb_create_dist.argtypes = [C.POINTER(vp), ci, ci, cf, cf, cf, ci, ci, ci, ci, C.c_char_p]
    L.xfb_profile_read_a2a.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(C.c_longlong)]
    L.xfb_slab_transport.argtypes = [vp]
    L.xfb_slab_fused.argtypes = [vp]
    L.xfb_loopback_create.argtypes = [C.POINTER(vp), ci, ci, cf, cf, cf, ci, ci, ci]
    L.xfb_loopback_destroy.argtypes = [vp]
    L.xfb_loopback_set_vorticity.argtypes = [vp, vp]
    L.xfb_loopback_set_source.argtypes = [vp, vp]
    L.xfb_loopback_step.argtypes = [vp, ci, cf]
    L.xfb_loopback_get_field.argtypes = [vp, ci, vp]
    L.xfb_loopback_set_tracer.argtypes = [vp, vp, cf]
    L.xfb_loopback_get_diagnostics.argtypes = [vp, vp, vp]
    L.xfb_loopback_get_keff_hist.argtypes = [vp, ci, cf, cf, vp, vp]
    L.xfb_loopback_launch_count.restype = C.c_longlong
    L.xfb_loopback_launch_count.argtypes = [vp]
    _lib = L
    return L


def slab_partition(nx, ny, nranks, nchunks, rank):
    """-> dict(row0, rows, col0, cols, chunk_cols, pitch_global); pure host arithmetic (no GPU needed)"""
    L = load()
    v = [C.c_int() for _ in range(6)]
    rc = L.xfb_slab_partition(nx, ny, nranks, nchunks, rank, *[C.byref(x) for x in v])
    if rc != 0:
        raise XfbError(f"xfb error {rc}: {L.xfb_last_error().decode()}")
    return dict(zip(("row0", "rows", "col0", "cols", "chunk_cols", "pitch_global"), (x.value for x in v)))


def shells_all(nx, ny, lx, ly=None) -> int:
    """Number of isotropic shells that holds every mode of an nx x ny grid: the shell of (nx/2, ny/2) plus one
    (DESIGN.md section 3; pure host arithmetic)."""
    ly = lx if ly is None else ly
    lx, ly = float(np.float32(lx)), float(np.float32(ly))
    ip, j = nx // 2, ny // 2
    if lx == ly:
        m = ip * ip + j * j
        s = math.isqrt(m)
        return s + (1 if m > s * s + s else 0) + 1
    big = max(lx, ly)
    a, b = ip * (big / lx), j * (big / ly)
    return int(math.floor(math.sqrt(a * a + b * b) + 0.5)) + 1


def _energy_spectrum(L, call, nshells, nx, ny, lx, ly):
    n = shells_all(nx, ny, lx, ly) if nshells is None else int(nshells)
    totals = np.zeros(3, np.float64)
    e = np.zeros(n, np.float64)
    z = np.zeros(n, np.float64)
    rc = call(_ptr(totals), _ptr(e) if n else None, _ptr(z) if n else None, n)
    if rc != 0:
        raise XfbError(f"xfb error {rc}: {L.xfb_last_error().decode()}")
    return totals, e, z


def nccl_unique_id() -> bytes:
    L = load()
    buf = C.create_string_buffer(128)
    rc = L.xfb_nccl_unique_id(buf)
    if rc != 0:
        raise XfbError(f"xfb error {rc}: {L.xfb_last_error().decode()}")
    return buf.raw


def _ptr(a):
    """host numpy array or raw device address (int) -> void*"""
    if isinstance(a, (int, np.integer)):
        return C.c_void_p(int(a))
    return a.ctypes.data_as(C.c_void_p)


class Backend:
    """Mirror of the reference operator class `fftwf_operation<XPTS,YPTS>` (src/fftwfop.hpp:9-29) plus the
    2-D transforms and the RK4 driver of src/main.cpp, on one B200.  Arrays are numpy, reference layout."""

    def __init__(self, nx: int, ny: int | None = None, lx: float = 600000.0, ly: float | None = None,
                 nu: float = 6.5, batch: int = 1, device: int = 0):
        ny = nx if ny is None else ny
        ly = lx if ly is None else ly
        self.nx, self.ny, self.hy, self.batch = nx, ny, ny // 2 + 1, batch
        self.lx, self.ly, self.nu = lx, ly, nu
        self._L = load()
        self._h = C.c_void_p()
        self._ck(self._L.xfb_create(C.byref(self._h), nx, ny, lx, ly, nu, batch, device))

    def _ck(self, rc):
        if rc != 0:
            raise XfbError(f"xfb error {rc}: {self._L.xfb_last_error().decode()}")

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self._L.xfb_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- operator tier ---------------------------------------------------------------------------
    def _spec(self, a):
        return np.ascontiguousarray(a, dtype=np.complex64).reshape(self.nx, self.hy)

    def _op(self, name, a):
        a = self._spec(a)
        out = np.empty_like(a)
        self._ck(getattr(self._L, name)(self._h, _ptr(a), _ptr(out)))
        return out

    def gradx(self, a): return self._op("xfb_gradx", a)
    def grady(self, a): return self._op("xfb_grady", a)
    def laplacian(self, a): return self._op("xfb_laplacian", a)
    def invertLaplacian(self, a): return self._op("xfb_invert_laplacian", a)
    def dealiase(self, a): return self._op("xfb_dealias", a)

    def table(self, which):
        shape = {0: (self.nx,), 1: (self.hy,)}.get(which, (self.nx, self.hy))
        out = np.empty(shape, np.float32)
        self._ck(self._L.xfb_get_table(self._h, which, _ptr(out)))
        return out

    def r2c(self, f):
        f = np.ascontiguousarray(f, dtype=np.float32).reshape(self.nx, self.ny)
        out = np.empty((self.nx, self.hy), np.complex64)
        self._ck(self._L.xfb_r2c(self._h, _ptr(f), _ptr(out)))
        return out

    def c2r(self, a):
        a = self._spec(a)
        out = np.empty((self.nx, self.ny), np.float32)
        self._ck(self._L.xfb_c2r(self._h, _ptr(a), _ptr(out)))
        return out

    # -- stepper tier ----------------------------------------------------------------------------
    def set_vorticity(self, f, member=0):
        if not isinstance(f, (int, np.integer)):
            f = np.ascontiguousarray(f, dtype=np.float32).reshape(self.nx, self.ny)
        self._ck(self._L.xfb_set_vorticity(self._h, member, _ptr(f)))

    def set_spectrum(self, z, member=0):
        z = self._spec(z)
        self._ck(self._L.xfb_set_spectrum(self._h, member, _ptr(z)))

    def get_spectrum(self, member=0):
        out = np.empty((self.nx, self.hy), np.complex64)
        self._ck(self._L.xfb_get_spectrum(self._h, member, _ptr(out)))
        return out

    def set_source(self, s, member=0):
        if s is None:
            self._ck(self._L.xfb_set_source(self._h, member, None))
        else:
            s = np.ascontiguousarray(s, dtype=np.float32).reshape(self.nx, self.ny)
            self._ck(self._L.xfb_set_source(self._h, member, _ptr(s)))

    def set_linear_terms(self, beta=0.0, mu=0.0, nu_h=0.0, order=4):
        """-beta v - mu zeta - nu_h (-lap)^order zeta added to the vorticity tendency of every member (DESIGN.md
        section 3); all zeros switches them off.  Slab ranks: every rank passes the same values."""
        self._ck(self._L.xfb_set_linear_terms(self._h, float(beta), float(mu), float(nu_h), int(order)))

    def step(self, nsteps, dt):
        self._ck(self._L.xfb_step(self._h, int(nsteps), float(dt)))

    def sync(self):
        self._ck(self._L.xfb_sync(self._h))

    def get_field(self, which, member=0, out=None):
        if out is None:
            out = np.empty((self.nx, self.ny), np.float32)
        self._ck(self._L.xfb_get_field(self._h, member, which, _ptr(out)))
        return out

    def get_field_async(self, which, pinned_ptr, member=0):
        """enqueue field -> pinned host buffer (address from xfb_host_alloc); returns a ticket for wait_field"""
        t = C.c_int()
        self._ck(self._L.xfb_get_field_async(self._h, member, which, C.c_void_p(pinned_ptr), C.byref(t)))
        return t.value

    def wait_field(self, ticket):
        self._ck(self._L.xfb_wait_field(self._h, ticket))

    def diagnostics(self, member=0):
        """-> (filamentation time, deformation factor), sharing the three second derivatives of psi"""
        t = np.empty((self.nx, self.ny), np.float32)
        d = np.empty((self.nx, self.ny), np.float32)
        self._ck(self._L.xfb_get_diagnostics(self._h, member, _ptr(t), _ptr(d)))
        return t, d

    def keff_hist(self, nbins, cmin, cmax, member=0):
        area = np.zeros(nbins, np.float64)
        g2 = np.zeros(nbins, np.float64)
        self._ck(self._L.xfb_get_keff_hist(self._h, member, nbins, cmin, cmax, _ptr(area), _ptr(g2)))
        return area, g2

    def energy_spectrum(self, nshells=None, which=VORT, member=0):
        """-> (totals [E, Z, P], e[nshells], z[nshells]): domain-mean kinetic energy, enstrophy, palinstrophy and the
        shell sums of E and Z (float64); nshells=None: every shell (shells_all).  which = VORT or TRACER."""
        return _energy_spectrum(self._L, lambda t, e, z, n: self._L.xfb_get_energy_spectrum(self._h, member, which, n, t, e, z),
                                nshells, self.nx, self.ny, self.lx, self.ly)

    # passive tracer: advected by xfb_step with the flow of each stage; read back with get_field(TRACER)
    def set_tracer(self, c, kappa, member=0):
        c = np.ascontiguousarray(c, dtype=np.float32).reshape(self.nx, self.ny)
        self._ck(self._L.xfb_set_tracer(self._h, member, _ptr(c), float(kappa)))

    def tracer_keff_hist(self, nbins, cmin, cmax, member=0):
        area = np.zeros(nbins, np.float64)
        g2 = np.zeros(nbins, np.float64)
        self._ck(self._L.xfb_get_tracer_keff_hist(self._h, member, nbins, cmin, cmax, _ptr(area), _ptr(g2)))
        return area, g2

    def invert_pres(self, psi, ref_x=0, ref_y=0, rho=1.0, f=1e-5):
        psi = np.ascontiguousarray(psi, dtype=np.float32).reshape(self.nx, self.ny)
        out = np.empty((self.nx, self.ny), np.float32)
        self._ck(self._L.xfb_invert_pres(self._h, _ptr(psi), _ptr(out), ref_x, ref_y, rho, f))
        return out

    def profile(self, enable=True):
        self._ck(self._L.xfb_profile(self._h, 1 if enable else 0))

    def profile_read(self):
        """-> dict(row_ms, row_launches, col_ms, col_launches) summed since profile(True)"""
        rm, cm = C.c_double(), C.c_double()
        rl, cl = C.c_longlong(), C.c_longlong()
        self._ck(self._L.xfb_profile_read(self._h, C.byref(rm), C.byref(rl), C.byref(cm), C.byref(cl)))
        return {"row_ms": rm.value, "row_launches": rl.value, "col_ms": cm.value, "col_launches": cl.value}

    @property
    def launch_count(self):
        return int(self._L.xfb_launch_count(self._h))

    @property
    def stream(self):
        return self._L.xfb_stream(self._h)


class SlabBackend(Backend):
    """One rank of a slab-decomposed grid (one process per GPU, NCCL all-to-all).  Fields are the LOCAL rows."""

    def __init__(self, n: int, rank: int, nranks: int, unique_id: bytes, nchunks: int = 8, lx: float = 600000.0,
                 nu: float = 6.5, device: int = 0, ny: int | None = None, ly: float | None = None):
        """n x ny grid (ny = n by default) on an lx x ly domain (ly = lx by default); n rows are split over the ranks"""
        ny = n if ny is None else ny
        ly = lx if ly is None else ly
        self.nx, self.ny, self.hy, self.batch = n, ny, ny // 2 + 1, 1
        self.lx, self.ly, self.nu = lx, ly, nu
        self.rank, self.nranks = rank, nranks
        self.part = slab_partition(n, ny, nranks, nchunks, rank) if nranks > 1 else dict(row0=0, rows=n)
        self.rows = self.part["rows"]
        self._L = load()
        self._h = C.c_void_p()
        self._ck(self._L.xfb_create_dist(C.byref(self._h), n, ny, lx, ly, nu, device, rank, nranks, nchunks, unique_id))

    def set_vorticity(self, f, member=0):
        if not isinstance(f, (int, np.integer)):
            f = np.ascontiguousarray(f, dtype=np.float32).reshape(self.rows, self.ny)
        self._ck(self._L.xfb_set_vorticity(self._h, 0, _ptr(f)))

    def get_field(self, which, member=0, out=None):
        if out is None:
            out = np.empty((self.rows, self.ny), np.float32)
        self._ck(self._L.xfb_get_field(self._h, 0, which, _ptr(out)))
        return out

    def set_tracer(self, c, kappa, member=0):
        if not isinstance(c, (int, np.integer)):
            c = np.ascontiguousarray(c, dtype=np.float32).reshape(self.rows, self.ny)
        self._ck(self._L.xfb_set_tracer(self._h, 0, _ptr(c), float(kappa)))

    def diagnostics(self, member=0):
        t = np.empty((self.rows, self.ny), np.float32)
        d = np.empty((self.rows, self.ny), np.float32)
        self._ck(self._L.xfb_get_diagnostics(self._h, 0, _ptr(t), _ptr(d)))
        return t, d

    @property
    def transport(self):
        t = {0: "none", 1: "nccl send/recv", 2: "p2p copy engines (CUDA IPC)", 3: "p2p SM push kernel (CUDA IPC)"}[int(self._L.xfb_slab_transport(self._h))]
        if self.fused:
            t += " for column->row, row->column fused into K-ROW (stores into peer memory)"
        return t

    @property
    def fused(self):
        """1: row->column transpose fused into K-ROW, else 0"""
        return int(self._L.xfb_slab_fused(self._h))

    def a2a_read(self):
        ms, n = C.c_double(), C.c_longlong()
        self._ck(self._L.xfb_profile_read_a2a(self._h, C.byref(ms), C.byref(n)))
        return {"a2a_ms": ms.value, "exchanges": n.value}


class LoopbackTeam:
    """All ranks of a slab decomposition in one process on one device (verification of the slab indexing
    on a single GPU; same kernels as the NCCL path, the exchange is a set of device copies)."""

    def __init__(self, n: int, nranks: int, nchunks: int = 1, lx: float = 600000.0, nu: float = 6.5, device: int = 0,
                 ny: int | None = None, ly: float | None = None):
        """n x ny grid (ny = n by default) on an lx x ly domain (ly = lx by default); n rows are split over the ranks"""
        ny = n if ny is None else ny
        ly = lx if ly is None else ly
        self.nx, self.ny, self.lx, self.ly = n, ny, lx, ly
        self._L = load()
        self._t = C.c_void_p()
        self._ck(self._L.xfb_loopback_create(C.byref(self._t), n, ny, lx, ly, nu, device, nranks, nchunks))

    def _ck(self, rc):
        if rc != 0:
            raise XfbError(f"xfb error {rc}: {self._L.xfb_last_error().decode()}")

    def close(self):
        if getattr(self, "_t", None) and self._t.value:
            self._L.xfb_loopback_destroy(self._t)
            self._t = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_vorticity(self, f):
        f = np.ascontiguousarray(f, dtype=np.float32).reshape(self.nx, self.ny)
        self._ck(self._L.xfb_loopback_set_vorticity(self._t, _ptr(f)))

    def set_source(self, s):
        if s is None:
            self._ck(self._L.xfb_loopback_set_source(self._t, None))
        else:
            s = np.ascontiguousarray(s, dtype=np.float32).reshape(self.nx, self.ny)
            self._ck(self._L.xfb_loopback_set_source(self._t, _ptr(s)))

    def set_tracer(self, c, kappa):
        c = np.ascontiguousarray(c, dtype=np.float32).reshape(self.nx, self.ny)
        self._ck(self._L.xfb_loopback_set_tracer(self._t, _ptr(c), float(kappa)))

    def set_linear_terms(self, beta=0.0, mu=0.0, nu_h=0.0, order=4):
        """Backend.set_linear_terms on every rank"""
        self._ck(self._L.xfb_loopback_set_linear_terms(self._t, float(beta), float(mu), float(nu_h), int(order)))

    def step(self, nsteps, dt):
        self._ck(self._L.xfb_loopback_step(self._t, int(nsteps), float(dt)))

    def get_field(self, which):
        out = np.empty((self.nx, self.ny), np.float32)
        self._ck(self._L.xfb_loopback_get_field(self._t, which, _ptr(out)))
        return out

    def diagnostics(self):
        t = np.empty((self.nx, self.ny), np.float32)
        d = np.empty((self.nx, self.ny), np.float32)
        self._ck(self._L.xfb_loopback_get_diagnostics(self._t, _ptr(t), _ptr(d)))
        return t, d

    def keff_hist(self, nbins, cmin, cmax):
        area = np.zeros(nbins, np.float64)
        g2 = np.zeros(nbins, np.float64)
        self._ck(self._L.xfb_loopback_get_keff_hist(self._t, nbins, cmin, cmax, _ptr(area), _ptr(g2)))
        return area, g2

    def energy_spectrum(self, nshells=None, which=VORT):
        """whole-domain (totals, e, z) as Backend.energy_spectrum"""
        return _energy_spectrum(self._L, lambda t, e, z, n: self._L.xfb_loopback_get_energy_spectrum(self._t, which, n, t, e, z),
                                nshells, self.nx, self.ny, self.lx, self.ly)

    @property
    def launch_count(self):
        return int(self._L.xfb_loopback_launch_count(self._t))

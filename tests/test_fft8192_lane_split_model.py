"""CPU model of the 8192-point line transforms with two shared-memory exchanges (csrc/xfb_fft.cuh, Split8192,
fft8192_to_split, fft8192_from_split), used by K-ROW and K-COL of the 8192^2 stepper.  Thread t of a 512-thread line
holds 16 complex values; the third radix-16 pass is run by the remapped Stockham thread tau(t) and the final radix-2
stage is split across the lane pair (t, t ^ 16).  Checked here in float64, without a GPU:
  * the split order is a bijection onto the 8192 positions;
  * natural -> split and split -> natural, step by step as the kernels do them, reproduce numpy.fft.fft;
  * every shared-memory write and read of both exchanges is conflict-free per half warp of 8-byte accesses with the
    padded layout pos + pos // 16;
  * every shuffle partner is in the same warp."""
import numpy as np

L, G = 8192, 512
T = np.arange(G)
H = (T >> 4) & 1                                   # lane half
J0 = ((T >> 5) << 4) | (T & 15)
TAU = (H << 8) | J0                                # Stockham thread of the third radix-16 pass
BASE = J0 + (H << 11)


def off(k):
    return ((k & 7) << 8) + ((k >> 3) << 12)


def pos(t, k):
    return BASE[t] + off(k)


def padpos(p):
    return p + (p >> 4)


def w(n, x):
    return np.exp(-2j * np.pi * np.asarray(x, dtype=np.float64) / n)


W32 = w(32, np.arange(8))
PARTNER = T ^ 16
# twiddle bases of Split8192::init_tw: b1 for the second pass, b2 (negated on lane half 1) for the third, b0 for the pair
B1 = w(256, T & 15)
B2 = np.where(H == 1, -1.0, 1.0) * w(4096, J0)
B0 = w(L, BASE)


def dft16(v):
    return np.fft.fft(v, axis=1)


def twiddle(v, b):
    return v * b[:, None] ** np.arange(16)[None, :]


def stockham_positions(t, ns):
    """exchange_write / exchange_read_stockham: slot s of thread t at (t // ns) * ns * 16 + t % ns + s * ns"""
    return ((t // ns) * ns * 16 + t % ns)[:, None] + np.arange(16)[None, :] * ns


def strided_positions(t):
    """exchange_read / exchange_write_strided: slot k of thread t at t + k * G"""
    return t[:, None] + np.arange(16)[None, :] * G


def exchange(v, write_pos, read_pos):
    buf = np.full(L + L // 16, np.nan, dtype=complex)
    buf[padpos(write_pos)] = v
    return buf[padpos(read_pos)]


def to_split(x):
    v = x[strided_positions(T)]
    v = dft16(v)
    v = exchange(v, stockham_positions(T, 1), strided_positions(T))
    v = dft16(twiddle(v, B1))
    v = exchange(v, stockham_positions(T, 16), strided_positions(TAU))
    v = dft16(twiddle(v, B2))
    out = v.copy()
    for i in range(8):
        r = v[PARTNER, 8 + i]                       # shfl.xor 16 of slot 8 + i
        e = np.where(H == 1, r, v[:, i])
        o = np.where(H == 1, v[:, i], r)
        b = o * (B0 * W32[i])
        out[:, i], out[:, 8 + i] = e + b, e - b
    return out


def from_split(v):
    v = v.copy()
    keep, send = np.empty((G, 8), complex), np.empty((G, 8), complex)
    for i in range(8):
        a = v[:, i] + v[:, 8 + i]
        b = (v[:, i] - v[:, 8 + i]) * (B0 * W32[i])
        keep[:, i] = np.where(H == 1, b, a)
        send[:, i] = np.where(H == 1, a, b)
    v[:, :8] = keep
    v[:, 8:] = send[PARTNER]
    v = twiddle(dft16(v), B2)
    v = exchange(v, strided_positions(TAU), stockham_positions(T, 16))
    v = twiddle(dft16(v), B1)
    v = exchange(v, strided_positions(T), stockham_positions(T, 1))
    return dft16(v)


def _signal(seed):
    rng = np.random.default_rng(seed)
    return rng.standard_normal(L) + 1j * rng.standard_normal(L)


def test_split_order_is_a_bijection():
    p = pos(T[:, None], np.arange(16)[None, :])
    assert np.array_equal(np.sort(p.ravel()), np.arange(L))
    assert np.array_equal(p, BASE[:, None] + np.array([off(k) for k in range(16)])[None, :])


def test_natural_to_split_is_the_dft():
    x = _signal(1)
    ref = np.fft.fft(x)
    out = to_split(x)
    got = np.empty(L, complex)
    got[pos(T[:, None], np.arange(16)[None, :])] = out
    assert np.max(np.abs(got - ref)) <= 1e-12 * np.max(np.abs(ref))


def test_split_to_natural_is_the_dft():
    x = _signal(2)
    ref = np.fft.fft(x)
    got = np.empty(L, complex)
    got[strided_positions(T)] = from_split(x[pos(T[:, None], np.arange(16)[None, :])])
    assert np.max(np.abs(got - ref)) <= 1e-12 * np.max(np.abs(ref))


def test_to_split_then_from_split_is_a_scaled_reversal():
    """two forward transforms: F(F(x))[n] = L x[-n], through the split order in between"""
    x = _signal(3)
    y = np.empty(L, complex)
    y[strided_positions(T)] = from_split(to_split(x))
    assert np.max(np.abs(y / L - x[(-np.arange(L)) % L])) <= 1e-12 * np.max(np.abs(x))


def _conflict_free(positions):
    for warp in range(G // 32):
        for half in range(2):
            rows = positions[32 * warp + 16 * half: 32 * warp + 16 * half + 16]
            for k in range(16):
                if np.unique(padpos(rows[:, k]) % 16).size != 16:     # 16 bank pairs of one 128-byte wavefront
                    return False
    return True


def test_exchanges_are_conflict_free():
    for p in (stockham_positions(T, 1), strided_positions(T), stockham_positions(T, 16), strided_positions(TAU)):
        assert _conflict_free(p)


def test_shuffle_partners_share_a_warp():
    assert np.array_equal(PARTNER >> 5, T >> 5)
    assert np.array_equal(J0[PARTNER], J0) and np.array_equal(H[PARTNER], 1 - H)

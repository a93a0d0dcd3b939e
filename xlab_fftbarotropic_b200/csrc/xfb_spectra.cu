// xfb_spectra.cu -- quadratic invariants of the spectral state and their isotropic shell spectra (xfb_get_energy_spectrum;
// no reference counterpart, definitions in DESIGN.md section 3).
//
// One read of one member's state array, float64 throughout.  Every state layout of the library is one 2-D view
// [W walk steps][Q elements], element (w, q) at w * Q + q:
//   tile-major (tw_state = T > 0): w = global column tile (chunk c of a slab handle starts at tile c * pitch / T, so the
//     chunks continue seamlessly), q = i * T + column-in-tile, global column col0 + w * T + q % T;
//   row-major (tw_state = 0, the generic path): w = i, q = j, Q = pitch.
// A warp owns 32 consecutive q and walks w, one coalesced 256-byte load per step.  Along the walk a lane keeps a run
// (shell, E sum, Z sum) and hands it on only when its shell changes, so neighbours along w in one shell cost nothing; the
// runs handed on in one step are merged across the warp by a segmented scan over the lanes of one column (neighbours
// along q in one shell), and only the run tails add into a per-CTA float64 histogram in shared memory.  Each CTA covers
// a compact box of the (i, j) plane and flushes its non-zero histogram entries with one global atomic each.
#include <cmath>

#include "xfb_handle.h"

namespace xfb {

constexpr int SP_THREADS = 512;
constexpr int SP_WALK = 32;          // walk steps of one warp task
constexpr int SP_UNROLL = 8;         // loads in flight per lane
constexpr int SP_BOX_Q = 16;         // warp tasks per CTA box along q ...
constexpr int SP_BOX_W = 8;          // ... and along w
constexpr unsigned SP_NONE = 0xffffffffu;
constexpr unsigned SP_FULL = 0xffffffffu;

struct SpecParams {
    const cpx *z;                    // member's state array
    const double *kx2, *ky2;         // squared float32 wavenumbers (ky2 indexed by the global column)
    double *out;                     // [3 + 2 * nshells]: raw sums of E, Z, P, then e[nshells], z[nshells]
    long long Q;                     // elements per walk step
    int W;                           // walk steps
    int T;                           // tile width (tile-major) or 0 (row-major)
    int tshift;                      // log2(T)
    int nx, ny, hy, col0;
    int nshells, nsm;                // shells wanted, of which the first nsm are held in shared memory
    int square;                      // lx == ly: integer shell rule
    double rx, ry;                   // L / lx, L / ly (float64 rule)
};

// shell of mode (i', j): see DESIGN.md section 3
__device__ __forceinline__ unsigned shell_of(const SpecParams &p, int ip, int j)
{
    if (p.square) {
        const unsigned m = (unsigned)ip * (unsigned)ip + (unsigned)j * (unsigned)j;      // < 2^31 up to 16384^2
        unsigned s = (unsigned)__fsqrt_rn((float)m);
        while (s * s > m) --s;
        while ((s + 1) * (s + 1) <= m) ++s;
        return s + (m > s * s + s ? 1u : 0u);
    }
    const double a = __dmul_rn((double)ip, p.rx), b = __dmul_rn((double)j, p.ry);
    const double r = __dsqrt_rn(__dadd_rn(__dmul_rn(a, a), __dmul_rn(b, b)));
    return (unsigned)floor(__dadd_rn(r, 0.5));
}

// runs (key, e, z) handed on by the lanes of one warp: a segmented inclusive scan over the lanes of one column (lane
// stride ts) leaves each run's sum in its last lane, which adds it to the histogram
template <int TS>
__device__ __forceinline__ void warp_flush(const SpecParams &p, double *sh, unsigned key, double e, double z, int lane)
{
    const unsigned prev = __shfl_up_sync(SP_FULL, key, TS);
    const bool head = lane < TS || prev != key;
    const unsigned H = __ballot_sync(SP_FULL, head);
    constexpr unsigned seq = TS == 1 ? 0xffffffffu : (TS == 2 ? 0x55555555u : 0x11111111u);
    const unsigned below = lane == 31 ? 0xffffffffu : ((2u << lane) - 1u);
    const int hl = 31 - __clz(H & (seq << (lane % TS)) & below);
#pragma unroll
    for (int d = TS; d < 32; d <<= 1) {
        const double xe = __shfl_up_sync(SP_FULL, e, d), xz = __shfl_up_sync(SP_FULL, z, d);
        if (lane - d >= hl) { e += xe; z += xz; }
    }
    const bool tail = lane + TS >= 32 || ((H >> (lane + TS)) & 1u);
    if (tail && key != SP_NONE) {
        if ((int)key < p.nsm) {
            atomicAdd(&sh[key], e);
            atomicAdd(&sh[p.nsm + key], z);
        } else {
            atomicAdd(&p.out[3 + key], e);
            atomicAdd(&p.out[3 + p.nshells + key], z);
        }
    }
}

template <bool SHELLS, int TS>
__global__ void __launch_bounds__(SP_THREADS) energy_spectrum_kernel(const SpecParams p)
{
    extern __shared__ double sp_hist[];          // [2 * nsm]: e then z of the shells held here
    __shared__ double sp_tot[SP_THREADS / 32][3];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (SHELLS) {
        for (int k = threadIdx.x; k < 2 * p.nsm; k += SP_THREADS) sp_hist[k] = 0.0;
        __syncthreads();
    }
    const int G = (int)((p.Q + 31) / 32), S = (p.W + SP_WALK - 1) / SP_WALK;
    const int boxes_q = (G + SP_BOX_Q - 1) / SP_BOX_Q;
    const int bq = blockIdx.x % boxes_q, bw = blockIdx.x / boxes_q;
    double te = 0.0, tz = 0.0, tp = 0.0;
    for (int task = warp; task < SP_BOX_Q * SP_BOX_W; task += SP_THREADS / 32) {
        const int g = bq * SP_BOX_Q + task % SP_BOX_Q, s = bw * SP_BOX_W + task / SP_BOX_Q;
        if (g >= G || s >= S) continue;                  // warp-uniform
        const long long q = (long long)g * 32 + lane;
        int i, jin;                                       // row; column within the tile (tile-major) or column (row-major)
        if (p.T) { i = (int)(q >> p.tshift); jin = (int)(q & (p.T - 1)); }
        else { i = 0; jin = (int)q; }
        const bool qok = q < p.Q;
        unsigned cur = SP_NONE;
        double ae = 0.0, az = 0.0;
        const int w0 = s * SP_WALK;
        for (int k0 = 0; k0 < SP_WALK; k0 += SP_UNROLL) {
            cpx v[SP_UNROLL];
            bool ok[SP_UNROLL];
#pragma unroll
            for (int u = 0; u < SP_UNROLL; ++u) {
                const int w = w0 + k0 + u;
                const int j = p.T ? p.col0 + w * p.T + jin : jin;
                ok[u] = qok && w < p.W && j < p.hy;
                v[u] = ok[u] ? __ldg(p.z + (size_t)w * p.Q + q) : mk(0.f, 0.f);
            }
#pragma unroll
            for (int u = 0; u < SP_UNROLL; ++u) {
                const int w = w0 + k0 + u;
                const int ii = p.T ? i : w, j = p.T ? p.col0 + w * p.T + jin : jin;
                double ke = 0.0, kz = 0.0;
                unsigned key = SP_NONE;
                if (ok[u]) {
                    const double z2 = (double)v[u].x * (double)v[u].x + (double)v[u].y * (double)v[u].y;
                    const double zw = (j == 0 || 2 * j == p.ny) ? z2 : 2.0 * z2;
                    const double k2 = __ldg(p.kx2 + ii) + __ldg(p.ky2 + j);
                    ke = k2 > 0.0 ? zw / k2 : 0.0;
                    kz = zw;
                    te += ke; tz += kz; tp += zw * k2;
                    if (SHELLS) {
                        const int ip = ii <= p.nx - ii ? ii : p.nx - ii;
                        const unsigned sh = shell_of(p, ip, j);
                        key = sh < (unsigned)p.nshells ? sh : SP_NONE;       // beyond the shells asked for: totals only
                    }
                }
                if (SHELLS) {
                    const bool starts = key != SP_NONE && key != cur;
                    const unsigned fkey = starts ? cur : SP_NONE;
                    if (__ballot_sync(SP_FULL, fkey != SP_NONE)) warp_flush<TS>(p, sp_hist, fkey, ae, az, lane);
                    if (starts) { cur = key; ae = ke; az = kz; }
                    else if (key != SP_NONE) { ae += ke; az += kz; }
                }
            }
        }
        if (SHELLS && __ballot_sync(SP_FULL, cur != SP_NONE)) warp_flush<TS>(p, sp_hist, cur, ae, az, lane);
    }
    // totals: warp shuffles, then one atomic per CTA and quantity
#pragma unroll
    for (int o = 16; o; o >>= 1) {
        te += __shfl_xor_sync(SP_FULL, te, o);
        tz += __shfl_xor_sync(SP_FULL, tz, o);
        tp += __shfl_xor_sync(SP_FULL, tp, o);
    }
    if (lane == 0) { sp_tot[warp][0] = te; sp_tot[warp][1] = tz; sp_tot[warp][2] = tp; }
    __syncthreads();
    if (threadIdx.x < 3) {
        double t = 0.0;
        for (int w = 0; w < SP_THREADS / 32; ++w) t += sp_tot[w][threadIdx.x];
        atomicAdd(&p.out[threadIdx.x], t);
    }
    if (SHELLS) {
        for (int k = threadIdx.x; k < p.nsm; k += SP_THREADS) {
            if (sp_hist[k] != 0.0) atomicAdd(&p.out[3 + k], sp_hist[k]);
            if (sp_hist[p.nsm + k] != 0.0) atomicAdd(&p.out[3 + p.nshells + k], sp_hist[p.nsm + k]);
        }
    }
}

constexpr int SP_SMEM_MAX = 200 * 1024;          // histogram bytes per CTA (the rest of the 227 KB stays free)

template <bool SHELLS, int TS>
static int launch_variant(const SpecParams &p, unsigned grid, int smem, cudaStream_t st)
{
    static PerDeviceInt configured;
    int err = 0;
    if (SHELLS && configured.get([](int *e) -> int {
            cudaError_t r = cudaFuncSetAttribute(energy_spectrum_kernel<SHELLS, TS>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                 SP_SMEM_MAX);
            if (r != cudaSuccess) { *e = (int)r; return 0; }
            return 1;
        }, &err) <= 0)
        return fail(XFB_E_CUDA, "energy_spectrum_kernel: %s", cudaGetErrorString((cudaError_t)err));
    energy_spectrum_kernel<SHELLS, TS><<<grid, SP_THREADS, smem, st>>>(p);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(XFB_E_CUDA, "energy_spectrum_kernel: %s", cudaGetErrorString(e));
    return 0;
}

// shell index by the rule of DESIGN.md section 3, on the host
static long long shell_host(long long ip, long long j, float lx, float ly)
{
    if (lx == ly) {
        const long long m = ip * ip + j * j;
        long long s = (long long)std::sqrt((double)m);
        while (s * s > m) --s;
        while ((s + 1) * (s + 1) <= m) ++s;
        return s + (m > s * s + s ? 1 : 0);
    }
    const double L = lx > ly ? (double)lx : (double)ly;
    const double a = (double)ip * (L / (double)lx), b = (double)j * (L / (double)ly);
    volatile double aa = a * a, bb = b * b;       // no contraction: the device rounds each operation
    volatile double sum = aa + bb;
    volatile double r = std::sqrt((double)sum);
    return (long long)std::floor((double)r + 0.5);
}

long long shells_all(int nx, int ny, float lx, float ly) { return shell_host(nx / 2, ny / 2, lx, ly) + 1; }

int launch_energy_spectrum(xfb_handle h, const cpx *state, int nshells, double *d_out)
{
    SpecParams p;
    p.z = state; p.kx2 = h->kx2; p.ky2 = h->ky2; p.out = d_out;
    p.T = h->tw_state;
    p.tshift = p.T == 4 ? 2 : (p.T == 2 ? 1 : 0);
    if (p.T) { p.Q = (long long)h->nx * p.T; p.W = h->pitch / p.T * h->nchunks; }
    else { p.Q = h->pitch; p.W = h->nx; }
    p.nx = h->nx; p.ny = h->ny; p.hy = h->hy; p.col0 = h->col0;
    p.nshells = nshells;
    const long long all = shells_all(h->nx, h->ny, h->lx, h->ly);
    long long held = nshells < all ? nshells : all;
    if (held * 2 * (long long)sizeof(double) > SP_SMEM_MAX) held = 0;     // too many shells: straight to global memory
    p.nsm = (int)held;
    p.square = h->lx == h->ly;
    const double L = h->lx > h->ly ? (double)h->lx : (double)h->ly;
    p.rx = L / (double)h->lx; p.ry = L / (double)h->ly;
    const int G = (int)((p.Q + 31) / 32), S = (p.W + SP_WALK - 1) / SP_WALK;
    const unsigned grid = (unsigned)(((G + SP_BOX_Q - 1) / SP_BOX_Q) * ((S + SP_BOX_W - 1) / SP_BOX_W));
    const int smem = (int)(2 * sizeof(double) * p.nsm);
    int e;
    if (nshells == 0) e = launch_variant<false, 1>(p, grid, 0, h->stream);
    else if (p.T == 4) e = launch_variant<true, 4>(p, grid, smem, h->stream);
    else if (p.T == 2) e = launch_variant<true, 2>(p, grid, smem, h->stream);
    else e = launch_variant<true, 1>(p, grid, smem, h->stream);
    if (e) return e;
    h->launches++;
    return 0;
}

int energy_spectrum_scratch(xfb_handle h)
{
    if (!h->espec && dev_alloc((void **)&h->espec, sizeof(double) * (3 + 2 * (size_t)XFB_SPECTRUM_MAX_SHELLS))) return XFB_E_CUDA;
    return 0;
}

// device sums (3 + 2 * nshells doubles) -> host, scaled to domain means (the 1 / (2 Np^2) of every term)
int energy_spectrum_finish(xfb_handle h, const double *d, int nshells, double *totals, double *e, double *z)
{
    std::vector<double> host(3 + 2 * (size_t)nshells);
    CK(cudaMemcpyAsync(host.data(), d, sizeof(double) * host.size(), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    const double np = (double)h->nx * (double)h->ny, scale = 1.0 / (2.0 * np * np);
    for (int k = 0; k < 3; ++k) totals[k] = host[k] * scale;
    for (int s = 0; s < nshells; ++s) {
        e[s] = host[3 + s] * scale;
        z[s] = host[3 + nshells + s] * scale;
    }
    return 0;
}

}  // namespace xfb

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
#include <cstring>

#include "xfb_handle.h"

namespace xfb {

constexpr int SP_THREADS = 512;
constexpr int SP_WALK = 32;          // walk steps of one warp task
constexpr int SP_BOX_Q = 16;         // warp tasks per CTA box along q ...
constexpr int SP_BOX_W = 8;          // ... and along w
constexpr unsigned SP_NONE = 0xffffffffu;
constexpr unsigned SP_FULL = 0xffffffffu;

struct SpecParams {
    const cpx *z;                    // member's state array
    const double *kx2, *ky2;         // squared float32 wavenumbers (ky2 indexed by the global column)
    double *out;                     // [NT + NV * nshells]: raw totals, then the NV shell spectra
    long long Q;                     // elements per walk step
    int W;                           // walk steps
    int T;                           // tile width (tile-major) or 0 (row-major)
    int tshift;                      // log2(T)
    int nx, ny, hy, col0;
    int nshells, nsm;                // shells wanted, of which the first nsm are held in shared memory
    int square;                      // lx == ly: integer shell rule
    double rx, ry;                   // L / lx, L / ly (float64 rule)
};

struct BudgetParams : SpecParams {
    const cpx *n, *s;                // the nonlinear tendency and the source (s may be null), in z's layout
    double mask_kd;                  // dealiasing mask radius^2 (as the handle holds it)
    double nu, mu, ch, inv_kc2;      // dissipation coefficients as the handle holds them
    int order;
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

// What one mode contributes.  A run kind R names NV values carried along a run and binned per shell, NT totals, the
// loads in flight per lane (UNROLL), what one mode loads (R::In) and `mode`, which adds the mode's totals and returns its run
// values and whether it belongs to a shell at all.
//
// Energy spectrum: runs (e, z), totals (E, Z, P); one array.
struct EnergyRun {
    typedef SpecParams Params;
    static constexpr int NV = 2, NT = 3, UNROLL = 8;
    struct In { cpx z; };
    static __device__ __forceinline__ In load(const SpecParams &p, size_t at) { return In{__ldg(p.z + at)}; }
    static __device__ __forceinline__ In none() { return In{mk(0.f, 0.f)}; }
    static __device__ __forceinline__ bool mode(const SpecParams &p, const In &v, int ii, int j, double (&r)[NV],
                                                double (&t)[NT])
    {
        const double z2 = (double)v.z.x * (double)v.z.x + (double)v.z.y * (double)v.z.y;
        const double zw = (j == 0 || 2 * j == p.ny) ? z2 : 2.0 * z2;
        const double k2 = __ldg(p.kx2 + ii) + __ldg(p.ky2 + j);
        r[0] = k2 > 0.0 ? zw / k2 : 0.0;
        r[1] = zw;
        t[0] += r[0]; t[1] += r[1]; t[2] += zw * k2;
        return true;
    }
};

// Spectral budget: runs and totals (T_E, F_E, D_E, T_Z, F_Z, D_Z) of the modes inside the dealiasing mask; three arrays
// (two without a source).  Per mode the Z rates are w_j Re(conj(Z) X) with X = N, S and d(k^2) Z, the E rates those over
// k^2 ((0,0) excluded).  The beta term is i beta kx / k^2 Z: Re(conj(Z) X) = 0, no term of the budget.
struct BudgetRun {
    typedef BudgetParams Params;
    static constexpr int NV = 6, NT = 6, UNROLL = 4;
    struct In { cpx z, n, s; };
    static __device__ __forceinline__ In load(const BudgetParams &p, size_t at)
    {
        return In{__ldg(p.z + at), __ldg(p.n + at), p.s ? __ldg(p.s + at) : mk(0.f, 0.f)};
    }
    static __device__ __forceinline__ In none() { return In{mk(0.f, 0.f), mk(0.f, 0.f), mk(0.f, 0.f)}; }
    static __device__ __forceinline__ bool mode(const BudgetParams &p, const In &v, int ii, int j, double (&r)[NV],
                                                double (&t)[NT])
    {
        const int ip = ii <= p.nx - ii ? ii : p.nx - ii;
        if ((double)((long long)ip * ip + (long long)j * j) >= p.mask_kd) return false;    // outside the mask: no rate
        const double w = (j == 0 || 2 * j == p.ny) ? 1.0 : 2.0;
        const double zx = v.z.x, zy = v.z.y;
        const double k2 = __ldg(p.kx2 + ii) + __ldg(p.ky2 + j);
        double hv = k2 * p.inv_kc2, x = hv;
        for (int o = 1; o < p.order; ++o) hv *= x;
        const double d = -p.nu * k2 - p.mu - p.ch * hv;
        r[3] = w * (zx * (double)v.n.x + zy * (double)v.n.y);
        r[4] = w * (zx * (double)v.s.x + zy * (double)v.s.y);
        r[5] = w * d * (zx * zx + zy * zy);
        const double ik = k2 > 0.0 ? 1.0 / k2 : 0.0;
#pragma unroll
        for (int q = 0; q < 3; ++q) r[q] = r[3 + q] * ik;
#pragma unroll
        for (int q = 0; q < 6; ++q) t[q] += r[q];
        return true;
    }
};

// runs (key, v[NV]) handed on by the lanes of one warp: a segmented inclusive scan over the lanes of one column (lane
// stride ts) leaves each run's sum in its last lane, which adds it to the histogram
template <class R, int TS>
__device__ __forceinline__ void warp_flush(const SpecParams &p, double *sh, unsigned key, const double (&run)[R::NV], int lane)
{
    double v[R::NV];           // the scan works on a copy: the caller's run goes on unless it ends here
#pragma unroll
    for (int q = 0; q < R::NV; ++q) v[q] = run[q];
    const unsigned prev = __shfl_up_sync(SP_FULL, key, TS);
    const bool head = lane < TS || prev != key;
    const unsigned H = __ballot_sync(SP_FULL, head);
    constexpr unsigned seq = TS == 1 ? 0xffffffffu : (TS == 2 ? 0x55555555u : 0x11111111u);
    const unsigned below = lane == 31 ? 0xffffffffu : ((2u << lane) - 1u);
    const int hl = 31 - __clz(H & (seq << (lane % TS)) & below);
#pragma unroll
    for (int d = TS; d < 32; d <<= 1) {
        double x[R::NV];
#pragma unroll
        for (int q = 0; q < R::NV; ++q) x[q] = __shfl_up_sync(SP_FULL, v[q], d);
        if (lane - d >= hl) {
#pragma unroll
            for (int q = 0; q < R::NV; ++q) v[q] += x[q];
        }
    }
    const bool tail = lane + TS >= 32 || ((H >> (lane + TS)) & 1u);
    if (tail && key != SP_NONE) {
        if ((int)key < p.nsm) {
#pragma unroll
            for (int q = 0; q < R::NV; ++q) atomicAdd(&sh[q * p.nsm + key], v[q]);
        } else {
#pragma unroll
            for (int q = 0; q < R::NV; ++q) atomicAdd(&p.out[R::NT + q * p.nshells + key], v[q]);
        }
    }
}

// The walk, run hand-off, warp scan, shared-memory histogram and flush shared by every run kind
template <class R, bool SHELLS, int TS>
__device__ __forceinline__ void shell_reduce(const typename R::Params &p)
{
    extern __shared__ double sp_hist[];          // [NV * nsm]: the shells held here, one spectrum after the other
    __shared__ double sp_tot[SP_THREADS / 32][R::NT];
    constexpr int NV = R::NV, NT = R::NT, UN = R::UNROLL;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (SHELLS) {
        for (int k = threadIdx.x; k < NV * p.nsm; k += SP_THREADS) sp_hist[k] = 0.0;
        __syncthreads();
    }
    const int G = (int)((p.Q + 31) / 32), S = (p.W + SP_WALK - 1) / SP_WALK;
    const int boxes_q = (G + SP_BOX_Q - 1) / SP_BOX_Q;
    const int bq = blockIdx.x % boxes_q, bw = blockIdx.x / boxes_q;
    double tot[NT];
#pragma unroll
    for (int q = 0; q < NT; ++q) tot[q] = 0.0;
    for (int task = warp; task < SP_BOX_Q * SP_BOX_W; task += SP_THREADS / 32) {
        const int g = bq * SP_BOX_Q + task % SP_BOX_Q, s = bw * SP_BOX_W + task / SP_BOX_Q;
        if (g >= G || s >= S) continue;                  // warp-uniform
        const long long q = (long long)g * 32 + lane;
        int i, jin;                                       // row; column within the tile (tile-major) or column (row-major)
        if (p.T) { i = (int)(q >> p.tshift); jin = (int)(q & (p.T - 1)); }
        else { i = 0; jin = (int)q; }
        const bool qok = q < p.Q;
        unsigned cur = SP_NONE;
        double acc[NV];
#pragma unroll
        for (int k = 0; k < NV; ++k) acc[k] = 0.0;
        const int w0 = s * SP_WALK;
        for (int k0 = 0; k0 < SP_WALK; k0 += UN) {
            typename R::In v[UN];
            bool ok[UN];
#pragma unroll
            for (int u = 0; u < UN; ++u) {
                const int w = w0 + k0 + u;
                const int j = p.T ? p.col0 + w * p.T + jin : jin;
                ok[u] = qok && w < p.W && j < p.hy;
                v[u] = ok[u] ? R::load(p, (size_t)w * p.Q + q) : R::none();
            }
#pragma unroll
            for (int u = 0; u < UN; ++u) {
                const int w = w0 + k0 + u;
                const int ii = p.T ? i : w, j = p.T ? p.col0 + w * p.T + jin : jin;
                double r[NV];
#pragma unroll
                for (int k = 0; k < NV; ++k) r[k] = 0.0;
                unsigned key = SP_NONE;
                if (ok[u] && R::mode(p, v[u], ii, j, r, tot)) {
                    if (SHELLS) {
                        const int ip = ii <= p.nx - ii ? ii : p.nx - ii;
                        const unsigned sh = shell_of(p, ip, j);
                        key = sh < (unsigned)p.nshells ? sh : SP_NONE;       // beyond the shells asked for: totals only
                    }
                }
                if (SHELLS) {
                    const bool starts = key != SP_NONE && key != cur;
                    const unsigned fkey = starts ? cur : SP_NONE;
                    if (__ballot_sync(SP_FULL, fkey != SP_NONE)) warp_flush<R, TS>(p, sp_hist, fkey, acc, lane);
                    if (starts) {
                        cur = key;
#pragma unroll
                        for (int k = 0; k < NV; ++k) acc[k] = r[k];
                    } else if (key != SP_NONE) {
#pragma unroll
                        for (int k = 0; k < NV; ++k) acc[k] += r[k];
                    }
                }
            }
        }
        if (SHELLS && __ballot_sync(SP_FULL, cur != SP_NONE)) warp_flush<R, TS>(p, sp_hist, cur, acc, lane);
    }
    // totals: warp shuffles, then one atomic per CTA and quantity
#pragma unroll
    for (int o = 16; o; o >>= 1) {
#pragma unroll
        for (int k = 0; k < NT; ++k) tot[k] += __shfl_xor_sync(SP_FULL, tot[k], o);
    }
    if (lane == 0) {
#pragma unroll
        for (int k = 0; k < NT; ++k) sp_tot[warp][k] = tot[k];
    }
    __syncthreads();
    if (threadIdx.x < NT) {
        double t = 0.0;
        for (int w = 0; w < SP_THREADS / 32; ++w) t += sp_tot[w][threadIdx.x];
        atomicAdd(&p.out[threadIdx.x], t);
    }
    if (SHELLS) {
        for (int k = threadIdx.x; k < p.nsm; k += SP_THREADS) {
#pragma unroll
            for (int q = 0; q < NV; ++q)
                if (sp_hist[q * p.nsm + k] != 0.0) atomicAdd(&p.out[NT + q * p.nshells + k], sp_hist[q * p.nsm + k]);
        }
    }
}

template <bool SHELLS, int TS>
__global__ void __launch_bounds__(SP_THREADS) energy_spectrum_kernel(const SpecParams p)
{
    shell_reduce<EnergyRun, SHELLS, TS>(p);
}

template <bool SHELLS, int TS>
__global__ void __launch_bounds__(SP_THREADS) spectral_budget_kernel(const BudgetParams p)
{
    shell_reduce<BudgetRun, SHELLS, TS>(p);
}

constexpr int SP_SMEM_MAX = 200 * 1024;          // histogram bytes per CTA (the rest of the 227 KB stays free)

template <class R, bool SHELLS, int TS>
struct KernelOf;
template <bool SHELLS, int TS>
struct KernelOf<EnergyRun, SHELLS, TS> {
    static constexpr auto k = energy_spectrum_kernel<SHELLS, TS>;
    static constexpr const char *name = "energy_spectrum_kernel";
};
template <bool SHELLS, int TS>
struct KernelOf<BudgetRun, SHELLS, TS> {
    static constexpr auto k = spectral_budget_kernel<SHELLS, TS>;
    static constexpr const char *name = "spectral_budget_kernel";
};

template <class R, bool SHELLS, int TS>
static int launch_variant(const typename R::Params &p, unsigned grid, int smem, cudaStream_t st)
{
    typedef KernelOf<R, SHELLS, TS> K;
    const char *name = K::name;
    static PerDeviceInt configured;
    int err = 0;
    if (SHELLS && configured.get([](int *e) -> int {
            cudaError_t r = cudaFuncSetAttribute(K::k, cudaFuncAttributeMaxDynamicSharedMemorySize, SP_SMEM_MAX);
            if (r != cudaSuccess) { *e = (int)r; return 0; }
            return 1;
        }, &err) <= 0)
        return fail(XFB_E_CUDA, "%s: %s", name, cudaGetErrorString((cudaError_t)err));
    K::k<<<grid, SP_THREADS, smem, st>>>(p);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(XFB_E_CUDA, "%s: %s", name, cudaGetErrorString(e));
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

// the walk over this rank's state layout, the shells and the grid; nsm is left to the caller
static unsigned fill_spec(xfb_handle h, int nshells, double *d_out, SpecParams &p, long long *all)
{
    p.kx2 = h->kx2; p.ky2 = h->ky2; p.out = d_out;
    p.T = h->tw_state;
    p.tshift = p.T == 4 ? 2 : (p.T == 2 ? 1 : 0);
    if (p.T) { p.Q = (long long)h->nx * p.T; p.W = h->pitch / p.T * h->nchunks; }
    else { p.Q = h->pitch; p.W = h->nx; }
    p.nx = h->nx; p.ny = h->ny; p.hy = h->hy; p.col0 = h->col0;
    p.nshells = nshells;
    *all = shells_all(h->nx, h->ny, h->lx, h->ly);
    p.square = h->lx == h->ly;
    const double L = h->lx > h->ly ? (double)h->lx : (double)h->ly;
    p.rx = L / (double)h->lx; p.ry = L / (double)h->ly;
    const int G = (int)((p.Q + 31) / 32), S = (p.W + SP_WALK - 1) / SP_WALK;
    return (unsigned)(((G + SP_BOX_Q - 1) / SP_BOX_Q) * ((S + SP_BOX_W - 1) / SP_BOX_W));
}

template <class R>
static int launch_shells(xfb_handle h, const typename R::Params &p, unsigned grid)
{
    const int smem = (int)(R::NV * sizeof(double) * p.nsm);
    int e;
    if (p.nshells == 0) e = launch_variant<R, false, 1>(p, grid, 0, h->stream);
    else if (p.T == 4) e = launch_variant<R, true, 4>(p, grid, smem, h->stream);
    else if (p.T == 2) e = launch_variant<R, true, 2>(p, grid, smem, h->stream);
    else e = launch_variant<R, true, 1>(p, grid, smem, h->stream);
    if (e) return e;
    h->launches++;
    return 0;
}

int launch_energy_spectrum(xfb_handle h, const cpx *state, int nshells, double *d_out)
{
    SpecParams p;
    long long all;
    const unsigned grid = fill_spec(h, nshells, d_out, p, &all);
    p.z = state;
    long long held = nshells < all ? nshells : all;
    if (held * 2 * (long long)sizeof(double) > SP_SMEM_MAX) held = 0;     // too many shells: straight to global memory
    p.nsm = (int)held;
    return launch_shells<EnergyRun>(h, p, grid);
}

int launch_spectral_budget(xfb_handle h, const cpx *state, const cpx *tend, const cpx *src, int nshells, double *d_out)
{
    BudgetParams p;
    memset(&p, 0, sizeof(p));
    long long all;
    const unsigned grid = fill_spec(h, nshells, d_out, p, &all);
    p.z = state; p.n = tend; p.s = src;
    // as many of the first shells as fit are held in shared memory, the rest go to global memory
    long long held = nshells < all ? nshells : all;
    const long long fit = SP_SMEM_MAX / (BudgetRun::NV * (long long)sizeof(double));
    p.nsm = (int)(held < fit ? held : fit);
    p.mask_kd = h->mask_kd;
    p.nu = (double)h->nu; p.mu = (double)h->lin.mu; p.ch = (double)h->lin.ch; p.inv_kc2 = (double)h->lin.inv_kc2;
    p.order = h->lin.on ? h->lin.order : 1;
    return launch_shells<BudgetRun>(h, p, grid);
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

int spectral_budget_scratch(xfb_handle h)
{
    if (!h->bspec && dev_alloc((void **)&h->bspec, sizeof(double) * XFB_BUDGET_N * (1 + (size_t)XFB_SPECTRUM_MAX_SHELLS)))
        return XFB_E_CUDA;
    return 0;
}

// device sums (6 + 6 * nshells doubles) -> host, scaled to rates of domain means (1 / Np^2)
int spectral_budget_finish(xfb_handle h, const double *d, int nshells, double *totals, double *budget)
{
    std::vector<double> host(XFB_BUDGET_N * (1 + (size_t)nshells));
    CK(cudaMemcpyAsync(host.data(), d, sizeof(double) * host.size(), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    const double np = (double)h->nx * (double)h->ny, scale = 1.0 / (np * np);
    for (int k = 0; k < XFB_BUDGET_N; ++k) totals[k] = host[k] * scale;
    for (size_t k = 0; k < (size_t)XFB_BUDGET_N * nshells; ++k) budget[k] = host[XFB_BUDGET_N + k] * scale;
    return 0;
}

}  // namespace xfb

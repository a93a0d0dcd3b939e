// xfb_col.cuh -- K-COL: transforms along x (the strided direction) on tiles of W adjacent
// spectral columns, with every pointwise spectral operator of the reference fused around them.
// This header holds the parameter block and the column transform shared by every K-COL kernel, and col_kernel, the
// plain forward and inverse column transforms of the operator tier (COL_FWD / COL_INV).
//
// One launch of COL_STEP (colt_kernel, xfb_colt.cuh; col2l_kernel, xfb_col2l.cuh) replaces, for its column tile
// (file:line in /root/reference/src):
//   first-dimension half of the r2c of the tendency                  main.cpp:237
//   fop.laplacian + `dvortdt_c += lvort_c * NU`                      main.cpp:148,240-243 ; fftwfop.cpp:105-110
//   fop.dealiase -> rk_k                                             main.cpp:296-306     ; fftwfop.cpp:119-124
//   evolve() / final RK4 combine                                     main.cpp:246-251,309-312
//   memcpy(vort_c0 <- vort_c)                                        main.cpp:286 (eliminated)
//   fop.gradx, fop.grady, fop.invertLaplacian of the NEXT stage      main.cpp:151,165,179,198,212 ; fftwfop.cpp:87-117
//   first-dimension half of the four c2r                             main.cpp:154,168,200,214
// The wavenumber/Laplacian/mask tables of fftwfop.cpp:5-79 are never materialised as H-sized
// arrays: kx[NX], ky[pitch] and their float64 squares are tiny tables, the mask is integer math.
#pragma once
#include "xfb_fft.cuh"

namespace xfb {

// COL_TSTEP / COL_TPRO: COL_STEP / COL_PRO of the passive tracer (xfb_set_tracer): same forward transform, RK epilogue
// (diffusivity in p.nu) and state update, but only the two gradient products i kx C, i ky C leave for K-ROW.
enum { COL_FWD = 0, COL_INV = 1, COL_STEP = 2, COL_PRO = 3, COL_DIAG = 4, COL_FWDT = 5, COL_TSTEP = 6, COL_TPRO = 7 };

// Linear terms of the vorticity equation (xfb_set_linear_terms, DESIGN.md section 3): beta-plane, linear drag and
// hyperviscosity.  Per mode L(k) = -mu - ch (k^2 / k_c^2)^order + i beta kx / k^2 multiplies the stage state inside the
// dealiasing mask; only the LIN instances of the stepper's K-COL and gen_stage read these fields.
struct LinCoef {
    float beta, mu;
    float ch;             // nu_h * k_c^(2 order), formed in float64 on the host (k_c^2 = kx(nx/2)^2 + ky(ny/2)^2)
    float inv_kc2;        // 1 / k_c^2: (k^2 / k_c^2) <= 1 on the grid, so no power of it overflows
    int order;            // 1..8
    int on;               // non-zero: some term is non-zero and the stepper runs the LIN instances
};

// L(k) z for one mode: kx the signed x wavenumber, k2 = kx^2 + ky^2 (0 only at (0,0), where kx = 0 and the beta term
// vanishes through the fmaxf guard)
__device__ __forceinline__ cpx lin_term(const LinCoef &L, const float kx, const float k2, const cpx z)
{
    const float b = __fdividef(L.beta * kx, fmaxf(k2, 1.17549435e-38f));
    // (k^2 / k_c^2)^order as a uniform loop: the fewest live registers of the forms tried (binary powering with selects or
    // predicated multiplies spilled more in the 8192 K-COL)
    const float x = k2 * L.inv_kc2;
    float xp = x;
#pragma unroll 1
    for (int o = 1; o < L.order; ++o) xp *= x;
    const float a = fmaf(-L.ch, xp, -L.mu);
    return mk(a * z.x - b * z.y, a * z.y + b * z.x);
}

struct ColParams {
    const cpx *jint;      // FWD/STEP: y-transformed lines, pair layout (see xfb_row.cuh): (i, j) at ((i>>1)*pitch + j)*2 + (i&1)
    cpx *z0;              // spectral state at the start of the step (FWD writes it)
    cpx *zk;              // stage state
    cpx *acc;             // running RK4 sum r1 + 2 r2 + 2 r3
    cpx *t_out[4];        // x-inverse-transformed i kx Z, i ky Z, i ky Psi, i kx Psi ; INV: [0]   (pair layout)
    const cpx *inv_in;    // INV: spectrum to transform
    const cpx *tw;
    int twn;
    const float *kx;      // [NX]    gradx_coe
    const float *ky;      // [pitch] grady_coe (pad columns continue the formula)
    const double *kx2;    // [NX]    (double)kx*kx
    const double *ky2;    // [pitch]
    int pitch;
    int j_base;           // global index of this rank's first column (0 on one GPU): ky, mask and the (0,0) entry use it
    // layout of the K-COL-private state arrays z0/zk/acc: element (i, j0 + c) of column tile b lives at
    //   member_offset + b * st_tile_stride + i * st_row_stride + c
    // row-major (operator tier):  st_tile_stride = W,      st_row_stride = pitch
    // tile-major (stepper):       st_tile_stride = NX * W, st_row_stride = W   (a tile is one contiguous block)
    long long st_tile_stride;
    int st_row_stride;
    long long member_stride;   // complex elements between ensemble members
    int ny;               // for the mask reflection nothing is needed in y; kept for clarity
    double mask_kd;       // generalized_wavenumber_square (fftwfop.cpp:57), as stored in float
    int mask_kd_i;        // the same as an integer (exact for every supported size)
    float kxscale;        // TWOPI / Lx: fused path forms kx = (signed index) * kxscale in registers
    float nu;
    float dt;             // full step
    float dt_stage;       // dt/2, dt/2, dt for stages 1..3
    int stage;            // 1..4 ; COL_DIAG: product set (0 strain, 1 tracer, 2 + field id: one record field)
    int nfields;          // COL_DIAG: number of products (3 or 1)
    // slab-decomposed runs, two-level kernel (xfb_col2l.cuh): the 16-byte pieces [self_piece0, self_piece0 + self_pieces) of a
    // column -- the row pairs this rank owns itself -- go straight into this rank's own receive arrays (self_out[f] points
    // at the block of this launch's chunk), so the exchange has no self-copy to do; self_pieces == 0: everything to t_out
    int self_piece0, self_pieces;
    cpx *self_out[4];
    LinCoef lin;          // COL_STEP: the linear terms (lin.on selects the LIN instances)
};

template <int NX, int W>
struct ColCfg {
    static constexpr int G = NX / 16;
    static constexpr int VT = G * W;                          // butterfly threads per tile
    static constexpr int THREADS = (VT > 512) ? 512 : VT;
    static constexpr int NIT = VT / THREADS;                  // butterflies per thread per pass
    static constexpr int SMEM = LinePlan<NX>::PADDED * W * (int)sizeof(cpx);
    static constexpr int MINB = (THREADS <= 128) ? 4 : (THREADS <= 256) ? 2 : 1;
    static_assert(THREADS >= 16 && NIT <= 2, "bad column tile");
};

// element (i, j) of a pair-layout array (rows 2m, 2m+1 interleaved): ((i >> 1) * pitch + j) * 2 + (i & 1).
// Rows i = t + k*G of one butterfly thread (G even) are k * G * pitch elements apart, as in a row-major array.
__device__ __forceinline__ size_t pair_base(const int t, const int j, const int pitch)
{
    return ((size_t)(t >> 1) * (size_t)pitch + (size_t)j) * 2 + (size_t)(t & 1);
}


// -(kx^2 + ky^2) narrowed to float, summed in float64 like pow(float,2)+pow(float,2) (fftwfop.cpp:42-45)
__device__ __forceinline__ float lap_coe(const double kx2, const double ky2) { return (float)(-(kx2 + ky2)); }

// signed x wavenumber index of row i = slot_pos(t, k) (k compile-time): i for i <= NX/2 (Nyquist keeps +), else i - NX.
// In both slot orders the slots k < 8 hold rows below NX/2, k > 8 rows above, and k = 8 row NX/2 exactly when the base is 0.
template <int NX, bool SPLIT = false>
__device__ __forceinline__ int signed_row(const int t, const int k)
{
    const int i = slot_pos<NX, SPLIT>(t, k);
    if (k < 8) return i;
    if (k == 8) return (slot_base<NX, SPLIT>(t) == 0) ? i : i - NX;
    return i - NX;
}

// hook(e, last): called by every thread after exchange e (0-based) has been read and its closing barrier passed --
// a CTA-uniform point between two barriers where the caller can slip in unrelated pipelined work.
// pre(): called by every thread right before the shared-memory writes of the LAST exchange: global loads issued there
// (the first operands of the caller's epilogue) complete under the exchange's two barriers and the final pass.
template <int NX, int W, int NIT, class Hook, class Pre>
__device__ __forceinline__ void col_fft(cpx (&v)[NIT][16], cpx *sm, const int (&t)[NIT], const int (&c)[NIT],
                                        const LineTw<NX> (&tw)[NIT], const bool drain_tma, Hook &hook, Pre &pre)
{
    typedef LinePlan<NX> P;
    // drain_tma (uniform over the CTA): the caller is going to overwrite a buffer that bulk stores may still be reading.
    // Thread 0 waits for them as late as possible -- before the first barrier of the LAST exchange --, so the stores
    // drain under the earlier passes and every thread that leaves the transform knows the buffer is free.
    constexpr int LAST_EX = (P::NPASS > P::N16) ? P::N16 - 1 : P::N16 - 2;
    if (LAST_EX < 0 && drain_tma && threadIdx.x == 0) tma_wait_read_all();
    if (LAST_EX < 0) pre();
    int ns = 1;
#pragma unroll
    for (int p = 0; p < P::N16; ++p) {
#pragma unroll
        for (int it = 0; it < NIT; ++it) pass16_compute<NX>(v[it], p, tw[it]);
        if (p != P::NPASS - 1) {
            if (p == LAST_EX) pre();
#pragma unroll
            for (int it = 0; it < NIT; ++it) exchange_write<W>(v[it], sm, t[it], c[it], ns);
            if (p == LAST_EX && drain_tma && threadIdx.x == 0) tma_wait_read_all();
            __syncthreads();
#pragma unroll
            for (int it = 0; it < NIT; ++it) exchange_read<P::G, W>(v[it], sm, t[it], c[it]);
            __syncthreads();
            hook(p, p == LAST_EX);
        }
        ns *= 16;
    }
#pragma unroll
    for (int it = 0; it < NIT; ++it) rem_pass<NX>(v[it], tw[it]);
}

template <int NX, int W, int NIT, class Hook>
__device__ __forceinline__ void col_fft(cpx (&v)[NIT][16], cpx *sm, const int (&t)[NIT], const int (&c)[NIT],
                                        const LineTw<NX> (&tw)[NIT], const bool drain_tma, Hook &hook)
{
    ColFftNoPre nopre;
    col_fft<NX, W, NIT, Hook, ColFftNoPre>(v, sm, t, c, tw, drain_tma, hook, nopre);
}

template <int NX, int W, int NIT>
__device__ __forceinline__ void col_fft(cpx (&v)[NIT][16], cpx *sm, const int (&t)[NIT], const int (&c)[NIT],
                                        const LineTw<NX> (&tw)[NIT], const bool drain_tma = false)
{
    ColFftNoHook nohook;
    col_fft<NX, W, NIT, ColFftNoHook>(v, sm, t, c, tw, drain_tma, nohook);
}

template <int NX, int W, int MODE>
__global__ void __launch_bounds__(ColCfg<NX, W>::THREADS, ColCfg<NX, W>::MINB)
col_kernel(const ColParams p)
{
    static_assert(MODE == COL_FWD || MODE == COL_INV, "col_kernel has the plain transforms only");
    typedef ColCfg<NX, W> C;
    constexpr int G = C::G, NIT = C::NIT;
    // the same symbol as col2l_kernel's staging buffer, which TMA needs 128-byte aligned: declarations that disagree
    // within one translation unit leave the alignment to the order in which the kernels are instantiated
    extern __shared__ __align__(128) unsigned char smem_raw[];
    cpx *sm = reinterpret_cast<cpx *>(smem_raw);

    const int j0 = blockIdx.x * W;
    const size_t moff = (size_t)blockIdx.y * (size_t)p.member_stride;
    const size_t soff = moff + (size_t)blockIdx.x * (size_t)p.st_tile_stride;   // state arrays: this tile
    const size_t srow = (size_t)p.st_row_stride;

    int t[NIT], c[NIT];
    LineTw<NX> tw[NIT];
#pragma unroll
    for (int it = 0; it < NIT; ++it) {
        const int vt = it * C::THREADS + threadIdx.x;
        c[it] = vt % W;
        t[it] = vt / W;
        tw[it].init(p.tw, p.twn, t[it]);
    }

    cpx v[NIT][16];
    if (MODE == COL_FWD) {
#pragma unroll
        for (int it = 0; it < NIT; ++it) {
            const cpx *src = p.jint + moff + pair_base(t[it], j0 + c[it], p.pitch);
#pragma unroll
            for (int k = 0; k < 16; ++k) v[it][k] = __ldg(src + (size_t)(k * G) * p.pitch);
        }
        col_fft<NX, W, NIT>(v, sm, t, c, tw);
#pragma unroll
        for (int it = 0; it < NIT; ++it) {
            const size_t e0 = soff + (size_t)t[it] * srow + c[it];
#pragma unroll
            for (int k = 0; k < 16; ++k) p.z0[e0 + (size_t)(k * G) * srow] = v[it][k];
        }
    } else {
#pragma unroll
        for (int it = 0; it < NIT; ++it) {
            const cpx *src = p.inv_in + moff + j0 + c[it];
#pragma unroll
            for (int k = 0; k < 16; ++k) v[it][k] = cswap(__ldg(src + (size_t)(t[it] + k * G) * p.pitch));
        }
        col_fft<NX, W, NIT>(v, sm, t, c, tw);
        cpx *out = p.t_out[0] + moff;
#pragma unroll
        for (int it = 0; it < NIT; ++it) {
#pragma unroll
            for (int k = 0; k < 16; ++k) *(out + pair_base(t[it], j0 + c[it], p.pitch) + (size_t)(k * G) * p.pitch) = cswap(v[it][k]);
        }
    }
}

}  // namespace xfb

// xfb_rowpair.cuh -- K-ROW for NY <= 8192: the two rows of a pair (2m, 2m+1) are transformed TOGETHER as one
// complex line of NY points ("two real transforms for one complex"):
//
//   c2r : Z[k] = A[k] + i B[k]            (k <= NY/2,  A, B the half spectra of the two rows)
//         Z[NY-k] = conj(A[k]) + i conj(B[k])
//         z = inverse complex DFT of Z    ->  z[n] = a[n] + i b[n]        (a, b the two real rows)
//   r2c : z = a + i b, Z = DFT(z),  A[k] = (Z[k] + conj Z[NY-k]) / 2,  B[k] = (Z[k] - conj Z[NY-k]) / (2i)
//
// In the pair layout (xfb_row.cuh) A[k] and B[k] are adjacent, so every global access of this kernel is a
// fully used 16-byte vector; there is no split/merge twiddle step at all.  Same reference loops as
// xfb_row.cuh: main.cpp:126-135,154,168,200-201,214,225-227,237 and fftwf_backward_normalize (:37-41).
// The imaginary parts of the DC and Nyquist bins are ignored like FFTW's c2r does.
#pragma once
#include "xfb_row.cuh"

namespace xfb {

template <int NY>
struct PairCfg {
    static constexpr int G = NY / 16;                          // threads per row pair
    static constexpr int THREADS = (G >= 128) ? G : 128;
    static constexpr int PPC = THREADS / G;                    // row pairs per CTA
    static constexpr int SMEM = PPC * LinePlan<NY>::PADDED * (int)sizeof(cpx);
    // JAC parks -u (then -u * dvortdx) and v (then v * dvortdy) of both rows between the transforms
    static constexpr int SMEM_JAC = SMEM + 2 * PPC * NY * (int)sizeof(cpx);
    static constexpr int MINB = (THREADS >= 512) ? 1 : (THREADS >= 256) ? 2 : 4;
};

// half spectra of a row pair -> on return v[q] = (b[n], a[n]) unscaled (swapped), n = t + q*G
template <int NY, bool DIST, typename Bar>
__device__ __forceinline__ void c2r_pair(cpx (&v)[16], const cpx *PB, const RowParams &p, cpx *sm, const int t,
                                         const LineTw<NY> &tw, const Bar &bar)
{
    constexpr int G = NY / 16;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        float4 ld[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const int n = t + (8 * h + e) * G;
            const int m = (h == 0) ? n : NY - n;               // h = 1: n >= NY/2, mirrored bin 1 .. NY/2
            ld[e] = *reinterpret_cast<const float4 *>(PB + line_pos<DIST>(p, m));
        }
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            float4 x = ld[e];                                  // (A.re, A.im, B.re, B.im)
            const int n = t + (8 * h + e) * G;
            if ((h == 0 && e == 0 && n == 0) || (h == 1 && e == 0 && n == NY / 2)) { x.y = 0.f; x.w = 0.f; }
            // swapped for the inverse transform: v = (Im Z, Re Z)
            v[8 * h + e] = (h == 0) ? mk(x.y + x.z, x.x - x.w) : mk(x.z - x.y, x.x + x.w);
        }
    }
    line_fft<NY, 1>(v, sm, t, 0, tw, bar);
}

// Same transform, the pair region (2 * pitch complex values, dense) already staged in this pair's FFT buffer by a
// TMA bulk copy.  The buffer is read (two conflict-free LDS.128 streams), then reused for the exchanges; with RELEASE
// it is handed back to the async proxy after the last exchange so the next field can be fetched during the tail.
template <int NY, typename Bar, bool RELEASE>
__device__ __forceinline__ void c2r_pair_staged(cpx (&v)[16], cpx *sm, const int t, const LineTw<NY> &tw, const Bar &bar)
{
    constexpr int G = NY / 16;
    const float4 *st = reinterpret_cast<const float4 *>(sm);
#pragma unroll
    for (int h = 0; h < 2; ++h) {
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const int n = t + (8 * h + e) * G;
            const int m = (h == 0) ? n : NY - n;
            float4 x = st[m];
            if ((h == 0 && e == 0 && n == 0) || (h == 1 && e == 0 && n == NY / 2)) { x.y = 0.f; x.w = 0.f; }
            v[8 * h + e] = (h == 0) ? mk(x.y + x.z, x.x - x.w) : mk(x.z - x.y, x.x + x.w);
        }
    }
    bar.sync();                                       // everyone has read the staged spectrum
    line_fft<NY, 1, Bar, RELEASE>(v, sm, t, 0, tw, bar);
}

// v[q] = (a[n], b[n]) -> half spectra of both rows written to the pair at PBout (+ zeroed pad columns)
// SPLIT (NY = 8192): v arrives in the Split8192 order and is transformed by fft8192_from_split, natural order out
template <int NY, bool DIST, typename Bar, bool RELEASE = false, bool SPLIT = false>
__device__ __forceinline__ void r2c_pair(cpx (&v)[16], cpx *__restrict__ PBout, const RowParams &p, const int pitch, cpx *sm,
                                         const int t, const LineTw<NY> &tw, const Bar &bar)
{
    constexpr int G = NY / 16;
    if constexpr (SPLIT) fft8192_from_split<1>(v, sm, t, 0, tw, bar);
    else line_fft<NY, 1>(v, sm, t, 0, tw, bar);
#pragma unroll
    for (int q = 0; q < 16; ++q) sm[padpos(t + q * G)] = v[q];
    bar.sync();
    cpx M8[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) M8[q] = sm[padpos((NY - (t + q * G)) & (NY - 1))];      // Z[NY - n]
    if (RELEASE) {                                              // the buffer goes back to the async proxy
        fence_proxy_async();
        bar.sync();
    }
#pragma unroll
    for (int q = 0; q < 8; ++q) {
        const int n = t + q * G;
        const cpx Z = v[q];
        const cpx M = M8[q];
        float4 o;
        o.x = 0.5f * (Z.x + M.x);                               // A = (Z + conj M) / 2
        o.y = 0.5f * (Z.y - M.y);
        o.z = 0.5f * (Z.y + M.y);                               // B = (Z - conj M) / (2i)
        o.w = 0.5f * (M.x - Z.x);
        *reinterpret_cast<float4 *>(out_addr<DIST>(p, PBout, n)) = o;
    }
    if (t == 0)                                                 // Nyquist bin: Z[NY/2] is its own mirror
        *reinterpret_cast<float4 *>(out_addr<DIST>(p, PBout, NY / 2)) = make_float4(v[8].x, 0.f, v[8].y, 0.f);
    for (int k = NY / 2 + 1 + t; k < pitch; k += G)
        *reinterpret_cast<float4 *>(out_addr<DIST>(p, PBout, k)) = make_float4(0.f, 0.f, 0.f, 0.f);
}

// forward transform in two halves so a bulk fetch can be issued between the transform and the stores:
// begin: Z = DFT(a + i b), on return v[q] = Z[n] for q < 8 and M[q] = Z[NY - n] packed into v[8 + q]; the shared
// buffer has been released to the async proxy.
template <int NY, typename Bar>
__device__ __forceinline__ void r2c_pair_begin(cpx (&v)[16], cpx *sm, const int t, const LineTw<NY> &tw, const Bar &bar)
{
    constexpr int G = NY / 16;
    line_fft<NY, 1>(v, sm, t, 0, tw, bar);
#pragma unroll
    for (int q = 0; q < 16; ++q) sm[padpos(t + q * G)] = v[q];
    bar.sync();
    const cpx nyq = v[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) v[8 + q] = sm[padpos((NY - (t + q * G)) & (NY - 1))];
    if (t == 0) v[8] = nyq;                                     // thread 0: Z[NY - 0] = Z[0] is not needed, keep Z[NY/2] there
    fence_proxy_async();
    bar.sync();
}

template <int NY, bool DIST>
__device__ __forceinline__ void r2c_pair_finish(const cpx (&v)[16], cpx *__restrict__ PBout, const RowParams &p, const int pitch,
                                                const int t)
{
    constexpr int G = NY / 16;
#pragma unroll
    for (int q = 0; q < 8; ++q) {
        const int n = t + q * G;
        const cpx Z = v[q];
        const cpx M = (q == 0 && t == 0) ? v[0] : v[8 + q];      // bin 0 mirrors itself
        float4 o;
        o.x = 0.5f * (Z.x + M.x);
        o.y = 0.5f * (Z.y - M.y);
        o.z = 0.5f * (Z.y + M.y);
        o.w = 0.5f * (M.x - Z.x);
        *reinterpret_cast<float4 *>(out_addr<DIST>(p, PBout, n)) = o;
    }
    if (t == 0) *reinterpret_cast<float4 *>(out_addr<DIST>(p, PBout, NY / 2)) = make_float4(v[8].x, 0.f, v[8].y, 0.f);
    for (int k = NY / 2 + 1 + t; k < pitch; k += G)
        *reinterpret_cast<float4 *>(out_addr<DIST>(p, PBout, k)) = make_float4(0.f, 0.f, 0.f, 0.f);
}

// JAC with plain vector loads (slab runs: a line is cut into panels, not one contiguous region)
template <int NY, bool DIST, typename Bar>
__device__ __forceinline__ void jac_pair_direct(const RowParams &p, unsigned char *smem_raw, cpx *sm, const int lane_pair, const int t,
                                                const size_t off, const size_t roff, const bool live, const LineTw<NY> &tw,
                                                const Bar &bar)
{
    typedef PairCfg<NY> C;
    constexpr int G = C::G;
    cpx v[16];
    cpx *park0 = reinterpret_cast<cpx *>(smem_raw) + (size_t)C::PPC * LinePlan<NY>::PADDED + (size_t)lane_pair * (2 * NY);
#pragma unroll 1
    for (int f = 0; f < 4; ++f) {
        const int src_field = (f == 0) ? 2 : (f == 1) ? 0 : (f == 2) ? 3 : 1;
        c2r_pair<NY, DIST>(v, p.spec_in[src_field] + off, p, sm, t, tw, bar);
        cpx *park = park0 + (f >> 1) * NY;
        if (f & 1) {
#pragma unroll
            for (int q = 0; q < 16; ++q) {
                const cpx a = park[q * G + t];
                park[q * G + t] = mk(a.x * (v[q].y * p.scale), a.y * (v[q].x * p.scale));
            }
        } else {
#pragma unroll
            for (int q = 0; q < 16; ++q) park[q * G + t] = mk(v[q].y * p.scale, v[q].x * p.scale);
        }
    }
    cpx J[16];
#pragma unroll
    for (int q = 0; q < 16; ++q) {
        const cpx j1 = park0[q * G + t], j2 = park0[NY + q * G + t];
        J[q] = mk(j1.x - j2.x, j1.y - j2.y);
    }
    if (p.real_in != nullptr) {
        const float *sa = p.real_in + roff, *sb = sa + NY;
#pragma unroll
        for (int q = 0; q < 16; ++q) J[q] = mk(J[q].x + __ldg(sa + t + q * G), J[q].y + __ldg(sb + t + q * G));
    }
    r2c_pair<NY, DIST>(J, p.spec_out + off, p, live ? p.pitch : 0, sm, t, tw, bar);
}

// ---- ROW_JAC with the parked products in TENSOR MEMORY and a double-buffered staging area -----------------------------
// The parked products are thread-private (a thread reads back exactly what it wrote), so they do not need shared
// memory at all: each thread keeps them in its own TMEM row (tcgen05.st / tcgen05.ld, 2 x 32 columns).  That takes
// 2 * NY * 8 bytes per pair out of shared memory (131 KB at NY = 8192) and a sixth of the traffic off the shared-memory
// pipe, and the freed space holds TWO staging buffers: the bulk fetch of field n+2 is issued as soon as field n has
// been read, a whole transform ahead, so no fetch latency is exposed any more.
// Default at NY >= 4096 (8192^2: 0.50 ms per launch against 0.58 with the shared-memory parks); below that several CTAs
// per SM already overlap fetch and transform and the shared-memory parks of rowpair_kernel stay faster -- see
// use_tmem_parks() in xfb_row.cu.
template <int NY>
struct PairTCfg {
    static constexpr int G = NY / 16;
    static constexpr int THREADS = (G >= 128) ? G : 128;
    static constexpr int PPC = THREADS / G;
    static constexpr int ST_ELEMS = 2 * (NY / 2 + 4);                     // complex elements of one pair region
    static constexpr int F_BYTES = PPC * LinePlan<NY>::PADDED * (int)sizeof(cpx);
    static constexpr int ST_BYTES = PPC * ST_ELEMS * (int)sizeof(cpx);    // one staging buffer, all pairs of the CTA
    static constexpr int SMEM = F_BYTES + 2 * ST_BYTES;
    static constexpr int WARPS = THREADS / 32;
    static constexpr int TCOLS = (WARPS > 8) ? 256 : (WARPS > 4) ? 128 : 64;     // 64 columns per group of four warps
    static constexpr int MINB = (THREADS >= 512) ? 1 : (THREADS >= 256) ? 2 : 4;
};

template <int NY>
__global__ void __launch_bounds__(PairTCfg<NY>::THREADS, PairTCfg<NY>::MINB)
rowpair_jac_tmem_kernel(const RowParams p)
{
    typedef PairTCfg<NY> C;
    constexpr int G = C::G;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ unsigned tmem_slot;
    __shared__ unsigned long long mbar_all[2 * C::PPC];
    const int lane_pair = threadIdx.x / G;
    const int t = threadIdx.x % G;
    cpx *sm = reinterpret_cast<cpx *>(smem_raw) + (size_t)lane_pair * LinePlan<NY>::PADDED;
    // staging buffer b of this pair slot: stage0 + b * (ST_BYTES / sizeof(cpx))
    cpx *const stage0 = reinterpret_cast<cpx *>(smem_raw + C::F_BYTES) + (size_t)lane_pair * C::ST_ELEMS;
    constexpr int ST_STRIDE = C::ST_BYTES / (int)sizeof(cpx);
    unsigned long long *mbar = &mbar_all[2 * lane_pair];
    const int npairs = p.nrows >> 1;

    // NY = 8192: the inverse transforms leave their products in the Split8192 order (two shared-memory exchanges instead of
    // three), the forward transform of J takes them from there
    constexpr bool SPLIT = (NY == 8192);
    LineTw<NY> tw;
    if constexpr (SPLIT) Split8192::init_tw(tw, p.tw, p.twn, t);
    else tw.init(p.tw, p.twn, t);
    typedef typename RowBarSel<(G >= 32 && C::PPC > 1)>::type Bar;
    const Bar bar = RowBarSel<(G >= 32 && C::PPC > 1)>::make(1 + lane_pair, G);

    if (t == 0) {
        mbar_init(&mbar[0], 1);
        mbar_init(&mbar[1], 1);
        mbar_fence_init();
    }
    const unsigned tbase = tmem_alloc_cta<C::TCOLS>(&tmem_slot);          // includes a CTA barrier
    const int warp = threadIdx.x >> 5;
    const unsigned park0 = tbase + ((unsigned)(32 * (warp & 3)) << 16) + (unsigned)((warp >> 2) * 64), park1 = park0 + 32;

    const int ngroups = (npairs + C::PPC - 1) / C::PPC;
    const int my_groups = (blockIdx.x < ngroups) ? (ngroups - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
    const int nfetch = 4 * my_groups;
    // fetch number n of this pair slot: pair group blockIdx.x + (n / 4) * gridDim.x, field n % 4 (T_u, T_zx, T_v, T_zy),
    // buffer n & 1
#define XFB_PAIR_OF(g_) (((g_) * C::PPC + lane_pair < npairs) ? ((g_) * C::PPC + lane_pair) : (npairs - 1))
#define XFB_FETCH(n_)                                                                                                  \
    do {                                                                                                               \
        const int nn_ = (n_);                                                                                          \
        if (t == 0 && nn_ < nfetch) {                                                                                  \
            const int pr_ = XFB_PAIR_OF((int)blockIdx.x + (nn_ >> 2) * (int)gridDim.x);                                \
            const int fi_ = nn_ & 3;                                                                                   \
            const cpx *base_ = (fi_ == 0) ? p.spec_in[2] : (fi_ == 1) ? p.spec_in[0] : (fi_ == 2) ? p.spec_in[3] : p.spec_in[1]; \
            mbar_expect_tx(mbar + (nn_ & 1), (unsigned)(2 * p.pitch * sizeof(cpx)));                                   \
            bulk_g2s(stage0 + (nn_ & 1) * ST_STRIDE, base_ + (size_t)pr_ * (size_t)(2 * p.pitch),                      \
                     (unsigned)(2 * p.pitch * sizeof(cpx)), mbar + (nn_ & 1));                                         \
        }                                                                                                              \
    } while (0)
    XFB_FETCH(0);
    XFB_FETCH(1);
    cpx v[16];
    // ONE flat loop over the fetches of this pair slot (field f = n & 3 of pair group n >> 2): the only loop-carried
    // scalar is n -- staging buffer n & 1 is on its (n >> 1)-th use, so its mbarrier parity is (n >> 1) & 1, and the
    // pair offsets are recomputed where they are needed instead of living (spilled) across the transforms.
#pragma unroll 1
    for (int n = 0; n < nfetch; ++n) {
        const int f = n & 3;
        {
            const int b = n & 1;
            mbar_wait(mbar + b, (unsigned)(n >> 1) & 1u);
            const float4 *st = reinterpret_cast<const float4 *>(stage0 + b * ST_STRIDE);
#pragma unroll
            for (int h = 0; h < 2; ++h) {
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                    const int pos = t + (8 * h + e) * G;
                    const int m = (h == 0) ? pos : NY - pos;
                    float4 x = st[m];
                    if ((h == 0 && e == 0 && pos == 0) || (h == 1 && e == 0 && pos == NY / 2)) { x.y = 0.f; x.w = 0.f; }
                    v[8 * h + e] = (h == 0) ? mk(x.y + x.z, x.x - x.w) : mk(x.z - x.y, x.x + x.w);
                }
            }
        }
        bar.sync();                 // everyone has read this staging buffer: refill it two fields ahead
        XFB_FETCH(n + 2);
        if constexpr (SPLIT) fft8192_to_split<1>(v, sm, t, 0, tw, bar);
        else line_fft<NY, 1>(v, sm, t, 0, tw, bar);
        // v = (b[n], a[n]) unscaled, swapped: .y is row 2m, .x row 2m+1.  Tensor-memory traffic in halves of
        // eight values (16 registers) so that nothing spills next to the live butterfly set.
        if (f == 0 || f == 2) {
            const unsigned park = (f == 0) ? park0 : park1;
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                cpx a[8];
#pragma unroll
                for (int q = 0; q < 8; ++q) a[q] = mk(v[8 * h + q].y * p.scale, v[8 * h + q].x * p.scale);      // -u ; v
                tmem_park8(park + 16 * h, a);
            }
            continue;
        }
        if (f == 1) {
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                cpx a[8];
                tmem_unpark8(park0 + 16 * h, a);
#pragma unroll
                for (int q = 0; q < 8; ++q)
                    a[q] = mk(a[q].x * (v[8 * h + q].y * p.scale), a[q].y * (v[8 * h + q].x * p.scale));           // -u dvortdx
                tmem_park8(park0 + 16 * h, a);
            }
            continue;
        }
        // f == 3: J = (-u dvortdx) - v dvortdy, formed in place in v                             main.cpp:225-227
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            cpx a[8];
            tmem_unpark8(park1 + 16 * h, a);
#pragma unroll
            for (int q = 0; q < 8; ++q)
                v[8 * h + q] = mk(a[q].x * (v[8 * h + q].y * p.scale), a[q].y * (v[8 * h + q].x * p.scale));          // v dvortdy
            tmem_unpark8(park0 + 16 * h, a);
#pragma unroll
            for (int q = 0; q < 8; ++q) v[8 * h + q] = mk(a[q].x - v[8 * h + q].x, a[q].y - v[8 * h + q].y);
        }
        const int g = (int)blockIdx.x + (n >> 2) * (int)gridDim.x;
        const int pr = XFB_PAIR_OF(g);
        const bool alive = g * C::PPC + lane_pair < npairs;
        if (p.real_in != nullptr) {
            const float *sa = p.real_in + (size_t)pr * (size_t)(2 * NY) + slot_base<NY, SPLIT>(t), *sb = sa + NY;
#pragma unroll
            for (int q = 0; q < 16; ++q)
                v[q] = mk(v[q].x + __ldg(sa + slot_off<NY, SPLIT>(q)), v[q].y + __ldg(sb + slot_off<NY, SPLIT>(q)));
        }
        // the thread index is laundered per pair: otherwise the 24 padded shared-memory positions of the forward
        // transform's tail are hoisted out of the pair loop and spilled (16 local loads per pair on the critical path)
        int tl = t;
        asm volatile("" : "+r"(tl));
        r2c_pair<NY, false, Bar, false, SPLIT>(v, p.spec_out + (size_t)pr * (size_t)(2 * p.pitch), p, alive ? p.pitch : 0, sm, tl, tw,
                                               bar);
    }
#undef XFB_FETCH
#undef XFB_PAIR_OF
    tmem_free_cta<C::TCOLS>(tbase);
}

template <int NY, int MODE, bool DIST>
__global__ void __launch_bounds__(PairCfg<NY>::THREADS, PairCfg<NY>::MINB)
rowpair_kernel(const RowParams p)
{
    typedef PairCfg<NY> C;
    constexpr int G = C::G;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane_pair = threadIdx.x / G;
    const int t = threadIdx.x % G;
    cpx *sm = reinterpret_cast<cpx *>(smem_raw) + (size_t)lane_pair * LinePlan<NY>::PADDED;
    const int npairs = p.nrows >> 1;
    int pair = blockIdx.x * C::PPC + lane_pair;
    const bool live = pair < npairs;
    if (!live) pair = npairs - 1;
    const int rowpitch = DIST ? p.cw : p.pitch;
    const size_t off = (size_t)pair * (size_t)(2 * rowpitch);       // pair base in a pair-layout array
    const size_t roff = (size_t)pair * (size_t)(2 * NY);            // first of the two physical rows

    LineTw<NY> tw;
    tw.init(p.tw, p.twn, t);
    typedef typename RowBarSel<(G >= 32 && C::PPC > 1)>::type Bar;
    const Bar bar = RowBarSel<(G >= 32 && C::PPC > 1)>::make(1 + lane_pair, G);

    cpx v[16];
    if (MODE == ROW_R2C) {
        const float *a = p.real_in + roff, *b = a + NY;
#pragma unroll
        for (int q = 0; q < 16; ++q) v[q] = mk(__ldg(a + t + q * G), __ldg(b + t + q * G));
        r2c_pair<NY, DIST>(v, p.spec_out + off, p, live ? p.pitch : 0, sm, t, tw, bar);
    } else if (MODE == ROW_C2R) {
        c2r_pair<NY, DIST>(v, p.spec_in[0] + off, p, sm, t, tw, bar);
        float *a = p.real_out + roff, *b = a + NY;
        const float s = p.negate ? -p.scale : p.scale;
#pragma unroll
        for (int q = 0; q < 16; ++q) {
            a[t + q * G] = v[q].y * s;
            b[t + q * G] = v[q].x * s;
        }
    } else if (DIST) {
        jac_pair_direct<NY, DIST>(p, smem_raw, sm, lane_pair, t, off, roff, live, tw, bar);
    } else if (MODE == ROW_DIAG) {
        // ---- diagnostics: three inverse transforms per row pair and a pointwise combine, same TMA-staged persistent
        // machinery as the Jacobian below.  kind 0: (psi_xy, psi_xx, psi_yy) -> filamentation time 2/sqrt(S1^2+S2^2-zeta^2)
        // (Rozoff et al. 2006) and deformation factor (README.md:5,7); kind 1: (zeta, zeta_x, zeta_y) -> zeta and
        // |grad zeta|^2 for the effective-diffusivity histograms (README.md:6, Hendricks & Schubert 2009).
        __shared__ unsigned long long mbar_all[C::PPC];
        unsigned long long *mbar = &mbar_all[lane_pair];
        if (t == 0) {
            mbar_init(mbar, 1);
            mbar_fence_init();
        }
        __syncthreads();
        const unsigned bytes = (unsigned)(2 * p.pitch * sizeof(cpx));
        const int ngroups = (npairs + C::PPC - 1) / C::PPC;
        unsigned phase = 0;
        cpx *park0 = reinterpret_cast<cpx *>(smem_raw) + (size_t)C::PPC * LinePlan<NY>::PADDED + (size_t)lane_pair * (2 * NY);
        const cpx *const f0 = p.spec_in[0], *const f1 = p.spec_in[1], *const f2 = p.spec_in[2];
        const size_t pair_stride = (size_t)(2 * p.pitch);
#define XFB_PAIR_OF(g_) (((g_) * C::PPC + lane_pair < npairs) ? ((g_) * C::PPC + lane_pair) : (npairs - 1))
#define XFB_FETCH(base_, pr_)                                                   \
    do {                                                                        \
        if (t == 0) {                                                           \
            mbar_expect_tx(mbar, bytes);                                        \
            bulk_g2s(sm, (base_) + (size_t)(pr_) * pair_stride, bytes, mbar);   \
        }                                                                       \
    } while (0)
        int g = blockIdx.x;
        if (g < ngroups) XFB_FETCH(f0, XFB_PAIR_OF(g));
        for (; g < ngroups; g += gridDim.x) {
            const int pr = XFB_PAIR_OF(g);
            const size_t ro = (size_t)pr * (size_t)(2 * NY);
#pragma unroll 1
            for (int f = 0; f < 3; ++f) {
                mbar_wait(mbar, phase);
                phase ^= 1;
                c2r_pair_staged<NY, Bar, true>(v, sm, t, tw, bar);
                if (f < 2) XFB_FETCH((f == 0) ? f1 : f2, pr);
                else {
                    const int gn = g + gridDim.x;
                    if (gn < ngroups) XFB_FETCH(f0, XFB_PAIR_OF(gn));
                }
                if (f < 2) {
                    cpx *park = park0 + f * NY;
#pragma unroll
                    for (int q = 0; q < 16; ++q) park[q * G + t] = mk(v[q].y * p.scale, v[q].x * p.scale);
                }
            }
            float *oa = p.real_out + ro, *ob = oa + NY, *o2a = p.real_out2 + ro, *o2b = o2a + NY;
#pragma unroll
            for (int q = 0; q < 16; ++q) {
                const cpx a0 = park0[q * G + t], a1 = park0[NY + q * G + t];
                const cpx a2 = mk(v[q].y * p.scale, v[q].x * p.scale);
                float r0[2], r1[2];
#pragma unroll
                for (int w = 0; w < 2; ++w) {
                    const float x0 = w ? a0.y : a0.x, x1 = w ? a1.y : a1.x, x2 = w ? a2.y : a2.x;
                    if (p.diag_kind == 0) {
                        // S1 = -2 psi_xy, S2 = psi_xx - psi_yy, zeta = psi_xx + psi_yy          (diag_kernel, xfb_api.cu)
                        const float s1 = __fmul_rn(-2.0f, x0), s2 = __fsub_rn(x1, x2), z = __fadd_rn(x1, x2);
                        const float ss = __fadd_rn(__fmul_rn(s1, s1), __fmul_rn(s2, s2)), zz = __fmul_rn(z, z);
                        const float qq = __fsub_rn(ss, zz), den = __fadd_rn(ss, zz);
                        r0[w] = (qq > 0.0f) ? __fdiv_rn(2.0f, __fsqrt_rn(qq)) : 0.0f;
                        r1[w] = (den > 0.0f) ? __fdiv_rn(qq, den) : 0.0f;
                    } else {
                        r0[w] = x0;
                        r1[w] = __fadd_rn(__fmul_rn(x1, x1), __fmul_rn(x2, x2));
                    }
                }
                oa[t + q * G] = r0[0]; ob[t + q * G] = r0[1];
                o2a[t + q * G] = r1[0]; o2b[t + q * G] = r1[1];
            }
        }
#undef XFB_FETCH
#undef XFB_PAIR_OF
    } else {
        // ---- persistent, TMA-staged: CTA g handles pair groups g, g + gridDim.x, ...  Every spectral line pair is
        // fetched by ONE cp.async.bulk into the FFT buffer (free at that moment) and the fetch of the next field is
        // issued as soon as the current transform has finished with the buffer, so it overlaps the last butterfly
        // pass and the Jacobian arithmetic; the first field of the NEXT pair is fetched under the output stores.
        __shared__ unsigned long long mbar_all[C::PPC];
        unsigned long long *mbar = &mbar_all[lane_pair];
        if (t == 0) {
            mbar_init(mbar, 1);
            mbar_fence_init();
        }
        __syncthreads();
        const unsigned bytes = (unsigned)(2 * p.pitch * sizeof(cpx));
        const int ngroups = (npairs + C::PPC - 1) / C::PPC;
        unsigned phase = 0;
        cpx *park0 = reinterpret_cast<cpx *>(smem_raw) + (size_t)C::PPC * LinePlan<NY>::PADDED + (size_t)lane_pair * (2 * NY);
        const cpx *const f_tu = p.spec_in[2], *const f_zx = p.spec_in[0], *const f_tv = p.spec_in[3], *const f_zy = p.spec_in[1];
        const size_t pair_stride = (size_t)(2 * p.pitch);
#define XFB_PAIR_OF(g_) (((g_) * C::PPC + lane_pair < npairs) ? ((g_) * C::PPC + lane_pair) : (npairs - 1))
#define XFB_FETCH(base_, pr_)                                                   \
    do {                                                                        \
        if (t == 0) {                                                           \
            mbar_expect_tx(mbar, bytes);                                        \
            bulk_g2s(sm, (base_) + (size_t)(pr_) * pair_stride, bytes, mbar);   \
        }                                                                       \
    } while (0)
        int g = blockIdx.x;
        if (g < ngroups) XFB_FETCH(f_tu, XFB_PAIR_OF(g));
        for (; g < ngroups; g += gridDim.x) {
            const int pr = XFB_PAIR_OF(g);
            const bool alive = g * C::PPC + lane_pair < npairs;
            const size_t po = (size_t)pr * (size_t)(2 * p.pitch), ro = (size_t)pr * (size_t)(2 * NY);
            for (int o = t * 128; o < (int)bytes; o += G * 128) {       // the other three fields towards L2
                prefetch_l2(reinterpret_cast<const char *>(p.spec_in[0] + po) + o);
                prefetch_l2(reinterpret_cast<const char *>(p.spec_in[3] + po) + o);
                prefetch_l2(reinterpret_cast<const char *>(p.spec_in[1] + po) + o);
            }
#pragma unroll 1
            for (int f = 0; f < 4; ++f) {
                mbar_wait(mbar, phase);
                phase ^= 1;
                c2r_pair_staged<NY, Bar, true>(v, sm, t, tw, bar);
                if (f < 3) XFB_FETCH((f == 0) ? f_zx : (f == 1) ? f_tv : f_zy, pr);      // order T_u, T_zx, T_v, T_zy
                cpx *park = park0 + (f >> 1) * NY;
                if (f == 1) {
#pragma unroll
                    for (int q = 0; q < 16; ++q) {
                        const cpx a = park[q * G + t];
                        park[q * G + t] = mk(a.x * (v[q].y * p.scale), a.y * (v[q].x * p.scale));
                    }
                } else if (f != 3) {
#pragma unroll
                    for (int q = 0; q < 16; ++q) park[q * G + t] = mk(v[q].y * p.scale, v[q].x * p.scale);
                }
            }
            // f = 3 left dvortdy in v: J = (-u dvortdx) - v dvortdy straight from the two parks (main.cpp:225-227)
            cpx J[16];
#pragma unroll
            for (int q = 0; q < 16; ++q) {
                const cpx j1 = park0[q * G + t], b = park0[NY + q * G + t];
                const cpx j2 = mk(b.x * (v[q].y * p.scale), b.y * (v[q].x * p.scale));
                J[q] = mk(j1.x - j2.x, j1.y - j2.y);
            }
            if (p.real_in != nullptr) {
                const float *sa = p.real_in + ro, *sb = sa + NY;
#pragma unroll
                for (int q = 0; q < 16; ++q) J[q] = mk(J[q].x + __ldg(sa + t + q * G), J[q].y + __ldg(sb + t + q * G));
            }
            // forward transform; the buffer is released before the output stores so the next pair's first field
            // is already on its way while they drain
            r2c_pair_begin<NY, Bar>(J, sm, t, tw, bar);
            const int gn = g + gridDim.x;
            if (gn < ngroups) XFB_FETCH(f_tu, XFB_PAIR_OF(gn));
            r2c_pair_finish<NY, DIST>(J, p.spec_out + po, p, alive ? p.pitch : 0, t);
        }
#undef XFB_FETCH
#undef XFB_PAIR_OF
    }
}

}  // namespace xfb

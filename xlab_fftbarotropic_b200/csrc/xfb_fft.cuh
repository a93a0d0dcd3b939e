// xfb_fft.cuh -- register/shared-memory FFT building blocks for sm_100a.
//
// Scheme (validated against numpy in the design prototype, see DESIGN.md "FFT engine"):
//   * one "butterfly thread" owns R = 16 complex values of a line of length L, at positions
//     t + k*G (G = L/16, k = 0..15) -- in EVERY pass and at the end of the transform, so
//     consecutive transforms (c2r -> Jacobian -> r2c, forward -> epilogue -> inverse) chain
//     in registers without a re-layout;
//   * Stockham autosort passes: radix-16 passes first, the remainder radix (2/4/8) last;
//     the first pass reads straight from global memory (coalesced across t), the last
//     pass leaves natural-order output in registers for a coalesced global store;
//     only the exchanges between passes go through shared memory (padded: pos + pos/16,
//     conflict-free for 8-byte accesses);
//   * twiddles: one table lookup per thread per pass (kept in registers for the whole
//     kernel), powers by a depth-4 multiplication tree;
//   * inverse transforms use the swap trick  ifft(x) = swap(fft(swap(x))).
#pragma once
#include <cuda_runtime.h>

namespace xfb {

typedef float2 cpx;

__device__ __forceinline__ cpx mk(float x, float y) { return make_float2(x, y); }
__device__ __forceinline__ cpx cadd(cpx a, cpx b) { return mk(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ cpx csub(cpx a, cpx b) { return mk(a.x - b.x, a.y - b.y); }
__device__ __forceinline__ cpx cmul(cpx a, cpx b) { return mk(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x); }
__device__ __forceinline__ cpx cconj(cpx a) { return mk(a.x, -a.y); }
__device__ __forceinline__ cpx cswap(cpx a) { return mk(a.y, a.x); }
__device__ __forceinline__ cpx mul_negi(cpx a) { return mk(a.y, -a.x); }   // a * (-i)
__device__ __forceinline__ cpx mul_i(cpx a) { return mk(-a.y, a.x); }      // a * (+i)

// Identity the compiler cannot see through.  The twiddle bases are per-thread constants for the whole
// kernel; without this the compiler keeps all their powers (60+ registers) live across the five
// transforms of a row/tile and spills.  Laundering the base at each use forces a cheap recomputation.
__device__ __forceinline__ cpx launder(cpx w)
{
    asm volatile("" : "+f"(w.x), "+f"(w.y));
    return w;
}

__device__ __forceinline__ void prefetch_l2(const void *ptr) { asm volatile("prefetch.global.L2 [%0];" ::"l"(ptr)); }
// one instruction pulls a whole contiguous range towards L2 (16-byte aligned, size a multiple of 16)
__device__ __forceinline__ void bulk_prefetch_l2(const void *ptr, unsigned bytes)
{
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(ptr), "r"(bytes) : "memory");
}

// ---- TMA bulk copies (cp.async.bulk, SASS UBLKCP) and their mbarrier --------------------------------------
__device__ __forceinline__ unsigned smem_u32(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void mbar_init(unsigned long long *bar, int count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(unsigned long long *bar, unsigned bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long *bar, unsigned parity)
{
    unsigned ok = 0;
    while (!ok) {
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n"
            : "=r"(ok)
            : "r"(smem_u32(bar)), "r"(parity)
            : "memory");
    }
}
// global -> shared, contiguous `bytes` (multiple of 16, both addresses 16-byte aligned), completion on `bar`
__device__ __forceinline__ void bulk_g2s(void *dst_smem, const void *src_gmem, unsigned bytes, unsigned long long *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// 2-D tiled TMA (cp.async.bulk.tensor.2d, SASS UTMALDG / UTMASTG); `map` is a CUtensorMap in kernel-parameter space
__device__ __forceinline__ void tma_load_2d(void *dst_smem, const void *map, int x, int y, unsigned long long *bar)
{
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
                     smem_u32(dst_smem)),
                 "l"(map), "r"(x), "r"(y), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void tma_store_2d(const void *map, int x, int y, const void *src_smem)
{
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.tile.bulk_group [%0, {%1, %2}], [%3];" ::"l"(map), "r"(x), "r"(y),
                 "r"(smem_u32(src_smem))
                 : "memory");
}
// pull a tile towards L2 only (no shared-memory destination): exactly the box's sectors, unlike prefetch.global.L2
__device__ __forceinline__ void tma_prefetch_2d(const void *map, int x, int y)
{
    asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global.tile [%0, {%1, %2}];" ::"l"(map), "r"(x), "r"(y) : "memory");
}
__device__ __forceinline__ void tma_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// all committed bulk stores have finished READING shared memory (the buffer may be overwritten)
__device__ __forceinline__ void tma_wait_read_all() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
// all but the N most recent committed bulk groups have finished reading shared memory
template <int N>
__device__ __forceinline__ void tma_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
// the same with a loop counter (0..15) that is constant after unrolling
__device__ __forceinline__ void tma_wait_read_n(const int n)
{
    switch (n) {
    case 0: tma_wait_read<0>(); break;   case 1: tma_wait_read<1>(); break;   case 2: tma_wait_read<2>(); break;
    case 3: tma_wait_read<3>(); break;   case 4: tma_wait_read<4>(); break;   case 5: tma_wait_read<5>(); break;
    case 6: tma_wait_read<6>(); break;   case 7: tma_wait_read<7>(); break;   case 8: tma_wait_read<8>(); break;
    case 9: tma_wait_read<9>(); break;   case 10: tma_wait_read<10>(); break; case 11: tma_wait_read<11>(); break;
    case 12: tma_wait_read<12>(); break; case 13: tma_wait_read<13>(); break; case 14: tma_wait_read<14>(); break;
    default: tma_wait_read<15>(); break;
    }
}
// all committed bulk stores are complete (global memory written)
__device__ __forceinline__ void tma_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// ---- tensor memory (TMEM) as thread-private scratch ------------------------------------------------------------
// 256 KB per SM next to the register file, reached with tcgen05.ld / tcgen05.st (SASS LDTM / STTM).  The .32x32b
// shape maps thread i of a warp to lane 32*(warp%4)+i and register r to column col+r: every thread owns a private row,
// which is exactly what "parking" 32 registers needs -- without touching the shared-memory pipe the FFT exchanges
// saturate.  One warp allocates `COLS` columns (power of two >= 32) for the CTA and frees them at the end.
template <int COLS>
__device__ __forceinline__ unsigned tmem_alloc_cta(unsigned *slot_smem)
{
    if ((threadIdx.x >> 5) == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot_smem)), "n"(COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    return *slot_smem;
}
template <int COLS>
__device__ __forceinline__ void tmem_free_cta(unsigned base)
{
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if ((threadIdx.x >> 5) == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(base), "n"(COLS) : "memory");
}
// 16 complex registers <-> 32 columns of this thread's TMEM row
__device__ __forceinline__ void tmem_park(unsigned taddr, const cpx (&r)[16])
{
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
        "{%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,%32};" ::"r"(taddr),
        "f"(r[0].x), "f"(r[0].y), "f"(r[1].x), "f"(r[1].y), "f"(r[2].x), "f"(r[2].y), "f"(r[3].x), "f"(r[3].y), "f"(r[4].x), "f"(r[4].y),
        "f"(r[5].x), "f"(r[5].y), "f"(r[6].x), "f"(r[6].y), "f"(r[7].x), "f"(r[7].y), "f"(r[8].x), "f"(r[8].y), "f"(r[9].x), "f"(r[9].y),
        "f"(r[10].x), "f"(r[10].y), "f"(r[11].x), "f"(r[11].y), "f"(r[12].x), "f"(r[12].y), "f"(r[13].x), "f"(r[13].y), "f"(r[14].x),
        "f"(r[14].y), "f"(r[15].x), "f"(r[15].y)
        : "memory");
}
// one complex register -> 2 columns
__device__ __forceinline__ void tmem_park1(unsigned taddr, const cpx r)
{
    asm volatile("tcgen05.st.sync.aligned.32x32b.x2.b32 [%0], {%1,%2};" ::"r"(taddr), "f"(r.x), "f"(r.y) : "memory");
}
// 8 complex registers -> 16 columns
__device__ __forceinline__ void tmem_park8(unsigned taddr, const cpx (&r)[8])
{
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};" ::"r"(taddr),
        "f"(r[0].x), "f"(r[0].y), "f"(r[1].x), "f"(r[1].y), "f"(r[2].x), "f"(r[2].y), "f"(r[3].x), "f"(r[3].y), "f"(r[4].x), "f"(r[4].y),
        "f"(r[5].x), "f"(r[5].y), "f"(r[6].x), "f"(r[6].y), "f"(r[7].x), "f"(r[7].y)
        : "memory");
}
// 16 columns -> 8 complex registers; waits for this thread's earlier stores and for the load itself inside ONE asm
// statement, so no use of the result can be scheduled ahead of the wait.  Eight values at a time keep the register
// peak at 16 + the consumer's state (a 32-register LDTM next to a live butterfly set spills).
__device__ __forceinline__ void tmem_unpark8(unsigned taddr, cpx (&r)[8])
{
    asm volatile(
        "tcgen05.wait::st.sync.aligned;\n\t"
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];\n\t"
        "tcgen05.wait::ld.sync.aligned;"
        : "=f"(r[0].x), "=f"(r[0].y), "=f"(r[1].x), "=f"(r[1].y), "=f"(r[2].x), "=f"(r[2].y), "=f"(r[3].x), "=f"(r[3].y), "=f"(r[4].x),
          "=f"(r[4].y), "=f"(r[5].x), "=f"(r[5].y), "=f"(r[6].x), "=f"(r[6].y), "=f"(r[7].x), "=f"(r[7].y)
        : "r"(taddr)
        : "memory");
}
// 8 columns -> 4 complex registers (same waits as tmem_unpark8)
__device__ __forceinline__ void tmem_unpark4(unsigned taddr, cpx (&r)[4])
{
    asm volatile(
        "tcgen05.wait::st.sync.aligned;\n\t"
        "tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];\n\t"
        "tcgen05.wait::ld.sync.aligned;"
        : "=f"(r[0].x), "=f"(r[0].y), "=f"(r[1].x), "=f"(r[1].y), "=f"(r[2].x), "=f"(r[2].y), "=f"(r[3].x), "=f"(r[3].y)
        : "r"(taddr)
        : "memory");
}
// the stores above complete asynchronously; a load of what they wrote waits for them first
__device__ __forceinline__ void tmem_unpark(unsigned taddr, cpx (&r)[16])
{
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
        : "=f"(r[0].x), "=f"(r[0].y), "=f"(r[1].x), "=f"(r[1].y), "=f"(r[2].x), "=f"(r[2].y), "=f"(r[3].x), "=f"(r[3].y), "=f"(r[4].x),
          "=f"(r[4].y), "=f"(r[5].x), "=f"(r[5].y), "=f"(r[6].x), "=f"(r[6].y), "=f"(r[7].x), "=f"(r[7].y), "=f"(r[8].x), "=f"(r[8].y),
          "=f"(r[9].x), "=f"(r[9].y), "=f"(r[10].x), "=f"(r[10].y), "=f"(r[11].x), "=f"(r[11].y), "=f"(r[12].x), "=f"(r[12].y),
          "=f"(r[13].x), "=f"(r[13].y), "=f"(r[14].x), "=f"(r[14].y), "=f"(r[15].x), "=f"(r[15].y)
        : "r"(taddr)
        : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

#define XFB_C8 0.70710678118654752440f
#define XFB_C16 0.92387953251128675613f
#define XFB_S16 0.38268343236508977173f

// ---- forward DFTs in registers, natural order in and out ---------------------------------

__device__ __forceinline__ void dft2(cpx &a, cpx &b)
{
    cpx t = a;
    a = cadd(t, b);
    b = csub(t, b);
}

__device__ __forceinline__ void dft4(cpx &a0, cpx &a1, cpx &a2, cpx &a3)
{
    cpx t0 = cadd(a0, a2), t1 = csub(a0, a2), t2 = cadd(a1, a3), t3 = mul_negi(csub(a1, a3));
    a0 = cadd(t0, t2);
    a1 = cadd(t1, t3);
    a2 = csub(t0, t2);
    a3 = csub(t1, t3);
}

__device__ __forceinline__ void dft8(cpx (&v)[8])
{
    // even/odd split: X[k] = E[k] + W8^k O[k], X[k+4] = E[k] - W8^k O[k]
    cpx e0 = v[0], e1 = v[2], e2 = v[4], e3 = v[6];
    cpx o0 = v[1], o1 = v[3], o2 = v[5], o3 = v[7];
    dft4(e0, e1, e2, e3);
    dft4(o0, o1, o2, o3);
    o1 = mk((o1.x + o1.y) * XFB_C8, (o1.y - o1.x) * XFB_C8);     // * (1 - i)/sqrt2
    o2 = mul_negi(o2);
    o3 = mk((o3.y - o3.x) * XFB_C8, -(o3.x + o3.y) * XFB_C8);    // * (-1 - i)/sqrt2
    v[0] = cadd(e0, o0); v[4] = csub(e0, o0);
    v[1] = cadd(e1, o1); v[5] = csub(e1, o1);
    v[2] = cadd(e2, o2); v[6] = csub(e2, o2);
    v[3] = cadd(e3, o3); v[7] = csub(e3, o3);
}

__device__ __forceinline__ void dft16(cpx (&v)[16])
{
    // n = c + 4a, q = k + 4m:  X[k+4m] = sum_c W4^(cm) [ W16^(ck) sum_a v[c+4a] W4^(ak) ]
#pragma unroll
    for (int c = 0; c < 4; ++c) dft4(v[c], v[c + 4], v[c + 8], v[c + 12]);
    // now v[c + 4k] holds u[c][k]; apply W16^(ck)
    const cpx w1 = mk(XFB_C16, -XFB_S16), w3 = mk(XFB_S16, -XFB_C16);
    v[1 + 4] = cmul(v[1 + 4], w1);                                                         // (1,1) W16^1
    v[1 + 8] = mk((v[1 + 8].x + v[1 + 8].y) * XFB_C8, (v[1 + 8].y - v[1 + 8].x) * XFB_C8); // (1,2) W16^2
    v[1 + 12] = cmul(v[1 + 12], w3);                                                       // (1,3) W16^3
    v[2 + 4] = mk((v[2 + 4].x + v[2 + 4].y) * XFB_C8, (v[2 + 4].y - v[2 + 4].x) * XFB_C8); // (2,1) W16^2
    v[2 + 8] = mul_negi(v[2 + 8]);                                                         // (2,2) W16^4
    v[2 + 12] = mk((v[2 + 12].y - v[2 + 12].x) * XFB_C8, -(v[2 + 12].x + v[2 + 12].y) * XFB_C8); // (2,3) W16^6
    v[3 + 4] = cmul(v[3 + 4], w3);                                                         // (3,1) W16^3
    v[3 + 8] = mk((v[3 + 8].y - v[3 + 8].x) * XFB_C8, -(v[3 + 8].x + v[3 + 8].y) * XFB_C8); // (3,2) W16^6
    v[3 + 12] = cmul(v[3 + 12], mk(-XFB_C16, XFB_S16));                                    // (3,3) W16^9
#pragma unroll
    for (int k = 0; k < 4; ++k) dft4(v[4 * k], v[4 * k + 1], v[4 * k + 2], v[4 * k + 3]);
    // v[4k + m] holds X[k + 4m]: transpose the 4x4 index back to natural order
#pragma unroll
    for (int k = 0; k < 4; ++k)
#pragma unroll
        for (int m = k + 1; m < 4; ++m) {
            cpx t = v[4 * k + m];
            v[4 * k + m] = v[4 * m + k];
            v[4 * m + k] = t;
        }
}

// w[s] = w1^s, s = 1..15 (w[0] unused); depth-4 product tree
__device__ __forceinline__ void pow_chain16(cpx w1, cpx (&w)[16])
{
    w[0] = mk(1.f, 0.f);
    w[1] = w1;
    w[2] = cmul(w1, w1);
    w[3] = cmul(w[2], w1);
    w[4] = cmul(w[2], w[2]);
    w[5] = cmul(w[4], w1);
    w[6] = cmul(w[3], w[3]);
    w[7] = cmul(w[4], w[3]);
    w[8] = cmul(w[4], w[4]);
#pragma unroll
    for (int s = 1; s < 8; ++s) w[8 + s] = cmul(w[8], w[s]);
}

// ---- line plan -----------------------------------------------------------------------------

template <int L>
struct LinePlan {
    static constexpr int R = 16;
    static constexpr int G = L / R;              // butterfly threads per line
    static constexpr int N16 = (L >= 65536) ? 4 : (L >= 4096) ? 3 : (L >= 256) ? 2 : (L >= 16) ? 1 : 0;
    static constexpr int P16 = (N16 == 4) ? 65536 : (N16 == 3) ? 4096 : (N16 == 2) ? 256 : (N16 == 1) ? 16 : 1;
    static constexpr int REM = L / P16;          // remainder radix: 1, 2, 4 or 8
    static constexpr int NPASS = N16 + (REM > 1 ? 1 : 0);
    static constexpr int PADDED = L + L / 16;    // shared-memory positions per line
    static_assert(L % 16 == 0 && P16 * REM == L, "line length must be 16^a * {1,2,4,8}");
};

__device__ __forceinline__ int padpos(int p) { return p + (p >> 4); }

// Per-thread twiddle bases for a line of length L, from the master table
// tw[k] = exp(-2 pi i k / TWN), k in [0, TWN) (TWN a multiple of L).
//   b[p], p = 1..N16-1 : radix-16 pass p      exp(-2 pi i (t mod 16^p) / 16^(p+1))
//   b[0]               : remainder pass       exp(-2 pi i t / L)
template <int L>
struct LineTw {
    cpx b[4];
    __device__ __forceinline__ void init(const cpx *__restrict__ tw, int twn, int t)
    {
        typedef LinePlan<L> P;
        int ns = 16;
#pragma unroll
        for (int p = 1; p < P::N16; ++p) {
            b[p] = __ldg(tw + (size_t)(t % ns) * (twn / (ns * 16)));
            ns *= 16;
        }
        b[0] = (P::REM > 1) ? __ldg(tw + (size_t)t * (twn / L)) : mk(1.f, 0.f);
    }
};

// ---- pass pieces (composed by line_fft below and by the multi-iteration column kernel) ----

// v[s] *= w1^s, s = 1..15.  Powers by a depth-4 product tree (w2, w4, w8 by squaring, the rest as
// products of two of them), generated and applied in an order that keeps few of them live.
__device__ __forceinline__ void apply_twiddles16(cpx (&v)[16], const cpx w1)
{
    const cpx w2 = cmul(w1, w1), w4 = cmul(w2, w2), w8 = cmul(w4, w4);
    v[1] = cmul(v[1], w1);
    v[2] = cmul(v[2], w2);
    v[4] = cmul(v[4], w4);
    v[8] = cmul(v[8], w8);
    v[9] = cmul(v[9], cmul(w8, w1));
    v[10] = cmul(v[10], cmul(w8, w2));
    v[12] = cmul(v[12], cmul(w8, w4));
    const cpx w3 = cmul(w2, w1);
    v[3] = cmul(v[3], w3);
    v[11] = cmul(v[11], cmul(w8, w3));
    const cpx w5 = cmul(w4, w1);
    v[5] = cmul(v[5], w5);
    v[13] = cmul(v[13], cmul(w8, w5));
    const cpx w6 = cmul(w4, w2);
    v[6] = cmul(v[6], w6);
    v[14] = cmul(v[14], cmul(w8, w6));
    const cpx w7 = cmul(w4, w3);
    v[7] = cmul(v[7], w7);
    v[15] = cmul(v[15], cmul(w8, w7));
}

// radix-16 pass p: twiddle (p > 0) + butterfly
template <int L>
__device__ __forceinline__ void pass16_compute(cpx (&v)[16], const int p, const LineTw<L> &tw)
{
    if (p > 0) apply_twiddles16(v, launder(tw.b[p]));
    dft16(v);
}

// Stockham scatter of pass-p results (ns = 16^p); element address = padpos(pos) * W + c.
// base % 16 + (s*ns) % 16 < 16 for every pass (ns = 1: base = 16 t; ns >= 16: s*ns % 16 = 0), so
// padpos(base + s*ns) = padpos(base) + s*ns + (s*ns >> 4): constant offsets from one address.
template <int W>
__device__ __forceinline__ void exchange_write(const cpx (&v)[16], cpx *sm, const int t, const int c, const int ns)
{
    const int base = (t / ns) * ns * 16 + (t % ns);
    cpx *dst = sm + padpos(base) * W + c;
#pragma unroll
    for (int s = 0; s < 16; ++s) dst[(s * ns + ((s * ns) >> 4)) * W] = v[s];
}

template <int G, int W>
__device__ __forceinline__ void exchange_read(cpx (&v)[16], const cpx *sm, const int t, const int c)
{
    if (G % 16 == 0) {
        const cpx *src = sm + padpos(t) * W + c;
#pragma unroll
        for (int k = 0; k < 16; ++k) v[k] = src[k * (G + G / 16) * W];
    } else {
#pragma unroll
        for (int k = 0; k < 16; ++k) v[k] = sm[padpos(t + k * G) * W + c];
    }
}

// remainder pass, radix r = REM (last pass): butterflies q = 0..16/r-1 at j = t + q*G use register
// slots q + s*(16/r); twiddle exp(-2 pi i j / L) = b[0] * exp(-2 pi i q / 16)
template <int L>
__device__ __forceinline__ void rem_pass(cpx (&v)[16], const LineTw<L> &tw)
{
    typedef LinePlan<L> P;
    if (P::REM > 1) {
        constexpr int r = (P::REM > 1) ? P::REM : 2, nb = 16 / r;
        const float CQ[8] = {1.f, XFB_C16, XFB_C8, XFB_S16, 0.f, -XFB_S16, -XFB_C8, -XFB_C16};
        const float SQ[8] = {0.f, -XFB_S16, -XFB_C8, -XFB_C16, -1.f, -XFB_C16, -XFB_C8, -XFB_S16};
        const cpx wb = launder(tw.b[0]);
#pragma unroll
        for (int q = 0; q < nb; ++q) {
            const cpx w1 = (q == 0) ? wb : cmul(wb, mk(CQ[q], SQ[q]));
            if (r == 2) {
                cpx a = v[q], b = cmul(v[q + nb], w1);
                v[q] = cadd(a, b);
                v[q + nb] = csub(a, b);
            } else if (r == 4) {
                cpx w2 = cmul(w1, w1), w3 = cmul(w2, w1);
                cpx a0 = v[q], a1 = cmul(v[q + nb], w1), a2 = cmul(v[q + 2 * nb], w2), a3 = cmul(v[q + 3 * nb], w3);
                dft4(a0, a1, a2, a3);
                v[q] = a0; v[q + nb] = a1; v[q + 2 * nb] = a2; v[q + 3 * nb] = a3;
            } else {
                cpx a[8];
                cpx w2 = cmul(w1, w1), w3 = cmul(w2, w1), w4 = cmul(w2, w2);
                a[0] = v[q];
                a[1] = cmul(v[q + nb], w1);
                a[2] = cmul(v[q + 2 * nb], w2);
                a[3] = cmul(v[q + 3 * nb], w3);
                a[4] = cmul(v[q + 4 * nb], w4);
                a[5] = cmul(v[q + 5 * nb], cmul(w4, w1));
                a[6] = cmul(v[q + 6 * nb], cmul(w3, w3));
                a[7] = cmul(v[q + 7 * nb], cmul(w4, w3));
                dft8(a);
#pragma unroll
                for (int s = 0; s < 8; ++s) v[q + s * nb] = a[s];
            }
        }
    }
}

// Barriers.  A CTA that transforms several independent lines gives each line its own named barrier so the
// lines do not wait for one another (they behave like separate CTAs sharing one SM's shared memory).
struct CtaBar {
    __device__ __forceinline__ void sync() const { __syncthreads(); }
};
struct NamedBar {
    int id, nthreads;      // id 1..4 (immediate barrier names keep the CTA's barrier allocation small), nthreads % 32 == 0
    __device__ __forceinline__ void sync() const
    {
        switch (id) {
        case 1: asm volatile("bar.sync 1, %0;" ::"r"(nthreads) : "memory"); break;
        case 2: asm volatile("bar.sync 2, %0;" ::"r"(nthreads) : "memory"); break;
        case 3: asm volatile("bar.sync 3, %0;" ::"r"(nthreads) : "memory"); break;
        default: asm volatile("bar.sync 4, %0;" ::"r"(nthreads) : "memory"); break;
        }
    }
};

// Forward FFT of one line held as v[k] = x[t + k*G].  `sm` points at this line's padded
// shared buffer; element address = (padpos(pos) * W + c).  All threads of the CTA must call
// this together (it uses __syncthreads()).  On return v[k] = X[t + k*G].
// RELEASE: the shared buffer is handed to the async proxy (a TMA bulk copy) right after the transform; every
// thread then fences its generic-proxy accesses before the last barrier.
template <int L, int W, typename Bar, bool RELEASE = false>
__device__ __forceinline__ void line_fft(cpx (&v)[16], cpx *sm, const int t, const int c, const LineTw<L> &tw, const Bar &bar)
{
    typedef LinePlan<L> P;
    constexpr int NEX = (P::REM > 1) ? P::N16 : P::N16 - 1;     // exchanges
    int ns = 1;
#pragma unroll
    for (int p = 0; p < P::N16; ++p) {
        pass16_compute<L>(v, p, tw);
        if (p != P::NPASS - 1) {
            exchange_write<W>(v, sm, t, c, ns);
            bar.sync();
            exchange_read<P::G, W>(v, sm, t, c);
            if (RELEASE && p == NEX - 1) fence_proxy_async();
            bar.sync();
        }
        ns *= 16;
    }
    rem_pass<L>(v, tw);
}

// no-op hooks of col_fft and of the split 8192-point transforms below
struct ColFftNoHook {
    __device__ __forceinline__ void operator()(int, bool) const {}
};
struct ColFftNoPre {
    __device__ __forceinline__ void operator()() const {}
};

// ---- 8192-point lines with two exchanges: the radix-2 stage across lane pairs ------------------------------------------
// line_fft<8192> is R16 -> ex -> R16 -> ex -> R16 -> ex -> R2; the third exchange only regroups the data for the radix-2
// butterflies (j, j + 4096).  Here the third radix-16 pass is run by a remapped thread: thread t (warp w, lane l, lane half
// h = l >> 4) does the pass of the Stockham thread tau = 256 h + 16 w + (l & 15), so it ends up with E[j0 + 256 s] (h = 0) or
// O[j0 + 256 s] (h = 1), j0 = 16 w + (l & 15), s = 0..15: the two halves of every radix-2 butterfly sit in lanes l and l ^ 16.
// Lane h = 1 runs that pass with its twiddle base negated, which rotates its outputs by 8 slots (O[j0 + 256 ((s + 8) & 15)]
// in slot s), so both lanes send slot 8 + i and keep slot i; 8 complex values cross each way (16 shfl.xor per thread), and
// lane h owns the butterflies s = 8 h + i, i = 0..7.  The result is in the SPLIT order of Split8192::pos: slot k of thread t
// holds X[j0 + 2048 h + 256 (k & 7) + 4096 (k >> 3)].
//   fft8192_to_split   : input at t + 512 k (natural), output in the split order
//   fft8192_from_split : the transposed algorithm (lane-pair stage first, butterflies before twiddles), input in the split
//                        order, output at t + 512 k
// Both are forward transforms and use the twiddle bases of Split8192::init_tw.  The line's threads must be aligned to warps
// (t % 32 = lane), which holds for every 512-thread line.  tests/test_fft8192_lane_split_model.py models the addressing.
struct Split8192 {
    static constexpr int L = 8192, G = 512;
    __device__ static __forceinline__ int half(const int t) { return (t >> 4) & 1; }
    __device__ static __forceinline__ int j0(const int t) { return ((t >> 5) << 4) | (t & 15); }
    // the Stockham thread whose third radix-16 pass thread t runs
    __device__ static __forceinline__ int tau(const int t) { return (half(t) << 8) | j0(t); }
    // position of slot k of thread t: base(t) + off(k)
    __device__ static __forceinline__ int base(const int t) { return j0(t) + (half(t) << 11); }
    __host__ __device__ static constexpr int off(const int k) { return ((k & 7) << 8) + ((k >> 3) << 12); }
    // b[1] = exp(-2 pi i (t mod 16) / 256) as LineTw (tau mod 16 = t mod 16), b[2] = (-1)^h exp(-2 pi i j0 / 4096) for the
    // third pass, b[0] = exp(-2 pi i base(t) / 8192) for the lane-pair stage (times W32^i for butterfly s = 8 h + i)
    __device__ static __forceinline__ void init_tw(LineTw<L> &tw, const cpx *__restrict__ tab, const int twn, const int t)
    {
        tw.b[1] = __ldg(tab + (size_t)(t & 15) * (twn / 256));
        const cpx b2 = __ldg(tab + (size_t)j0(t) * (twn / 4096));
        tw.b[2] = half(t) ? mk(-b2.x, -b2.y) : b2;
        tw.b[0] = __ldg(tab + (size_t)base(t) * (twn / L));
    }
};

// slot k of thread t of a transformed line of length L: position t + k * L/16, or Split8192 order
template <int L, bool SPLIT>
__device__ __forceinline__ int slot_base(const int t) { return SPLIT ? Split8192::base(t) : t; }
template <int L, bool SPLIT>
__host__ __device__ __forceinline__ constexpr int slot_off(const int k) { return SPLIT ? Split8192::off(k) : k * (L / 16); }
template <int L, bool SPLIT>
__device__ __forceinline__ int slot_pos(const int t, const int k) { return slot_base<L, SPLIT>(t) + slot_off<L, SPLIT>(k); }

// W32^i = exp(-2 pi i i / 32), i = 0..7
#define XFB_C32 0.98078528040323044913f
#define XFB_S32 0.19509032201612826785f
#define XFB_C32_3 0.83146961230254523708f
#define XFB_S32_3 0.55557023301960222474f
__device__ __forceinline__ cpx lane_pair_twiddle(const cpx wb, const int i)
{
    const float CQ[8] = {1.f, XFB_C32, XFB_C16, XFB_C32_3, XFB_C8, XFB_S32_3, XFB_S16, XFB_S32};
    const float SQ[8] = {0.f, -XFB_S32, -XFB_S16, -XFB_S32_3, -XFB_C8, -XFB_C32_3, -XFB_C16, -XFB_C32};
    return (i == 0) ? wb : cmul(wb, mk(CQ[i], SQ[i]));
}
__device__ __forceinline__ cpx shfl_xor16(const cpx a)
{
    return mk(__shfl_xor_sync(0xffffffffu, a.x, 16), __shfl_xor_sync(0xffffffffu, a.y, 16));
}

// the exchange patterns of exchange_read / exchange_write, the other way round (transposed transforms)
template <int G, int W>
__device__ __forceinline__ void exchange_write_strided(const cpx (&v)[16], cpx *sm, const int t, const int c)
{
    static_assert(G % 16 == 0, "constant offsets need G % 16 == 0");
    cpx *dst = sm + padpos(t) * W + c;
#pragma unroll
    for (int k = 0; k < 16; ++k) dst[k * (G + G / 16) * W] = v[k];
}
template <int W>
__device__ __forceinline__ void exchange_read_stockham(cpx (&v)[16], const cpx *sm, const int t, const int c, const int ns)
{
    const int base = (t / ns) * ns * 16 + (t % ns);
    const cpx *src = sm + padpos(base) * W + c;
#pragma unroll
    for (int s = 0; s < 16; ++s) v[s] = src[(s * ns + ((s * ns) >> 4)) * W];
}

// hook(e, last) after exchange e has been read and its closing barrier passed; pre() right before the writes of the last
// exchange; drain_tma: thread 0 waits for the bulk stores reading shared memory before the last exchange's first barrier
// (the same points as col_fft)
template <int W, typename Bar, class Hook, class Pre>
__device__ __forceinline__ void fft8192_to_split(cpx (&v)[16], cpx *sm, const int t, const int c, const LineTw<8192> &tw,
                                                 const Bar &bar, const bool drain_tma, Hook &hook, Pre &pre)
{
    constexpr int G = Split8192::G;
    pass16_compute<8192>(v, 0, tw);
    exchange_write<W>(v, sm, t, c, 1);
    bar.sync();
    exchange_read<G, W>(v, sm, t, c);
    bar.sync();
    hook(0, false);
    pass16_compute<8192>(v, 1, tw);
    pre();
    exchange_write<W>(v, sm, t, c, 16);
    if (drain_tma && threadIdx.x == 0) tma_wait_read_all();
    bar.sync();
    exchange_read<G, W>(v, sm, Split8192::tau(t), c);
    bar.sync();
    hook(1, true);
    pass16_compute<8192>(v, 2, tw);
    // lane h: e = E (own slot i for h = 0, received for h = 1), o = O; butterfly s = 8 h + i -> slots i, 8 + i
    const bool hi = Split8192::half(t);
    const cpx wb = launder(tw.b[0]);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const cpx r = shfl_xor16(v[8 + i]);
        const cpx e = hi ? r : v[i], o = hi ? v[i] : r;
        const cpx b = cmul(o, lane_pair_twiddle(wb, i));
        v[i] = cadd(e, b);
        v[8 + i] = csub(e, b);
    }
}

template <int W, typename Bar, class Hook, class Pre>
__device__ __forceinline__ void fft8192_from_split(cpx (&v)[16], cpx *sm, const int t, const int c, const LineTw<8192> &tw,
                                                   const Bar &bar, const bool drain_tma, Hook &hook, Pre &pre)
{
    constexpr int G = Split8192::G;
    // transposed radix-2 butterflies (E' = x_j + x_(j+4096), O' = w^j (x_j - x_(j+4096))); lane h keeps E' (h = 0) or O'
    // (h = 1) in slot i and receives the partner's in slot 8 + i: the rotated order the transposed third pass expects
    const bool hi = Split8192::half(t);
    const cpx wb = launder(tw.b[0]);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const cpx a = cadd(v[i], v[8 + i]), b = cmul(csub(v[i], v[8 + i]), lane_pair_twiddle(wb, i));
        v[i] = hi ? b : a;
        v[8 + i] = shfl_xor16(hi ? a : b);
    }
    dft16(v);
    apply_twiddles16(v, launder(tw.b[2]));
    exchange_write_strided<G, W>(v, sm, Split8192::tau(t), c);
    bar.sync();
    exchange_read_stockham<W>(v, sm, t, c, 16);
    bar.sync();
    hook(0, false);
    dft16(v);
    apply_twiddles16(v, launder(tw.b[1]));
    pre();
    exchange_write_strided<G, W>(v, sm, t, c);
    if (drain_tma && threadIdx.x == 0) tma_wait_read_all();
    bar.sync();
    exchange_read_stockham<W>(v, sm, t, c, 1);
    bar.sync();
    hook(1, true);
    dft16(v);
}

template <int W, typename Bar>
__device__ __forceinline__ void fft8192_to_split(cpx (&v)[16], cpx *sm, const int t, const int c, const LineTw<8192> &tw, const Bar &bar)
{
    ColFftNoHook hook;
    ColFftNoPre pre;
    fft8192_to_split<W>(v, sm, t, c, tw, bar, false, hook, pre);
}
template <int W, typename Bar>
__device__ __forceinline__ void fft8192_from_split(cpx (&v)[16], cpx *sm, const int t, const int c, const LineTw<8192> &tw, const Bar &bar)
{
    ColFftNoHook hook;
    ColFftNoPre pre;
    fft8192_from_split<W>(v, sm, t, c, tw, bar, false, hook, pre);
}

}  // namespace xfb

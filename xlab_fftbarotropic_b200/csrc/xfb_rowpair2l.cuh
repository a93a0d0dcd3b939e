// xfb_rowpair2l.cuh -- K-ROW (ROW_JAC) for lines of NY = 16384 points: the two rows of a pair as ONE complex line of NY
// points (as in xfb_rowpair.cuh), transformed in TWO LEVELS: two half-length transforms of NY/2 points on NY/32 = 512
// threads with one butterfly each, and one radix-2 stage in registers.
//
// Same reference loops as xfb_rowpair.cuh: main.cpp:126-135,154,168,200-201,214,225-227,237 and
// fftwf_backward_normalize (:37-41).  Why a kernel of its own: a 16384-point line does not fit 512 threads x 16 values;
// the first-generation JAC kernel (since removed) addressed the pair layout with 8-byte loads at stride 16 and touched
// every spectral element twice (k and its mirror): 572 M global sectors for 134 M sectors of payload, stall_lg 2.4, 42 % of the
// issue slots used (profiles/r02_16384_gen1_ncu_full_summary.txt).  Here, like the 8192 kernel:
//   * persistent CTAs; the pair's contiguous region of a field (2 * pitch complex values, 131 KB) is fetched by
//     cp.async.bulk into ONE staging buffer in two halves with an mbarrier each, a field ahead of its use;
//   * inverse transform by decimation in frequency (swap trick): with U = swap(Z),
//       S[k] = U[k] + U[k + NY/2],  D[k] = (U[k] - U[k + NY/2]) W^k,   W = exp(-2 pi i / NY),  k < NY/2
//       even points = FFT_{NY/2}(S), odd points = FFT_{NY/2}(D).
//     U[k] comes from entry k of the staged spectrum, U[k + NY/2] from the mirror entry NY/2 - k: every thread reads its
//     32 entries once, keeps S, writes D into the LOWER half of the staging buffer (free once everybody has read), and
//     the upper half is refilled with the next field at once, the lower half after D has been read back;
//   * the products (-u, -u dvortdx, v) of the even and of the odd points are parked in TENSOR MEMORY (4 x 32 columns per
//     thread: all 512 columns of the SM);
//   * forward transform by decimation in time: O = FFT(J odd), E = FFT(J even), Z[k] = E + W^k O, Z[k + NY/2] = E - W^k O;
//     the half spectra of the two rows need Z[k] and Z[NY - k] = (E - W O)[NY/2 - k]: one mirror exchange of the upper
//     half through the transform buffer, then 16-byte stores of (A[k], B[k]).
#pragma once
#include "xfb_rowpair.cuh"

namespace xfb {

template <int NY>
struct Pair2LCfg {
    static constexpr int H = NY / 2;                                  // sub-transform length
    static constexpr int G = H / 16;                                  // threads
    static constexpr int THREADS = G;
    static constexpr int F_BYTES = LinePlan<H>::PADDED * (int)sizeof(cpx);
    static constexpr int LO_ENTRIES = H / 2;                          // entries [0, LO) = lower half of the staging buffer:
    static constexpr int LO_BYTES = LO_ENTRIES * 16;                  // exactly the H complex values of D
    static constexpr int TCOLS = (THREADS / 128) * 128;               // 4 parks of 32 columns per thread
    static_assert(THREADS == 512, "rowpair2l: NY = 16384 (512 threads, all of tensor memory)");
    static int smem_bytes(int pitch) { return F_BYTES + 2 * pitch * (int)sizeof(cpx); }
};

// DIST (slab-decomposed runs): a spectral line is cut into panels of p.cw columns (xfb_row.cuh); the pair's piece of every
// panel is contiguous, so the staging buffer is filled by one bulk copy per panel, and the output goes through
// out_addr<DIST> (local panels, or straight into the peers' receive arrays: the fused row -> column exchange).
template <int NY, bool DIST>
__global__ void __launch_bounds__(Pair2LCfg<NY>::THREADS, 1)
rowpair2l_jac_kernel(const RowParams p)
{
    typedef Pair2LCfg<NY> C;
    constexpr int H = C::H, G = C::G;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ unsigned tmem_slot;
    __shared__ unsigned long long mbar[2];                            // [0] lower half, [1] upper half of the staging buffer
    const int t = threadIdx.x;
    cpx *F = reinterpret_cast<cpx *>(smem_raw);
    unsigned char *stage_b = smem_raw + C::F_BYTES;
    const float4 *st = reinterpret_cast<const float4 *>(stage_b);      // staged spectrum: entry k = (A[k], B[k])
    cpx *dpark = reinterpret_cast<cpx *>(stage_b);                     // D[k] at complex index k (lower half)
    const int npairs = p.nrows >> 1;

    LineTw<H> tw;
    tw.init(p.tw, p.twn, t);
    const cpx wt = __ldg(p.tw + (size_t)t * (p.twn / NY));              // exp(-2 pi i t / NY)
    const CtaBar bar;

    if (t == 0) {
        mbar_init(&mbar[0], 1);
        mbar_init(&mbar[1], 1);
        mbar_fence_init();
    }
    const unsigned tbase = tmem_alloc_cta<C::TCOLS>(&tmem_slot);        // includes a CTA barrier
    const int warp = t >> 5;
    // parks of this thread: [0] products of the even points, [1] of the odd points (-u then -u dvortdx), [2]/[3] v
    const unsigned tp = tbase + ((unsigned)(32 * (warp & 3)) << 16) + (unsigned)((warp >> 2) * 128);

    const int my_pairs = (blockIdx.x < npairs) ? (npairs - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
    const int nfetch = 4 * my_pairs;
    // fetch number n: pair blockIdx.x + (n / 4) * gridDim.x, field n % 4 in the order T_u, T_zx, T_v, T_zy
    const int cw = DIST ? p.cw : p.pitch;                               // entries per contiguous piece of a pair region
    const size_t pstride = DIST ? (size_t)p.panel_stride : 0;           // complex elements between panels
    auto fetch_half = [&](const int n, const int upper) {                // thread 0 only
        if (n >= nfetch) return;
        const int fi = n & 3;
        const cpx *base = (fi == 0) ? p.spec_in[2] : (fi == 1) ? p.spec_in[0] : (fi == 2) ? p.spec_in[3] : p.spec_in[1];
        const int pr = (int)blockIdx.x + (n >> 2) * (int)gridDim.x;
        base += (size_t)pr * (size_t)(2 * cw);
        const int e_lo = upper ? C::LO_ENTRIES : 0, e_hi = upper ? p.pitch : C::LO_ENTRIES;     // entries [e_lo, e_hi)
        mbar_expect_tx(&mbar[upper], (unsigned)(e_hi - e_lo) * 16u);
        for (int panel = e_lo / cw; panel * cw < e_hi; ++panel) {
            const int e0 = panel * cw > e_lo ? panel * cw : e_lo;
            const int e1 = (panel + 1) * cw < e_hi ? (panel + 1) * cw : e_hi;
            bulk_g2s(stage_b + (size_t)e0 * 16, base + (size_t)panel * pstride + (size_t)(e0 - panel * cw) * 2, (unsigned)(e1 - e0) * 16u,
                     &mbar[upper]);
        }
    };
    if (t == 0) {
        fetch_half(0, 0);
        fetch_half(0, 1);
    }

    cpx v[16];
#pragma unroll 1
    for (int n = 0; n < nfetch; ++n) {
        const int f = n & 3;
        const unsigned par = (unsigned)n & 1u;
        mbar_wait(&mbar[0], par);
        mbar_wait(&mbar[1], par);
        // ---- S and D from the 32 entries of this thread: k = t + q G and its mirror H - k
        {
            const cpx wl = launder(wt);
            cpx d[16];
#pragma unroll
            for (int q = 0; q < 16; ++q) {
                const int k = t + q * G;
                float4 x = st[k];                                       // (A.re, A.im, B.re, B.im) of bin k
                float4 y = st[H - k];                                   // bin H - k (k = 0: the Nyquist bin H itself)
                if (q == 0 && k == 0) { x.y = 0.f; x.w = 0.f; y.y = 0.f; y.w = 0.f; }     // c2r ignores Im of DC and Nyquist
                // swapped for the inverse transform: U[k] = swap(A + iB), U[k + H] = swap(conj(A') + i conj(B')) (mirror),
                // or swap(A' + iB') for the Nyquist bin
                const cpx ud = mk(x.y + x.z, x.x - x.w);
                const cpx um = (q == 0 && k == 0) ? mk(y.y + y.z, y.x - y.w) : mk(y.z - y.y, y.x + y.w);
                v[q] = cadd(ud, um);
                d[q] = cmul(csub(ud, um), (q == 0) ? wl : cmul(wl, w32(q)));
            }
            fence_proxy_async();
            __syncthreads();                                            // everybody has read the staged spectrum
            if (t == 0) fetch_half(n + 1, 1);                           // upper half: next field, now
#pragma unroll
            for (int q = 0; q < 16; ++q) dpark[q * G + t] = d[q];       // D waits in the lower half
        }
        // two sub-transforms: sub = 0 even points (S), sub = 1 odd points (D)
#pragma unroll 1
        for (int sub = 0; sub < 2; ++sub) {
            if (sub == 1) {
#pragma unroll
                for (int q = 0; q < 16; ++q) v[q] = dpark[q * G + t];
                fence_proxy_async();
                __syncthreads();                                        // everybody has read D back
                if (t == 0) fetch_half(n + 1, 0);                       // lower half: next field
            }
            line_fft<H, 1>(v, F, t, 0, tw, bar);
            // v = (b, a) unscaled, swapped: .y is row 2m, .x row 2m+1, at the points 2 (t + q G) + sub
            const unsigned pk0 = tp + (unsigned)(sub * 32), pk1 = tp + 64u + (unsigned)(sub * 32);
            if (f == 0 || f == 2) {
                const unsigned park = (f == 0) ? pk0 : pk1;
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    cpx a[8];
#pragma unroll
                    for (int q = 0; q < 8; ++q) a[q] = mk(v[8 * h + q].y * p.scale, v[8 * h + q].x * p.scale);       // -u ; v
                    tmem_park8(park + 16 * h, a);
                }
            } else if (f == 1) {
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    cpx a[8];
                    tmem_unpark8(pk0 + 16 * h, a);
#pragma unroll
                    for (int q = 0; q < 8; ++q)
                        a[q] = mk(a[q].x * (v[8 * h + q].y * p.scale), a[q].y * (v[8 * h + q].x * p.scale));           // -u dvortdx
                    tmem_park8(pk0 + 16 * h, a);
                }
            } else {
                // f == 3: J = (-u dvortdx) - v dvortdy at these points (+ source), main.cpp:225-227
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    cpx a[8];
                    tmem_unpark8(pk1 + 16 * h, a);
#pragma unroll
                    for (int q = 0; q < 8; ++q)
                        v[8 * h + q] = mk(a[q].x * (v[8 * h + q].y * p.scale), a[q].y * (v[8 * h + q].x * p.scale));    // v dvortdy
                    tmem_unpark8(pk0 + 16 * h, a);
#pragma unroll
                    for (int q = 0; q < 8; ++q) v[8 * h + q] = mk(a[q].x - v[8 * h + q].x, a[q].y - v[8 * h + q].y);
                }
                if (p.real_in != nullptr) {
                    const int pr = (int)blockIdx.x + (n >> 2) * (int)gridDim.x;
                    const float *sa = p.real_in + (size_t)pr * (size_t)(2 * NY), *sb = sa + NY;
#pragma unroll
                    for (int q = 0; q < 16; ++q) {
                        const int pt = 2 * (t + q * G) + sub;
                        v[q] = mk(v[q].x + __ldg(sa + pt), v[q].y + __ldg(sb + pt));
                    }
                }
                if (sub == 0) {
                    // the even points wait in tensor memory while the odd points are transformed back
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        cpx a[8];
#pragma unroll
                        for (int q = 0; q < 8; ++q) a[q] = v[8 * h + q];
                        tmem_park8(pk0 + 16 * h, a);
                    }
                }
            }
        }
        if (f != 3) continue;

        // ---- forward transform of z = J_a + i J_b by decimation in time; v holds the odd points
        const cpx wl = launder(wt);
        line_fft<H, 1>(v, F, t, 0, tw, bar);                            // O
        {
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                cpx a[8];
#pragma unroll
                for (int q = 0; q < 8; ++q) a[q] = cmul(v[8 * h + q], (8 * h + q == 0) ? wl : cmul(wl, w32(8 * h + q)));   // W^k O
                tmem_park8(tp + 64u + 16 * h, a);
            }
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                cpx a[8];
                tmem_unpark8(tp + 16 * h, a);                           // the even points
#pragma unroll
                for (int q = 0; q < 8; ++q) v[8 * h + q] = a[q];
            }
        }
        line_fft<H, 1>(v, F, t, 0, tw, bar);                            // E
        // Zlo = E + W O (bins k), Zhi = E - W O (bins k + H); the mirror Z[NY - k] = Zhi[H - k] travels through F
        cpx zhi0;
        {
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                cpx a[8];
                tmem_unpark8(tp + 64u + 16 * h, a);
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    const cpx e = v[8 * h + q];
                    v[8 * h + q] = cadd(e, a[q]);
                    const cpx zh = csub(e, a[q]);
                    if (h == 0 && q == 0) zhi0 = zh;
                    F[padpos(t + (8 * h + q) * G)] = zh;
                }
            }
        }
        bar.sync();
        const int pr = (int)blockIdx.x + (n >> 2) * (int)gridDim.x;
        cpx *PBout = p.spec_out + (size_t)pr * (size_t)(2 * cw);
        int tl = t;
        asm volatile("" : "+r"(tl));
#pragma unroll
        for (int q = 0; q < 16; ++q) {
            const int k = tl + q * G;
            const cpx Z = v[q];
            // bin 0 mirrors itself (Z[NY] = Z[0])
            const cpx M = (q == 0 && tl == 0) ? Z : F[padpos(H - k)];
            float4 o;
            o.x = 0.5f * (Z.x + M.x);                                   // A = (Z + conj M) / 2
            o.y = 0.5f * (Z.y - M.y);
            o.z = 0.5f * (Z.y + M.y);                                   // B = (Z - conj M) / (2i)
            o.w = 0.5f * (M.x - Z.x);
            *reinterpret_cast<float4 *>(out_addr<DIST>(p, PBout, k)) = o;
        }
        if (tl == 0)                                                    // Nyquist bin H = Zhi[0] is its own mirror
            *reinterpret_cast<float4 *>(out_addr<DIST>(p, PBout, H)) = make_float4(zhi0.x, 0.f, zhi0.y, 0.f);
        for (int k = H + 1 + tl; k < p.pitch; k += G)
            *reinterpret_cast<float4 *>(out_addr<DIST>(p, PBout, k)) = make_float4(0.f, 0.f, 0.f, 0.f);
        bar.sync();                                                     // F is reused by the next pair's first transform
    }
    tmem_free_cta<C::TCOLS>(tbase);
}

}  // namespace xfb

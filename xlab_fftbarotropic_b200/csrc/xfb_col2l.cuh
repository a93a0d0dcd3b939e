// xfb_col2l.cuh -- K-COL of the stepper for columns of 16384 points: a TWO-LEVEL transform (2 x 8192 + one radix-2 stage
// in registers) that matches the pair layout of the exchange arrays piece for piece.
//
// Same fusion as colt_kernel<COL_STEP / COL_PRO> (reference loops main.cpp:148,237,240-243,246-251,286-312 and
// fftwfop.cpp:87-124).  Why a kernel of its own: a column of 16384 complex values is 128 KB -- a two-column TMA tile
// does not fit in shared memory, a one-column tile has 16-byte rows (the TMA engine then runs at a quarter of its
// rate), and the first-generation kernel (since removed) held two butterflies per thread (NX / 16 = 1024 butterflies on
// 512 threads): it spilled 280 bytes per thread and issued 8-byte accesses (profiles/r02_16384_gen1_ncu_full_summary.txt:
// 174 M local-memory sectors, 613 M global sectors for 335 M sectors of payload, stall_lg 2.9, 29 % issue slots used).
// Here a thread owns the rows {2m, 2m+1, 2m + NX/2 ... } that one 16-byte piece of the pair layout holds:
//   forward  (decimation in time):  E = FFT_{NX/2}(x[2n]), O = FFT_{NX/2}(x[2n+1])  -- the two rows of the piece (m = n);
//            X[k] = E[k] + W^k O[k], X[k + NX/2] = E[k] - W^k O[k]   (W = exp(-2 pi i / NX)): natural order, so the
//            tile-major state arrays z0 / zk / acc are read and written with fully used 256-byte warp accesses;
//   inverse  (decimation in frequency, swap trick): S[k] = Y[k] + Y[k + NX/2], D[k] = (Y[k] - Y[k + NX/2]) W^k;
//            y[2n] = FFT(S)[n], y[2n+1] = FFT(D)[n]  -- again the two rows of one piece: one 16-byte store.
// One butterfly per thread in every pass (no spills); the half that waits for its transform is parked in a
// thread-private shared-memory slot, the new stage state of the column in tensor memory (64 columns per thread).
// Persistent CTAs walk over the columns; the state blocks of the next column are pulled towards L2 while the current one
// is transformed.  What bounds it (profiles/r02_16384_*): a one-column tile moves 16-byte pieces, one 32-byte sector per
// lane -- 1280 fully divergent load/store instructions per column next to the shared-memory exchanges of ten 8192-point
// transforms in the same load/store unit.
#pragma once
#include <cuda.h>

#include "xfb_col.cuh"
#include "xfb_row.cuh"      // w32()

namespace xfb {

template <int NX>
struct Col2LCfg {
    static constexpr int H = NX / 2;
    static constexpr int G = H / 16;                    // threads: one butterfly of the half-length transform each
    static constexpr int THREADS = G;
    static constexpr int F_BYTES = LinePlan<H>::PADDED * (int)sizeof(cpx);
    static constexpr int PARK_BYTES = H * (int)sizeof(cpx);
    // the NEXT column of the tendency is streamed in through a ring of TMA boxes while the current one is transformed
    static constexpr int BOXR = (G >= 256) ? 256 : G;                 // row pairs per TMA box (a box row = one 16-byte piece)
    static constexpr int NB = G / BOXR;                              // boxes per ring slot: a slot = one piece of every thread
    static constexpr int SLOT_BYTES = G * 16;
    static constexpr int RING_SLOTS = 3;
    static constexpr int SMEM = F_BYTES + PARK_BYTES + RING_SLOTS * SLOT_BYTES + 128;      // + alignment slack
    static constexpr int TCOLS = (THREADS / 128) * 128;               // per thread: 64 columns of stage state + 64 of incoming column
    static_assert(THREADS % 128 == 0 && THREADS <= 512, "col2l: NX / 32 threads, whole groups of four warps");
};

// exp(-2 pi i (t + k G) / NX) = wt * exp(-2 pi i k / 32)   (G = NX / 32)
__device__ __forceinline__ cpx col2l_tw(const cpx wt, const int k) { return (k == 0) ? wt : cmul(wt, w32(k)); }

// Streaming of the next column into tensor memory.  Ring slot q of a column = pieces [q G, q G + G): exactly ONE piece
// (rows 2m, 2m+1) of every thread, its k = q.  The hook of col_fft calls step() at two barrier-separated points of each of
// the eight inverse transforms of a column = 16 points: thread 0 issues the TMA loads of slot q + 2 into the buffer slot
// q - 1 left, every thread waits for slot q and copies its piece into its TMEM lane (E[q] and O[q]).  A one-column tile
// has 16-byte box rows -- the TMA engine's slow case (profiles/r01_probe_tma_tile.txt) -- but one column per ~80 us is
// 1 % of even that rate, it costs no load/store-unit time and no thread ever waits for it.
template <int NX>
struct Col2LRing {
    typedef Col2LCfg<NX> C;
    const CUtensorMap *map;
    unsigned char *ring;
    unsigned long long *bar;
    unsigned tin;         // this thread's incoming TMEM region: E[k] at + 2k, O[k] at + 32 + 2k
    int cx, cy;           // TMA coordinates of piece 0 of the column being streamed in
    int q;                // next slot of that column to consume; >= 16: nothing to do
    int slot;
    unsigned parity;

    __device__ __forceinline__ void issue(const int qq, const int sl) const      // thread 0
    {
        mbar_expect_tx(bar + sl, (unsigned)C::SLOT_BYTES);
#pragma unroll
        for (int b = 0; b < C::NB; ++b)
            tma_load_2d(ring + (size_t)sl * C::SLOT_BYTES + (size_t)b * C::BOXR * 16, map, cx, cy + qq * C::G + b * C::BOXR, bar + sl);
    }
    __device__ __forceinline__ void begin(const int x, const int y)
    {
        cx = x; cy = y; q = 0;
        if (threadIdx.x == 0) {
            issue(0, slot);
            issue(1, slot == 2 ? 0 : slot + 1);
        }
    }
    __device__ __forceinline__ void step()
    {
        if (q >= 16) return;
        if (threadIdx.x == 0 && q + 2 < 16) issue(q + 2, slot == 0 ? 2 : slot - 1);      // (slot + 2) mod 3
        mbar_wait(bar + slot, parity);
        const float4 x = *reinterpret_cast<const float4 *>(ring + (size_t)slot * C::SLOT_BYTES + (size_t)threadIdx.x * 16);
        tmem_park1(tin + (unsigned)(2 * q), mk(x.x, x.y));              // row 2m   -> E
        tmem_park1(tin + (unsigned)(32 + 2 * q), mk(x.z, x.w));         // row 2m+1 -> O
        ++q;
        if (slot == 2) { slot = 0; parity ^= 1u; } else ++slot;
    }
    __device__ __forceinline__ void operator()(const int e, const bool) { if (e < 2) step(); }
};

// LIN: COL_STEP with the linear terms of p.lin in the epilogue (a separate instance: the default one keeps its registers)
template <int NX, int MODE_, bool LIN = false>
__global__ void __launch_bounds__(Col2LCfg<NX>::THREADS, 1)
col2l_kernel(const ColParams p, const __grid_constant__ CUtensorMap jmap, const int ncols)
{
    typedef Col2LCfg<NX> C;
    static_assert(!LIN || MODE_ == COL_STEP, "the linear terms act on the vorticity step only");
    // the tracer modes are the stepper's modes with two products (i kx C, i ky C) instead of four
    constexpr bool TRACER = (MODE_ == COL_TSTEP || MODE_ == COL_TPRO);
    constexpr int MODE = (MODE_ == COL_TSTEP) ? COL_STEP : (MODE_ == COL_TPRO) ? COL_PRO : MODE_;
    // the ring needs the 16 hook points of EIGHT inverse transforms per column; the tracer step has four: its columns all
    // come with the burst of 16-byte loads (a half-streamed column would leave loads in flight behind the next begin())
    constexpr bool RING = !TRACER;
    constexpr int H = C::H, G = C::G;
    // TMA needs 128-byte aligned shared addresses: the declared alignment makes every offset below a link-time constant
    // (an alignment computed at run time costs registers that the transforms then spill)
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ unsigned tmem_slot;
    __shared__ unsigned long long ring_bar[C::RING_SLOTS];
    cpx *F = reinterpret_cast<cpx *>(smem_raw);
    cpx *park = reinterpret_cast<cpx *>(smem_raw + C::F_BYTES);      // park[k * G + t]: thread-private, conflict-free

    const int t = threadIdx.x;
    const int tt[1] = {t}, cc[1] = {0};
    LineTw<H> tw[1];
    tw[0].init(p.tw, p.twn, t);
    const cpx wt = __ldg(p.tw + (size_t)t * (p.twn / NX));
    if (t == 0) {
        for (int i = 0; i < C::RING_SLOTS; ++i) mbar_init(&ring_bar[i], 1);
        mbar_fence_init();
    }
    const unsigned tbase = tmem_alloc_cta<C::TCOLS>(&tmem_slot);       // includes a CTA barrier
    const int warp = t >> 5;
    const unsigned tkeep = tbase + ((unsigned)(32 * (warp & 3)) << 16) + (unsigned)((warp >> 2) * 128);  // lo: +0..31, hi: +32..63
    const size_t srow = (size_t)p.st_row_stride;                      // = tile width of the state arrays
    Col2LRing<NX> rs;
    rs.map = &jmap;
    rs.ring = smem_raw + C::F_BYTES + C::PARK_BYTES;
    rs.bar = ring_bar;
    rs.tin = tkeep + 64u;
    rs.slot = 0; rs.parity = 0; rs.q = 16; rs.cx = 0; rs.cy = 0;
    for (int col = blockIdx.x; col < ncols; col += gridDim.x) {
        const int member = col / p.pitch, jl = col - member * p.pitch;
        const size_t moff = (size_t)member * (size_t)p.member_stride;
        const int j = p.j_base + jl;
        const float ky = __ldg(p.ky + j);
        const float ky2 = ky * ky;
        // state arrays: element (row i, column jl) of the tile-major layout
        const size_t s0 = moff + (size_t)(jl / p.st_row_stride) * (size_t)p.st_tile_stride + (size_t)(jl % p.st_row_stride);
        // 16-byte piece m of this column in a pair-layout array: rows 2m and 2m+1
        const size_t piece0 = moff + (size_t)jl * 2;
        const size_t pstride = (size_t)p.pitch * 2;
        {
            // the epilogue operands of this CTA's NEXT column towards L2: with a tile width of one the column's block of
            // each state array is contiguous, three bulk prefetches.  (16384^2, per launch: 6.43 ms without, 5.42 ms with;
            // pulling the column's 8192 scattered 16-byte pieces of the tendency in as well -- one prefetch instruction
            // each -- costs more load/store-unit time than it saves: 5.46 ms.)
            const int nc = col + gridDim.x;
            if (nc < ncols && MODE == COL_STEP && p.st_row_stride == 1) {
                const int nm = nc / p.pitch, njl = nc - nm * p.pitch;
                const size_t ns0 = (size_t)nm * (size_t)p.member_stride + (size_t)njl * (size_t)p.st_tile_stride;
                constexpr unsigned bytes = NX * (unsigned)sizeof(cpx);
                if (t == 0) bulk_prefetch_l2(p.z0 + ns0, bytes);
                if (p.stage != 1) {
                    if (t == 32) bulk_prefetch_l2(p.zk + ns0, bytes);
                    if (t == 64) bulk_prefetch_l2(p.acc + ns0, bytes);
                }
            }
        }
        cpx v[1][16];

        if (MODE == COL_STEP) {
            // ------------------------------------------------------------ forward (decimation in time) + epilogue
            if (!RING || col == (int)blockIdx.x) {
                // the CTA's first column has nothing to hide a stream behind (a slab chunk may hold a single column per
                // CTA, and a one-column TMA box moves 16-byte rows at a crawl): its sixteen pieces come with one burst of
                // 16-byte loads and take the same way through tensor memory as the streamed columns
                const cpx *src = p.jint + piece0;
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    float4 x[8];
#pragma unroll
                    for (int q = 0; q < 8; ++q) x[q] = __ldg(reinterpret_cast<const float4 *>(src + (size_t)(t + (8 * h + q) * G) * pstride));
#pragma unroll
                    for (int q = 0; q < 8; ++q) {
                        tmem_park1(rs.tin + (unsigned)(2 * (8 * h + q)), mk(x[q].x, x[q].y));            // row 2m   -> E
                        tmem_park1(rs.tin + (unsigned)(32 + 2 * (8 * h + q)), mk(x[q].z, x[q].w));       // row 2m+1 -> O
                    }
                }
            }
#pragma unroll
            for (int h = 0; h < 2; ++h) {                    // E = the rows 2m of this thread's sixteen pieces
                cpx a[8];
                tmem_unpark8(rs.tin + (unsigned)(16 * h), a);
#pragma unroll
                for (int q = 0; q < 8; ++q) v[0][8 * h + q] = a[q];
            }
            col_fft<H, 1, 1>(v, F, tt, cc, tw);
#pragma unroll
            for (int k = 0; k < 16; ++k) park[k * G + t] = v[0][k];          // E waits in the slot
#pragma unroll
            for (int h = 0; h < 2; ++h) {                    // O = the rows 2m+1
                cpx a[8];
                tmem_unpark8(rs.tin + (unsigned)(32 + 16 * h), a);
#pragma unroll
                for (int q = 0; q < 8; ++q) v[0][8 * h + q] = a[q];
            }
            {
                // the incoming region is free: the next column of this CTA streams into it under the inverse transforms
                const int nc = col + gridDim.x;
                if (RING && nc < ncols) {
                    const int nm = nc / p.pitch, njl = nc - nm * p.pitch;
                    rs.begin(njl * 2, nm * (NX / 2));
                } else {
                    rs.q = 16;
                }
            }
            // epilogue operands (z0, zk, acc) travel in quarters of four rows, one quarter ahead of the arithmetic; the first
            // quarter is requested inside the second transform, before its last exchange
            cpx qz0[4], qzk[4], qac[4];
            auto load_quarter = [&](const int half, const int qd, cpx (&a0)[4], cpx (&ak)[4], cpx (&aa)[4]) {
                const size_t eq = s0 + (size_t)(t + half * H + 4 * qd * G) * srow;
#pragma unroll
                for (int q = 0; q < 4; ++q) a0[q] = p.z0[eq + (size_t)(q * G) * srow];
                if (p.stage != 1) {
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        ak[q] = p.zk[eq + (size_t)(q * G) * srow];
                        aa[q] = p.acc[eq + (size_t)(q * G) * srow];
                    }
                }
            };
            auto pre = [&]() { load_quarter(0, 0, qz0, qzk, qac); };
            ColFftNoHook nohook;
            col_fft<H, 1, 1, ColFftNoHook, decltype(pre)>(v, F, tt, cc, tw, false, nohook, pre);
            const cpx wl = launder(wt);
#pragma unroll
            for (int k = 0; k < 16; ++k) v[0][k] = cmul(v[0][k], col2l_tw(wl, k));      // W^(t + k G) O
            // epilogue: rows i = t + k G (X = E + W O) and i + H (X = E - W O)
#pragma unroll 1
            for (int half = 0; half < 2; ++half) {
                const size_t e0 = s0 + (size_t)(t + half * H) * srow;
                cpx znew[8];
#pragma unroll
                for (int qd = 0; qd < 4; ++qd) {
                    cpx nz0[4], nzk[4], nac[4];
                    if (qd < 3) load_quarter(half, qd + 1, nz0, nzk, nac);
                    else if (half == 0) load_quarter(1, 0, nz0, nzk, nac);
                    if (p.stage == 1) {
#pragma unroll
                        for (int q = 0; q < 4; ++q) { qzk[q] = qz0[q]; qac[q] = mk(0.f, 0.f); }
                    }
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const int k = 4 * qd + q;
                        const int i = t + k * G + half * H;
                        const size_t e = e0 + (size_t)(k * G) * srow;
                        const cpx E = park[k * G + t];
                        const cpx X = half ? csub(E, v[0][k]) : cadd(E, v[0][k]);
                        // signed x wavenumber index: i for i <= NX/2 (the Nyquist row keeps +, fftwfop.cpp:15-20), else i - NX
                        const int si = (i <= NX / 2) ? i : i - NX;
                        const float kxv = (float)si * p.kxscale;
                        const float lap = -fmaf(kxv, kxv, ky2);
                        // dvortdt_c += (vort_c * laplacian_coe) * NU                                  main.cpp:240-243
                        float tx = __fadd_rn(X.x, __fmul_rn(__fmul_rn(qzk[q].x, lap), p.nu));
                        float ty2 = __fadd_rn(X.y, __fmul_rn(__fmul_rn(qzk[q].y, lap), p.nu));
                        if constexpr (LIN) {                                 // + L(k) Z_k (DESIGN.md section 3)
                            const cpx l = lin_term(p.lin, kxv, -lap, qzk[q]);
                            tx = __fadd_rn(tx, l.x);
                            ty2 = __fadd_rn(ty2, l.y);
                        }
                        // dealiasing mask (fftwfop.cpp:57-68)
                        const int ii = (i <= NX / 2) ? i : NX - i;
                        const float m = (ii * ii + j * j >= p.mask_kd_i) ? 0.0f : 1.0f;
                        const float rx = __fmul_rn(tx, m), ry = __fmul_rn(ty2, m);
                        cpx zn;
                        if (p.stage == 4) {                                                          // main.cpp:309-312
                            zn.x = __fadd_rn(qz0[q].x, __fdiv_rn(__fmul_rn(__fadd_rn(qac[q].x, rx), p.dt), 6.0f));
                            zn.y = __fadd_rn(qz0[q].y, __fdiv_rn(__fmul_rn(__fadd_rn(qac[q].y, ry), p.dt), 6.0f));
                            p.z0[e] = zn;
                        } else {                                                                     // main.cpp:246-251
                            const cpx an = (p.stage == 1) ? mk(rx, ry)
                                                          : mk(__fadd_rn(qac[q].x, __fmul_rn(2.0f, rx)),
                                                               __fadd_rn(qac[q].y, __fmul_rn(2.0f, ry)));
                            p.acc[e] = an;
                            zn.x = __fadd_rn(qz0[q].x, __fmul_rn(rx, p.dt_stage));
                            zn.y = __fadd_rn(qz0[q].y, __fmul_rn(ry, p.dt_stage));
                            p.zk[e] = zn;
                        }
                        znew[(qd & 1) * 4 + q] = zn;
                    }
                    if (qd & 1) tmem_park8(tkeep + (unsigned)(half * 32 + (qd >> 1) * 16), znew);
#pragma unroll
                    for (int q = 0; q < 4; ++q) { qz0[q] = nz0[q]; qzk[q] = nzk[q]; qac[q] = nac[q]; }
                }
            }
        } else {
            // COL_PRO: the state of the step's start goes to tensor memory, the products below read it from there
#pragma unroll
            for (int half = 0; half < 2; ++half)
#pragma unroll
                for (int h8 = 0; h8 < 2; ++h8) {
                    cpx z[8];
#pragma unroll
                    for (int q = 0; q < 8; ++q) z[q] = p.z0[s0 + (size_t)(t + (8 * h8 + q) * G + half * H) * srow];
                    tmem_park8(tkeep + (unsigned)(half * 32 + h8 * 16), z);
                }
        }

        // ---------------------------------------------------------------- prologue of the next stage + 4 inverse
        // (decimation in frequency; inverse transforms by the swap trick: every value enters and leaves swapped)
#pragma unroll 1
        for (int f = 0; f < (TRACER ? 2 : 4); ++f) {
            const cpx wl = launder(wt);
            // the thread index is laundered per field: otherwise the sixteen 64-bit store addresses are hoisted out of
            // this loop and spilled
            int tl = t;
            asm volatile("" : "+r"(tl));
#pragma unroll
            for (int h4 = 0; h4 < 4; ++h4) {                 // four rows of each half at a time: 16 registers of state in flight
                cpx lo[4], hi[4];
                tmem_unpark4(tkeep + (unsigned)(h4 * 8), lo);
                tmem_unpark4(tkeep + (unsigned)(32 + h4 * 8), hi);
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int k = 4 * h4 + q;
                    const int i = t + k * G;                                   // row i and row i + H
                    // f = 0: i kx Z, 1: i ky Z, 2: i ky Psi (u before negation), 3: i kx Psi (v);
                    // Psi = Z / -(kx^2+ky^2), (0,0) entry divides by 1                 (fftwfop.cpp:43,112-117)
                    const float kxl = (float)i * p.kxscale;
                    const float kxh = (float)((i == 0) ? H : i - H) * p.kxscale;
                    float kl = (f == 0 || f == 3) ? kxl : ky, kh = (f == 0 || f == 3) ? kxh : ky;
                    if (f >= 2) {
                        const float ll = (i == 0 && j == 0) ? 1.0f : -fmaf(kxl, kxl, ky2);
                        const float lh = -fmaf(kxh, kxh, ky2);
                        kl = __fdividef(kl, ll);
                        kh = __fdividef(kh, lh);
                    }
                    const cpx a = mk(lo[q].x * kl, -lo[q].y * kl);              // swap(i kk z)
                    const cpx b = mk(hi[q].x * kh, -hi[q].y * kh);
                    v[0][k] = cadd(a, b);                                       // S
                    park[k * G + t] = cmul(csub(a, b), col2l_tw(wl, k));        // D, waits in the slot
                }
            }
            col_fft<H, 1, 1, Col2LRing<NX>>(v, F, tt, cc, tw, false, rs);
#pragma unroll
            for (int k = 0; k < 16; ++k) {                   // rows 2m into the slot, D out of it
                const cpx d = park[k * G + t];
                park[k * G + t] = v[0][k];
                v[0][k] = d;
            }
            col_fft<H, 1, 1, Col2LRing<NX>>(v, F, tt, cc, tw, false, rs);
            cpx *dst = p.t_out[f] + piece0;
            cpx *dself = p.self_out[f] + (size_t)jl * 2;
#pragma unroll
            for (int k = 0; k < 16; ++k) {
                const cpx e = park[k * G + t];
                // rows 2m, 2m+1 of piece m = t + k G, un-swapped; this rank's own row pairs (slab runs) skip the exchange
                const int m = tl + k * G;
                const unsigned ms = (unsigned)(m - p.self_piece0);
                float4 *o = reinterpret_cast<float4 *>(ms < (unsigned)p.self_pieces ? dself + (size_t)ms * pstride : dst + (size_t)m * pstride);
                *o = make_float4(e.y, e.x, v[0][k].y, v[0][k].x);
            }
        }
    }
    tmem_free_cta<C::TCOLS>(tbase);
}

}  // namespace xfb

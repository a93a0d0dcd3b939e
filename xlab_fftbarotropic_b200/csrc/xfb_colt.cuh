// xfb_colt.cuh -- K-COL of the stepper, second generation: persistent CTAs, every strided (transposed) access
// done by the TMA engine.
//
// The fusion of COL_STEP / COL_PRO listed in xfb_col.cuh (reference loops main.cpp:148,237,240-243,
// 246-251,286-312 and fftwfop.cpp:87-124), with this data movement:
//   * a tile is TW adjacent spectral columns x all NX rows.  In the pair layout of the exchange arrays a tile
//     row pair is one contiguous piece of TW*2 complex values (32 bytes for TW = 2: whole sectors), so a
//     tile is a 2-D TMA box {TW*2, NX/2}: cp.async.bulk.tensor.2d loads the y-transformed tendency into the
//     dense staging buffer S and stores the four x-inverse-transformed products from S.  No LDG/STG
//     instruction touches a strided array, the loads of the NEXT tile run under the current tile's tail
//     and the stores of field f run under the transform of field f+1.
//   * the transforms work on FW <= TW columns at a time in a separate Stockham buffer F.  At NX = 8192 a
//     two-column tile is transformed one column after the other (FW = 1): one butterfly per thread per pass
//     (no register spills), at the access granularity of two columns.
//   * CTAs are persistent (one per SM) and walk over tiles.
//   * NX = 8192 (one staging buffer only) uses TENSOR MEMORY for what shared memory and registers cannot hold:
//     the new stage state of both columns between the epilogue and the four products (TKEEP), and the NEXT tile,
//     streamed in through a three-slot ring of TMA boxes while the current tile's inverse transforms run (ColtRing,
//     hooked into col_fft between its exchanges).  All 512 TMEM columns of the SM are allocated by the CTA.
// State arrays z0 / zk / acc are tile-major with tile width FW (one column group = one contiguous block); a tile's
// blocks are pulled towards L2 with cp.async.bulk.prefetch.L2 at tile start.
#pragma once
#include <cuda.h>

#include "xfb_col.cuh"

// XFB_COLT_SWZ=0 at compile time builds the unswizzled tile staging (A/B: tools/ab_lib.py with XFB_LIB)
#ifndef XFB_COLT_SWZ
#define XFB_COLT_SWZ 1
#endif

namespace xfb {

template <int NX>
struct ColTCfg {
    // staged tile width / columns transformed together
    static constexpr int TW = (NX >= 4096) ? 2 : 4;
    static constexpr int FW = (NX >= 8192) ? 1 : TW;
    static constexpr int G = NX / 16;
    static constexpr int THREADS = G * FW;
    static constexpr int NG = TW / FW;                                   // column groups per tile
    static constexpr int BOXR = (NX / 2 >= 256) ? 256 : NX / 2;          // row pairs per TMA box
    static constexpr int NBOX = (NX / 2) / BOXR;
    static constexpr int S_BYTES = NX * TW * (int)sizeof(cpx);
    static constexpr int F_BYTES = LinePlan<NX>::PADDED * FW * (int)sizeof(cpx);
    // a second staging buffer for the incoming tendency tile where it fits (NX <= 4096): the next tile is then
    // fetched during the whole current tile.  At 8192 one buffer serves both directions (pulling the next tile
    // into L2 early -- prefetch.global.L2 or cp.async.bulk.prefetch.tensor -- was measured SLOWER: 0.96 vs 0.92 ms).
    static constexpr bool SPLIT_IN = (2 * S_BYTES + F_BYTES + 1024 <= 227 * 1024);
    // 8192: no room for a second staging buffer.  The NEXT tile is streamed in, box by box, through a small ring of
    // TMA boxes and parked in TENSOR MEMORY (each thread keeps the 2 x 16 values it will feed to the forward
    // transforms in its own TMEM lane) while the current tile's inverse transforms run; see ColtRing below.
#ifndef XFB_COLT_NO_RING
    static constexpr bool RING = !SPLIT_IN && (TW / FW == 2) && ((NX / 2) / BOXR == 16) && (G * FW == 512);
#else
    static constexpr bool RING = false;
#endif
    // FW == 1 with two-column tiles (8192): a warp's 8-byte accesses to a staged tile touch 16 of every 32 bytes -- row pair
    // p and row pair p + 4 share their shared-memory banks (2-way conflicts on every tile store and ring read, 8.4 M
    // extra wavefronts per launch).  The tiles are therefore staged with the TMA engine's 32-byte swizzle (address bit 4
    // ^= bit 7: the two 16-byte column chunks of a row pair trade places in every other group of four row pairs) and the
    // threads apply the same exchange to their column index: conflict-free, no extra instruction in the loops.
    static constexpr bool SWZ = (XFB_COLT_SWZ != 0) && (TW == 2) && (FW == 1);
    static constexpr int RING_SLOTS = 3;
    static constexpr int BOX_BYTES = BOXR * TW * 2 * (int)sizeof(cpx);
    static constexpr int SMEM = (SPLIT_IN ? 2 : 1) * S_BYTES + F_BYTES + (RING ? RING_SLOTS * BOX_BYTES : 0) + 1024;   // + alignment slack
    static constexpr int MINB = (THREADS >= 512) ? 1 : (THREADS >= 256) ? 2 : 4;
    // NG > 1 (8192): the new stage state of the tile's columns cannot stay in registers across the column groups; it
    // is parked in TENSOR MEMORY (each thread's own 32 columns per column group, tcgen05.st / tcgen05.ld) instead of
    // being re-read from global memory for each of the four products
    static constexpr int TCOLS = (THREADS / 128) * NG * 32;
    static_assert(RING_SLOTS == 3, "ColtRing counts modulo 3");
    static_assert(THREADS >= 32 && THREADS <= 512, "bad column-group size");
};

struct ColTMaps {
    CUtensorMap jint;
    CUtensorMap t[4];
};

// Streaming of the next tile into tensor memory (ColTCfg::RING).  Box q of a tile = row pairs [256 q, 256 q + 256) x TW
// columns = rows [512 q, 512 q + 512): exactly ONE row of every butterfly thread (its k = q).  The hook of col_fft
// calls step() at two barrier-separated points of each of the eight inverse transforms of a tile = 16 points:
//   thread 0 issues the TMA load of box q + 2 into the slot box q - 1 left (everyone read it before the last barrier),
//   every thread waits for box q and copies its two values (one per column) from the ring into its TMEM lane.
// Box counters run on over the tiles of the CTA (slot = counter mod 3, mbarrier parity = (counter / 3) & 1).
// Issuing earlier (three boxes at the start, the next box ahead of each field's bulk stores) was measured slower
// (0.821 vs 0.795 ms per launch): the loads then delay the stores the next transform has to wait for.
template <int NX>
struct ColtRing {
    typedef ColTCfg<NX> C;
    static constexpr int BOX_ELEMS = C::BOX_BYTES / (int)sizeof(cpx);
    const CUtensorMap *map;
    cpx *ring;
    unsigned long long *bar;
    int s_off;            // this thread's element of a box: ((t >> 1) * TW) * 2 + (t & 1), + 2 * column
    int c0_off;           // 2 * (shared-memory chunk of column 0): 0, or 2 where the 32-byte swizzle exchanges the columns
    unsigned tin;         // this thread's incoming TMEM region: + cg * 32 + 2 * q
    int cx, cy;           // TMA coordinates of box 0 of the tile being streamed in
    int q;                // next box of that tile to consume; >= 16: nothing to do
    int slot;             // ring slot of box q
    unsigned parity;      // mbarrier parity of that slot's current use

    __device__ __forceinline__ void issue(const int box, const int sl) const     // thread 0
    {
        mbar_expect_tx(bar + sl, (unsigned)C::BOX_BYTES);
        tma_load_2d(ring + (size_t)sl * BOX_ELEMS, map, cx, cy + box * C::BOXR, bar + sl);
    }
    // start streaming the tile at TMA coordinates (x, y): boxes 0 and 1 (their slots are free: barriers have passed
    // since the previous tile's last boxes were consumed)
    __device__ __forceinline__ void begin(const int x, const int y)
    {
        cx = x; cy = y; q = 0;
        if (threadIdx.x == 0) {
            issue(0, slot);
            issue(1, slot == 2 ? 0 : slot + 1);
        }
    }
    // right behind a CTA barrier that follows the previous step()
    __device__ __forceinline__ void step()
    {
        if (q >= 16) return;
        if (threadIdx.x == 0 && q + 2 < 16) issue(q + 2, slot == 0 ? 2 : slot - 1);      // (slot + 2) mod 3
        mbar_wait(bar + slot, parity);
        const cpx *src = ring + (size_t)slot * BOX_ELEMS + s_off;
        const cpx a = src[c0_off], b = src[2 - c0_off];
        tmem_park1(tin + (unsigned)(2 * q), a);
        tmem_park1(tin + (unsigned)(32 + 2 * q), b);
        ++q;
        if (slot == 2) { slot = 0; parity ^= 1u; } else ++slot;
    }
    __device__ __forceinline__ void operator()(const int e, const bool last)
    {
        if (e == 0 || last) step();
    }
};

// LIN: COL_STEP with the linear terms of p.lin in the epilogue (a separate instance: the default one keeps its registers)
template <int NX, int MODE_, bool LIN = false>
__global__ void __launch_bounds__(ColTCfg<NX>::THREADS, ColTCfg<NX>::MINB)
colt_kernel(const ColParams p, const __grid_constant__ ColTMaps maps, const int tiles_per_member, const int tiles_total)
{
    typedef ColTCfg<NX> C;
    static_assert(!LIN || MODE_ == COL_STEP, "the linear terms act on the vorticity step only");
    // the tracer modes are the stepper's modes with two products instead of four
    constexpr bool TRACER = (MODE_ == COL_TSTEP || MODE_ == COL_TPRO);
    constexpr int MODE = (MODE_ == COL_TSTEP) ? COL_STEP : (MODE_ == COL_TPRO) ? COL_PRO : MODE_;
    constexpr int G = C::G, TW = C::TW, FW = C::FW, NG = C::NG;
    constexpr bool KEEP = (NG == 1);
    constexpr bool TKEEP = (NG > 1) && (MODE == COL_STEP) && (C::THREADS % 128 == 0) && (C::TCOLS >= 32) && (C::TCOLS <= 512) &&
                           ((C::TCOLS & (C::TCOLS - 1)) == 0);
    extern __shared__ unsigned char smem_dyn[];
    // TMA needs 128-byte aligned shared addresses
    unsigned char *smem_raw = smem_dyn + ((1024 - (smem_u32(smem_dyn) & 1023)) & 1023);
    cpx *S = reinterpret_cast<cpx *>(smem_raw);                                   // outgoing products (and incoming tile if !SPLIT_IN)
    cpx *F = reinterpret_cast<cpx *>(smem_raw + C::S_BYTES);
    cpx *SI = C::SPLIT_IN ? reinterpret_cast<cpx *>(smem_raw + C::S_BYTES + C::F_BYTES) : S;   // incoming tendency tile
    constexpr bool TRING = C::RING && TKEEP && !TRACER;       // the tracer step has 4 inverse transforms: too few hook points
    constexpr int TMEM_COLS = TRING ? 512 : (TKEEP ? C::TCOLS : 32);
    __shared__ unsigned long long full;
    __shared__ unsigned long long ring_bar[C::RING_SLOTS];
    __shared__ unsigned tmem_slot;

    const int tid = threadIdx.x;
    int t[1], c[1];
    c[0] = tid % FW;
    t[0] = tid / FW;
    // NX = 8192 stepper: the forward transform leaves the tendency in the Split8192 order (two shared-memory exchanges instead
    // of three); the epilogue, the state-array accesses and the parked stage state follow that order and the inverse
    // transforms take it back to natural order for the staged tile
    constexpr bool SPLIT = (NX == 8192) && (MODE == COL_STEP || MODE == COL_PRO);
    LineTw<NX> tw[1];
    if constexpr (SPLIT) Split8192::init_tw(tw[0], p.tw, p.twn, t[0]);
    else tw[0].init(p.tw, p.twn, t[0]);
    if (tid == 0) {
        mbar_init(&full, 1);
        for (int i = 0; i < C::RING_SLOTS; ++i) mbar_init(&ring_bar[i], 1);
        mbar_fence_init();
    }
    __syncthreads();
    unsigned tbase = 0, tpark = 0;
    if (TKEEP) {
        tbase = tmem_alloc_cta<TMEM_COLS>(&tmem_slot);
        const int warp = tid >> 5;
        tpark = tbase + ((unsigned)(32 * (warp & 3)) << 16) + (unsigned)((warp >> 2) * (NG * 32));     // + cg * 32
    }
    ColtRing<NX> rs;
    if (TRING) {
        const int warp = tid >> 5;
        rs.map = &maps.jint;
        rs.ring = reinterpret_cast<cpx *>(smem_raw + C::S_BYTES + C::F_BYTES);
        rs.bar = ring_bar;
        rs.tin = tbase + ((unsigned)(32 * (warp & 3)) << 16) + 256u + (unsigned)((warp >> 2) * 64);
        rs.slot = 0; rs.parity = 0; rs.q = 16; rs.cx = 0; rs.cy = 0;
    }
    unsigned phase = 0;
    const size_t srow = (size_t)p.st_row_stride;

    // element (row i = t + k*G, tile column col) of S: ((i >> 1) * TW + col) * 2 + (i & 1); k-stride = G * TW
    const int s_base = ((t[0] >> 1) * TW) * 2 + (t[0] & 1);
    // 32-byte swizzle of the staged tiles (ColTCfg::SWZ): byte address bit 7 = bit 3 of the row
    const int swz = C::SWZ ? ((t[0] >> 3) & 1) : 0;
    if (TRING) { rs.s_off = s_base; rs.c0_off = 2 * swz; }

    constexpr bool HAS_FWD = (MODE == COL_STEP || MODE == COL_FWDT);
    constexpr bool PIPE_TAIL = (MODE == COL_STEP) && !C::SPLIT_IN && (C::NBOX > 1) && (C::NBOX <= 16) && !TRING;
    int tile = blockIdx.x;
    if (TRING && tile < tiles_total) {
        // the CTA's first tile: streamed into tensor memory with nothing to hide behind
        const int member = tile / tiles_per_member, tl = tile - member * tiles_per_member;
        rs.begin(tl * TW * 2, member * (NX / 2));
#pragma unroll 1
        for (int b = 0; b < 16; ++b) {
            rs.step();
            __syncthreads();
        }
    }
    if (HAS_FWD && !TRING && tile < tiles_total && tid == 0) {
        const int member = tile / tiles_per_member, tl = tile - member * tiles_per_member;
        mbar_expect_tx(&full, C::S_BYTES);
#pragma unroll 1
        for (int b = 0; b < C::NBOX; ++b)
            tma_load_2d(SI + (size_t)b * C::BOXR * TW * 2, &maps.jint, tl * TW * 2, member * (NX / 2) + b * C::BOXR, &full);
    }

    // ky of this thread's column in each column group of a tile, loaded a tile ahead: a __ldg right in front of its first
    // use -- behind the asm volatile statements of the tensor-memory traffic the compiler cannot hoist it over -- left its
    // whole L2 latency exposed with all warps waiting at the same point, ten times per tile at 8192 (4.4 % of the
    // kernel's stall samples on the first one alone, profiles/r02c_8192_*)
    float ky_n0 = 0.f, ky_n1 = 0.f;
    if (tile < tiles_total) {
        const int jn = p.j_base + (tile % tiles_per_member) * TW + c[0];
        ky_n0 = __ldg(p.ky + jn);
        if (NG > 1) ky_n1 = __ldg(p.ky + jn + FW);
    }
    for (; tile < tiles_total; tile += gridDim.x) {
        const int member = tile / tiles_per_member, tl = tile - member * tiles_per_member;
        const int j0 = tl * TW;
        const float ky_t0 = ky_n0, ky_t1 = ky_n1;
        if (tile + (int)gridDim.x < tiles_total) {
            const int jn = p.j_base + ((tile + (int)gridDim.x) % tiles_per_member) * TW + c[0];
            ky_n0 = __ldg(p.ky + jn);
            if (NG > 1) ky_n1 = __ldg(p.ky + jn + FW);
        }
        const size_t moff = (size_t)member * (size_t)p.member_stride;
        const int tmy = member * (NX / 2), tmx = tl * TW * 2;      // TMA coordinates of this tile
        cpx v[1][16];
        cpx zkeep[KEEP ? 16 : 1];

        // ------------------------------------------------------------------ forward + epilogue
        if (HAS_FWD) {
            // epilogue operands of this tile towards L2 (needed after the forward transform)
            if (MODE == COL_STEP) {
                // (the tile's blocks of the tile-major state arrays are contiguous: three bulk prefetches by three
                // threads; one prefetch.global.L2 per 128 bytes from every thread cost 5 % of the kernel at 8192)
                const size_t e = moff + (size_t)(tl * NG) * (size_t)p.st_tile_stride;
                constexpr unsigned bytes = NX * TW * (unsigned)sizeof(cpx);
                if (tid == 0) bulk_prefetch_l2(p.z0 + e, bytes);
                if (p.stage != 1) {
                    if (tid == 32) bulk_prefetch_l2(p.zk + e, bytes);
                    if (tid == 64) bulk_prefetch_l2(p.acc + e, bytes);
                }
            }
            if (!TRING) {
                mbar_wait(&full, phase);
                phase ^= 1;
            }
#pragma unroll 1
            for (int cg = 0; cg < NG; ++cg) {
                const int col = cg * FW + c[0];
                if (TRING) {
                    tmem_unpark(rs.tin + (unsigned)(cg * 32), v[0]);       // this tile was parked while the previous one ran
                } else {
                    const cpx *src = SI + s_base + 2 * (col ^ swz);
#pragma unroll
                    for (int k = 0; k < 16; ++k) v[0][k] = src[k * G * TW];
                }
                const int j = p.j_base + j0 + col;
                const float kyv = (NG == 1 || cg == 0) ? ky_t0 : ky_t1;
                const float ky2 = kyv * kyv;
                const size_t soff = moff + (size_t)(tl * NG + cg) * (size_t)p.st_tile_stride;
                const size_t e0 = soff + (size_t)slot_base<NX, SPLIT>(t[0]) * srow + c[0];
                // Epilogue operands (z0, zk, acc of this column group) in quarters of four rows.  The loads of the first
                // quarter are issued INSIDE the forward transform, right before its last exchange, so that their L2
                // latency passes under the exchange's two barriers and the final pass; the loads of quarter q + 1 are
                // issued before the arithmetic of quarter q.  Measured NEUTRAL against one batch of 24 loads per half after
                // the transform (8192^2: 0.785 vs 0.782 ms per launch, 4096^2: 0.153 both): the scoreboard samples of
                // profiles/r01f_8192_stall_segments.txt seg 9 are where the warps wait, not what bounds the tile -- ten
                // 8192-point transforms per tile (instruction issue + shared-memory exchange) do.
                cpx qz0[4], qzk[4], qac[4];
                auto pre = [&]() {
                    if (MODE == COL_STEP) {
#pragma unroll
                        for (int q = 0; q < 4; ++q) qz0[q] = p.z0[e0 + (size_t)slot_off<NX, SPLIT>(q) * srow];
                        if (p.stage != 1) {
#pragma unroll
                            for (int q = 0; q < 4; ++q) {
                                qzk[q] = p.zk[e0 + (size_t)slot_off<NX, SPLIT>(q) * srow];
                                qac[q] = p.acc[e0 + (size_t)slot_off<NX, SPLIT>(q) * srow];
                            }
                        }
                    }
                };
                ColFftNoHook nohook;
                if constexpr (SPLIT) fft8192_to_split<FW>(v[0], F, t[0], c[0], tw[0], CtaBar(), false, nohook, pre);
                else col_fft<NX, FW, 1, ColFftNoHook, decltype(pre)>(v, F, t, c, tw, false, nohook, pre);
                if (MODE == COL_FWDT) {
                    // plain forward transform of the tile into the tile-major state (xfb_set_vorticity: main.cpp:256)
#pragma unroll
                    for (int k = 0; k < 16; ++k) p.z0[e0 + (size_t)slot_off<NX, SPLIT>(k) * srow] = v[0][k];
                }
                cpx znew[TKEEP ? 8 : 1];
#pragma unroll
                for (int qd = 0; qd < (MODE == COL_FWDT ? 0 : 4); ++qd) {
                    cpx nz0[4], nzk[4], nac[4];
                    if (qd < 3) {
#pragma unroll
                        for (int q = 0; q < 4; ++q) nz0[q] = p.z0[e0 + (size_t)slot_off<NX, SPLIT>(4 * qd + 4 + q) * srow];
                        if (p.stage != 1) {
#pragma unroll
                            for (int q = 0; q < 4; ++q) {
                                nzk[q] = p.zk[e0 + (size_t)slot_off<NX, SPLIT>(4 * qd + 4 + q) * srow];
                                nac[q] = p.acc[e0 + (size_t)slot_off<NX, SPLIT>(4 * qd + 4 + q) * srow];
                            }
                        }
                    }
                    if (p.stage == 1) {
#pragma unroll
                        for (int q = 0; q < 4; ++q) { qzk[q] = qz0[q]; qac[q] = mk(0.f, 0.f); }
                    }
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const int k = 4 * qd + q;
                        const int i = slot_pos<NX, SPLIT>(t[0], k);
                        const size_t e = e0 + (size_t)slot_off<NX, SPLIT>(k) * srow;
                        const cpx X = v[0][k];
                        const float kxv = (float)signed_row<NX, SPLIT>(t[0], k) * p.kxscale;
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
                        if (KEEP) zkeep[k] = zn;
                        if (TKEEP) znew[(qd & 1) * 4 + q] = zn;
                    }
                    if (TKEEP && (qd & 1)) tmem_park8(tpark + (unsigned)(cg * 32 + (qd >> 1) * 16), reinterpret_cast<const cpx(&)[8]>(znew));
                    if (qd < 3) {
#pragma unroll
                        for (int q = 0; q < 4; ++q) { qz0[q] = nz0[q]; qzk[q] = nzk[q]; qac[q] = nac[q]; }
                    }
                }
            }
        }

        if (TRING) {
            // both columns have left the incoming TMEM region (the forward transforms' barriers are behind every
            // thread): stream the next tile of this CTA into it under the eight inverse transforms below
            const int nt = tile + gridDim.x;
            if (nt < tiles_total) {
                const int nm = nt / tiles_per_member, ntl = nt - nm * tiles_per_member;
                rs.begin(ntl * TW * 2, nm * (NX / 2));
            } else {
                rs.q = 16;
            }
        }
        if (HAS_FWD && C::SPLIT_IN) {
            // every thread has read SI (it is behind the forward transform's barriers): fetch the next tile now
            const int nt = tile + gridDim.x;
            if (nt < tiles_total && tid == 0) {
                const int nm = nt / tiles_per_member, ntl = nt - nm * tiles_per_member;
                mbar_expect_tx(&full, C::S_BYTES);
#pragma unroll 1
                for (int b = 0; b < C::NBOX; ++b)
                    tma_load_2d(SI + (size_t)b * C::BOXR * TW * 2, &maps.jint, ntl * TW * 2, nm * (NX / 2) + b * C::BOXR, &full);
            }
        }

        // ------------------------------------------------------------------ prologue of the next stage + 4 inverse
        const cpx *zsrc = (MODE == COL_PRO || MODE == COL_DIAG || p.stage == 4) ? p.z0 : p.zk;
        const int NF = (MODE == COL_FWDT) ? 0 : (MODE == COL_DIAG) ? p.nfields : TRACER ? 2 : 4;
        if (KEEP && (MODE == COL_PRO || MODE == COL_DIAG)) {
            const size_t e0 = moff + (size_t)tl * (size_t)p.st_tile_stride + (size_t)slot_base<NX, SPLIT>(t[0]) * srow + c[0];
#pragma unroll
            for (int k = 0; k < 16; ++k) zkeep[k] = zsrc[e0 + (size_t)slot_off<NX, SPLIT>(k) * srow];
        }
#pragma unroll 1
        for (int f = 0; f < NF; ++f) {
#pragma unroll 1
            for (int cg = 0; cg < NG; ++cg) {
                const int col = cg * FW + c[0];
                const int j = p.j_base + j0 + col;
                const float ky = (NG == 1 || cg == 0) ? ky_t0 : ky_t1;
                const float ky2 = ky * ky;
                if (TKEEP) {
                    tmem_unpark(tpark + (unsigned)(cg * 32), v[0]);
                } else if (!KEEP) {
                    const size_t e0 =
                        moff + (size_t)(tl * NG + cg) * (size_t)p.st_tile_stride + (size_t)slot_base<NX, SPLIT>(t[0]) * srow + c[0];
#pragma unroll
                    for (int k = 0; k < 16; ++k) v[0][k] = zsrc[e0 + (size_t)slot_off<NX, SPLIT>(k) * srow];
                }
#pragma unroll
                for (int k = 0; k < 16; ++k) {
                    const int i = slot_pos<NX, SPLIT>(t[0], k);
                    const cpx z = KEEP ? zkeep[k] : v[0][k];
                    const float kx = (float)signed_row<NX, SPLIT>(t[0], k) * p.kxscale;
                    if (MODE == COL_DIAG) {
                        // p.stage 0: psi_xy, psi_xx, psi_yy = (kx ky, kx^2, ky^2) Z / (kx^2+ky^2)   [(i kx)(i ky) Z/-(k^2) ...]
                        // p.stage 1: zeta, zeta_x, zeta_y   = (1, i kx, i ky) Z
                        if (p.stage == 0) {
                            const float k2 = (i == 0 && j == 0) ? 1.0f : fmaf(kx, kx, ky2);
                            const float num = (f == 0) ? kx * ky : (f == 1) ? kx * kx : ky2;
                            const float rr = __fdividef(num, k2);
                            v[0][k] = mk(z.y * rr, z.x * rr);            // swap(rr z)
                        } else if (p.stage == 1) {
                            if (f == 0) v[0][k] = mk(z.y, z.x);
                            else {
                                const float kk = (f == 1) ? kx : ky;
                                v[0][k] = mk(z.x * kk, -z.y * kk);       // swap(i kk z)
                            }
                        } else {
                            // one record field: 0 vort, 1 psi, 2 u (negated after the y pass), 3 v, 7 dvortdx, 8 dvortdy
                            const int w = p.stage - 2;
                            const float li = (i == 0 && j == 0) ? 1.0f : -fmaf(kx, kx, ky2);
                            if (w == 0) v[0][k] = mk(z.y, z.x);
                            else if (w == 1) {
                                const float rr = __fdividef(1.0f, li);
                                v[0][k] = mk(z.y * rr, z.x * rr);
                            } else {
                                float kk = (w == 3 || w == 7) ? kx : ky;
                                if (w == 2 || w == 3) kk = __fdividef(kk, li);
                                v[0][k] = mk(z.x * kk, -z.y * kk);
                            }
                        }
                        continue;
                    }
                    // f = 0: i kx Z, 1: i ky Z, 2: i ky Psi (u before negation), 3: i kx Psi (v);
                    // Psi = Z / -(kx^2+ky^2), (0,0) entry divides by 1                 (fftwfop.cpp:43,112-117)
                    float kk = (f == 0 || f == 3) ? kx : ky;
                    if (f >= 2) {
                        const float li = (i == 0 && j == 0) ? 1.0f : -fmaf(kx, kx, ky2);
                        kk = __fdividef(kk, li);
                    }
                    v[0][k] = mk(z.x * kk, -z.y * kk);       // swap(i kk z)
                }
                // S is about to be overwritten: the bulk store of the previous field (or tile) must have read it.
                // Thread 0 waits inside the transform, before its last exchange barrier (col_fft, drain_tma).
                if constexpr (SPLIT) {
                    ColFftNoHook nohook;
                    ColFftNoPre nopre;
                    if (TRING) fft8192_from_split<FW>(v[0], F, t[0], c[0], tw[0], CtaBar(), cg == 0, rs, nopre);
                    else fft8192_from_split<FW>(v[0], F, t[0], c[0], tw[0], CtaBar(), cg == 0, nohook, nopre);
                } else if (TRING) {
                    col_fft<NX, FW, 1, ColtRing<NX>>(v, F, t, c, tw, cg == 0, rs);
                } else {
                    col_fft<NX, FW, 1>(v, F, t, c, tw, cg == 0);
                }
                cpx *dst = S + s_base + 2 * (col ^ swz);
#pragma unroll
                for (int k = 0; k < 16; ++k) dst[k * G * TW] = cswap(v[0][k]);
            }
            fence_proxy_async();
            __syncthreads();
            if (tid == 0) {
                const CUtensorMap *mt = &maps.t[f];
                if (PIPE_TAIL && f == NF - 1) {
                    // last field of the tile: one bulk group per box, so that the next tile's boxes can be fetched as the
                    // store engine releases them (below)
#pragma unroll 1
                    for (int b = 0; b < C::NBOX; ++b) {
                        tma_store_2d(mt, tmx, tmy + b * C::BOXR, S + (size_t)b * C::BOXR * TW * 2);
                        tma_commit();
                    }
                } else {
#pragma unroll 1
                    for (int b = 0; b < C::NBOX; ++b) tma_store_2d(mt, tmx, tmy + b * C::BOXR, S + (size_t)b * C::BOXR * TW * 2);
                    tma_commit();
                }
            }
        }

        // single staging buffer: next tile's tendency into S as soon as the last store has read it
        if (HAS_FWD && !C::SPLIT_IN && !TRING) {
            const int nt = tile + gridDim.x;
            if (nt < tiles_total && tid == 0) {
                const int nm = nt / tiles_per_member, ntl = nt - nm * tiles_per_member;
                mbar_expect_tx(&full, C::S_BYTES);
                if (PIPE_TAIL) {
                    // box b of the incoming tile as soon as the store of box b (bulk group b of the last NBOX) has read it
#pragma unroll
                    for (int b = 0; b < C::NBOX; ++b) {
                        tma_wait_read_n(C::NBOX - 1 - b);
                        tma_load_2d(S + (size_t)b * C::BOXR * TW * 2, &maps.jint, ntl * TW * 2, nm * (NX / 2) + b * C::BOXR, &full);
                    }
                } else {
                    tma_wait_read_all();
#pragma unroll 1
                    for (int b = 0; b < C::NBOX; ++b)
                        tma_load_2d(S + (size_t)b * C::BOXR * TW * 2, &maps.jint, ntl * TW * 2, nm * (NX / 2) + b * C::BOXR, &full);
                }
            }
        }
    }
    if (tid == 0) tma_wait_all();
    if (TKEEP) tmem_free_cta<TMEM_COLS>(tbase);
}

}  // namespace xfb

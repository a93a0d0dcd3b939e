// xfb_col.cu -- instantiations and launcher of the K-COL kernels.
#include "xfb_internal.h"
#include "xfb_colt.cuh"
#include "xfb_col2l.cuh"

namespace xfb {

#include <cstdlib>

static int env_int(const char *name, int dflt)
{
    const char *e = getenv(name);
    return e ? atoi(e) : dflt;
}

// Tile width of the K-COL-private state arrays (z0 / zk / acc are tile-major, one column group per block) = the
// number of columns the stepper transforms together: ColTCfg<NX>::FW (1 at 8192: a staged two-column tile is
// transformed one column at a time); 16384 runs the two-level kernel with one column per CTA.
int col_tile_width(int nx)
{
    switch (nx) {
    case 256: case 512: case 1024: case 2048: return 4;
    case 4096: return 2;
    case 8192: return 1;
    case 16384: return 1;
    default: return 0;
    }
}

// the stepper's K-COL on the two-level kernel: always at 16384; XFB_COL_2L=1 also puts 4096-point columns on it (a test
// knob that checks the 16384 kernel against colt_kernel)
bool col_two_level(int nx)
{
    static const bool at_4096 = env_int("XFB_COL_2L", 0) == 1;
    return nx == 16384 || (nx == 4096 && at_4096);
}

// ---- tensor maps for the TMA tiles of colt_kernel ------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_tiled()
{
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void *f = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) == cudaSuccess) fn = (EncodeTiledFn)f;
    }
    return fn;
}

// pair-layout array of `rows` rows x `pitch` complex columns as a 2-D tensor of 8-byte elements:
// inner dimension 2*pitch (column-major within a row pair: x = 2*j + (i & 1)), outer dimension rows/2
static int make_pair_map(CUtensorMap *m, const void *base, long long rows, int pitch, int tw, int boxr, bool swizzle32 = false)
{
    EncodeTiledFn enc = encode_tiled();
    if (!enc) return (int)cudaErrorNotSupported;
    cuuint64_t dims[2] = {(cuuint64_t)pitch * 2, (cuuint64_t)(rows / 2)};
    cuuint64_t strides[1] = {(cuuint64_t)pitch * 2 * sizeof(cpx)};
    cuuint32_t box[2] = {(cuuint32_t)(tw * 2), (cuuint32_t)boxr};
    cuuint32_t es[2] = {1, 1};
    CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, const_cast<void *>(base), dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle32 ? CU_TENSOR_MAP_SWIZZLE_32B : CU_TENSOR_MAP_SWIZZLE_NONE,
                     CU_TENSOR_MAP_L2_PROMOTION_NONE,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? 0 : (int)cudaErrorInvalidValue;
}

template <int NX, int MODE, bool LIN = false>
static int launch_colt_t(const ColParams &p, int batch, cudaStream_t st)
{
    typedef ColTCfg<NX> C;
    static PerDeviceInt cfg;
    int err = 0;
    const int resident = cfg.get([&](int *e) { return resident_ctas(colt_kernel<NX, MODE, LIN>, C::THREADS, C::SMEM, 0, e); }, &err);
    if (resident <= 0) return err;
    ColTMaps maps;
    const long long rows = (long long)NX * batch;
    if (MODE == COL_STEP || MODE == COL_FWDT || MODE == COL_TSTEP) {
        if (int e = make_pair_map(&maps.jint, p.jint, rows, p.pitch, C::TW, C::BOXR, C::SWZ)) return e;
    } else {
        maps.jint = CUtensorMap();
    }
    const int nout = (MODE == COL_FWDT) ? 0 : (MODE == COL_DIAG) ? p.nfields : (MODE == COL_TSTEP || MODE == COL_TPRO) ? 2 : 4;
    for (int f = 0; f < 4; ++f) {
        if (f < nout) {
            if (int e = make_pair_map(&maps.t[f], p.t_out[f], rows, p.pitch, C::TW, C::BOXR, C::SWZ)) return e;
        } else {
            maps.t[f] = (f > 0 && nout > 0) ? maps.t[0] : CUtensorMap();
        }
    }
    const int tiles_per_member = p.pitch / C::TW, tiles_total = tiles_per_member * batch;
    const int blocks = tiles_total < resident ? tiles_total : resident;
    colt_kernel<NX, MODE, LIN><<<blocks, C::THREADS, C::SMEM, st>>>(p, maps, tiles_per_member, tiles_total);
    return (int)cudaGetLastError();
}

// two-level K-COL (xfb_col2l.cuh): columns of 16384 points (and 4096 under XFB_COL_2L=1, a test knob)
template <int NX, int MODE, bool LIN = false>
static int launch_col2l_t(const ColParams &p, int batch, cudaStream_t st)
{
    typedef Col2LCfg<NX> C;
    static PerDeviceInt cfg;
    int err = 0;
    const int resident = cfg.get([&](int *e) { return resident_ctas(col2l_kernel<NX, MODE, LIN>, C::THREADS, C::SMEM, C::TCOLS, e); }, &err);
    if (resident <= 0) return err;
    CUtensorMap jmap = CUtensorMap();
    if (MODE == COL_STEP || MODE == COL_TSTEP)      // one-column boxes of the tendency: 2 elements (one 16-byte piece) x BOXR row pairs
        if (int e = make_pair_map(&jmap, p.jint, (long long)NX * batch, p.pitch, 1, C::BOXR)) return e;
    const int ncols = p.pitch * batch;
    int blocks = ncols < resident ? ncols : resident;
    // slab runs with the SM push kernel: a persistent grid on every SM would keep the push CTAs of the previous chunk
    // waiting until this launch ends; a few SMs are left to them (XFB_SLAB_SPARE_SMS)
    static const int spare = env_int("XFB_SLAB_SPARE_SMS", 8);      // 2 GPUs, 16384^2: 0 -> 19.25, 8 -> 18.72, 16 -> 18.89, 32 -> 20.58 ms per step
    if (p.self_pieces > 0 && resident > 2 * spare) {
        // ... unless that costs a whole extra wave of columns (8 GPUs: 132 columns per chunk on 140 CTAs is one wave, on
        // 124 it is two -- 5.8 -> 7.9 ms per step)
        const int fewer = resident - spare;
        if ((ncols + fewer - 1) / fewer == (ncols + resident - 1) / resident) blocks = ncols < fewer ? ncols : fewer;
    }
    col2l_kernel<NX, MODE, LIN><<<blocks, C::THREADS, C::SMEM, st>>>(p, jmap, ncols);
    return (int)cudaGetLastError();
}

template <int NX>
static int launch_colt_n(int mode, const ColParams &p, int batch, cudaStream_t st)
{
    if (mode == COL_DIAG) return launch_colt_t<NX, COL_DIAG>(p, batch, st);
    if (mode == COL_FWDT) return launch_colt_t<NX, COL_FWDT>(p, batch, st);
    if (mode == COL_TSTEP) return launch_colt_t<NX, COL_TSTEP>(p, batch, st);
    if (mode == COL_TPRO) return launch_colt_t<NX, COL_TPRO>(p, batch, st);
    if (mode == COL_STEP) return p.lin.on ? launch_colt_t<NX, COL_STEP, true>(p, batch, st) : launch_colt_t<NX, COL_STEP>(p, batch, st);
    return launch_colt_t<NX, COL_PRO>(p, batch, st);
}

template <int NX, int W, int MODE>
static int launch_col_t(const ColParams &p, int batch, cudaStream_t st)
{
    typedef ColCfg<NX, W> C;
    static PerDeviceInt cfg;
    int err = 0;
    if (cfg.get([&](int *e) { return resident_ctas(col_kernel<NX, W, MODE>, C::THREADS, C::SMEM, 0, e); }, &err) <= 0) return err;
    dim3 grid(p.pitch / W, batch);
    col_kernel<NX, W, MODE><<<grid, C::THREADS, C::SMEM, st>>>(p);
    return (int)cudaGetLastError();
}

template <int NX, int W>
static int launch_col_n(int mode, const ColParams &p, int batch, cudaStream_t st)
{
    return mode == COL_FWD ? launch_col_t<NX, W, COL_FWD>(p, batch, st) : launch_col_t<NX, W, COL_INV>(p, batch, st);
}

int launch_col(int nx, int mode, const ColParams &p, int batch, cudaStream_t st)
{
    // the operator tier's plain transforms
    if (mode == COL_FWD || mode == COL_INV) {
        switch (nx) {
        case 256: return launch_col_n<256, 4>(mode, p, batch, st);
        case 512: return launch_col_n<512, 4>(mode, p, batch, st);
        case 1024: return launch_col_n<1024, 4>(mode, p, batch, st);
        case 2048: return launch_col_n<2048, 4>(mode, p, batch, st);
        case 4096: return launch_col_n<4096, 2>(mode, p, batch, st);
        case 8192: return launch_col_n<8192, 1>(mode, p, batch, st);
        case 16384: return launch_col_n<16384, 1>(mode, p, batch, st);
        }
        return (int)cudaErrorInvalidValue;
    }
    // the stepper's modes: two-level kernel on 16384-point columns, TMA-staged persistent kernel on shorter ones;
    // COL_STEP with a non-zero linear term (p.lin.on, xfb_set_linear_terms) runs the LIN instance of the same kernel
    if ((mode == COL_STEP || mode == COL_PRO) && col_two_level(nx)) {
        const bool lin = (mode == COL_STEP) && p.lin.on;
        if (nx == 16384) {
            if (lin) return launch_col2l_t<16384, COL_STEP, true>(p, batch, st);
            return mode == COL_STEP ? launch_col2l_t<16384, COL_STEP>(p, batch, st) : launch_col2l_t<16384, COL_PRO>(p, batch, st);
        }
        if (lin) return launch_col2l_t<4096, COL_STEP, true>(p, batch, st);
        return mode == COL_STEP ? launch_col2l_t<4096, COL_STEP>(p, batch, st) : launch_col2l_t<4096, COL_PRO>(p, batch, st);
    }
    if (nx == 16384) {      // passive tracer on the 16384 grid; the diagnostics modes have no 16384 kernel
        if (mode == COL_TSTEP || mode == COL_TPRO)
            return mode == COL_TSTEP ? launch_col2l_t<16384, COL_TSTEP>(p, batch, st) : launch_col2l_t<16384, COL_TPRO>(p, batch, st);
        return (int)cudaErrorNotSupported;
    }
    switch (nx) {
    case 256: return launch_colt_n<256>(mode, p, batch, st);
    case 512: return launch_colt_n<512>(mode, p, batch, st);
    case 1024: return launch_colt_n<1024>(mode, p, batch, st);
    case 2048: return launch_colt_n<2048>(mode, p, batch, st);
    case 4096: return launch_colt_n<4096>(mode, p, batch, st);
    case 8192: return launch_colt_n<8192>(mode, p, batch, st);
    }
    return (int)cudaErrorInvalidValue;
}

}  // namespace xfb

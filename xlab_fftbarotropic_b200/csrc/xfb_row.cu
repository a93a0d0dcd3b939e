// xfb_row.cu -- instantiations and launcher of the K-ROW kernels.
#include "xfb_internal.h"
#include "xfb_rowpair.cuh"
#include "xfb_rowpair2l.cuh"

#include <cstdlib>

namespace xfb {

bool row_size_ok(int ny)
{
    switch (ny) {
    case 256: case 512: case 1024: case 2048: case 4096: case 8192: case 16384: return true;
    default: return false;
    }
}

template <int NY, int MODE, bool DIST>
static int launch_row_t(const RowParams &p, cudaStream_t st)
{
    typedef RowCfg<NY> C;
    static PerDeviceInt cfg;
    int err = 0;
    if (cfg.get([&](int *e) { return resident_ctas(row_kernel<NY, MODE, DIST>, C::THREADS, C::SMEM, 0, e); }, &err) <= 0) return err;
    const int blocks = (p.nrows + C::LPC - 1) / C::LPC;
    row_kernel<NY, MODE, DIST><<<blocks, C::THREADS, C::SMEM, st>>>(p);
    return (int)cudaGetLastError();
}

// NY <= 8192: both rows of a pair as one complex line (xfb_rowpair.cuh)
template <int NY, int MODE, bool DIST>
static int launch_pair_t(const RowParams &p, cudaStream_t st)
{
    typedef PairCfg<NY> C;
    constexpr int smem = (MODE == ROW_JAC || MODE == ROW_DIAG) ? C::SMEM_JAC : C::SMEM;
    static PerDeviceInt cfg;
    int err = 0;
    const int resident = cfg.get([&](int *e) { return resident_ctas(rowpair_kernel<NY, MODE, DIST>, C::THREADS, smem, 0, e); }, &err);
    if (resident <= 0) return err;
    const int npairs = p.nrows / 2;
    int blocks = (npairs + C::PPC - 1) / C::PPC;
    // persistent: as many CTAs as are resident at once, each walks over pair groups
    if ((MODE == ROW_JAC || MODE == ROW_DIAG) && !DIST && blocks > resident) blocks = resident;
    rowpair_kernel<NY, MODE, DIST><<<blocks, C::THREADS, smem, st>>>(p);
    return (int)cudaGetLastError();
}

// ROW_JAC with the parked products in TENSOR MEMORY and double-buffered staging.  Default at NY >= 4096 (per launch:
// 8192^2 0.496 vs 0.58 ms, 4096^2 0.122 vs 0.126 ms); at 2048 and below several CTAs per SM already hide the fetches and
// the shared-memory parks are faster (2048^2: 0.037 vs 0.042 ms).  XFB_ROW_TMEM=0 / 1 forces either kernel (A/B knob).
// The first version moved 32 registers per tcgen05.ld / st and spilled 300 bytes per thread (0.62 ms at 8192^2); halves
// of 16 registers, a laundered thread index and one flat loop over the fetches brought it to zero spills.
template <int NY>
static int launch_pair_tmem(const RowParams &p, cudaStream_t st)
{
    typedef PairTCfg<NY> C;
    static PerDeviceInt cfg;
    int err = 0;
    const int resident = cfg.get([&](int *e) { return resident_ctas(rowpair_jac_tmem_kernel<NY>, C::THREADS, C::SMEM, C::TCOLS, e); }, &err);
    if (resident <= 0) return err;
    const int npairs = p.nrows / 2;
    int blocks = (npairs + C::PPC - 1) / C::PPC;
    if (blocks > resident) blocks = resident;
    rowpair_jac_tmem_kernel<NY><<<blocks, C::THREADS, C::SMEM, st>>>(p);
    return (int)cudaGetLastError();
}

// ROW_JAC for lines of 16384 points: two-level pair kernel (xfb_rowpair2l.cuh), TMA-staged and persistent.
template <int NY, bool DIST>
static int launch_pair2l(const RowParams &p, cudaStream_t st)
{
    typedef Pair2LCfg<NY> C;
    const int smem = C::smem_bytes(p.pitch);
    constexpr int SMEM_MAX = 226 * 1024;      // 227 KB per CTA minus the kernel's static shared memory
    if (smem > SMEM_MAX) return (int)cudaErrorInvalidValue;
    static PerDeviceInt cfg;
    int err = 0;
    // the shared-memory limit is raised to the hardware maximum once per device: the staging buffer follows the pitch
    const int resident = cfg.get([&](int *e) { return resident_ctas(rowpair2l_jac_kernel<NY, DIST>, C::THREADS, SMEM_MAX, C::TCOLS, e); }, &err);
    if (resident <= 0) return err;
    const int npairs = p.nrows / 2;
    const int blocks = npairs < resident ? npairs : resident;
    rowpair2l_jac_kernel<NY, DIST><<<blocks, C::THREADS, smem, st>>>(p);
    return (int)cudaGetLastError();
}

static bool use_tmem_parks(int ny)
{
    static const int forced = getenv("XFB_ROW_TMEM") ? (atoi(getenv("XFB_ROW_TMEM")) != 0 ? 1 : 0) : -1;
    return forced >= 0 ? forced == 1 : ny >= 4096;
}

// lines of up to 8192 points run on the pair kernels; 16384-point lines on the two-level kernel (JAC) and on
// row_kernel (the plain transforms)
template <int NY>
static int launch_row_n(int mode, const RowParams &p, cudaStream_t st)
{
    const bool dist = p.cw > 0;
    if constexpr (NY <= 8192) {
        switch (mode) {
        case ROW_R2C: return dist ? launch_pair_t<NY, ROW_R2C, true>(p, st) : launch_pair_t<NY, ROW_R2C, false>(p, st);
        case ROW_C2R: return dist ? launch_pair_t<NY, ROW_C2R, true>(p, st) : launch_pair_t<NY, ROW_C2R, false>(p, st);
        case ROW_JAC:
            if (!dist && use_tmem_parks(NY)) return launch_pair_tmem<NY>(p, st);
            return dist ? launch_pair_t<NY, ROW_JAC, true>(p, st) : launch_pair_t<NY, ROW_JAC, false>(p, st);
        case ROW_DIAG: return dist ? (int)cudaErrorInvalidValue : launch_pair_t<NY, ROW_DIAG, false>(p, st);
        }
    } else {
        switch (mode) {
        case ROW_R2C: return dist ? launch_row_t<NY, ROW_R2C, true>(p, st) : launch_row_t<NY, ROW_R2C, false>(p, st);
        case ROW_C2R: return dist ? launch_row_t<NY, ROW_C2R, true>(p, st) : launch_row_t<NY, ROW_C2R, false>(p, st);
        case ROW_JAC: return dist ? launch_pair2l<NY, true>(p, st) : launch_pair2l<NY, false>(p, st);
        }
    }
    return (int)cudaErrorInvalidValue;
}

int launch_row(int ny, int mode, const RowParams &p, cudaStream_t st)
{
    switch (ny) {
    case 256: return launch_row_n<256>(mode, p, st);
    case 512: return launch_row_n<512>(mode, p, st);
    case 1024: return launch_row_n<1024>(mode, p, st);
    case 2048: return launch_row_n<2048>(mode, p, st);
    case 4096: return launch_row_n<4096>(mode, p, st);
    case 8192: return launch_row_n<8192>(mode, p, st);
    case 16384: return launch_row_n<16384>(mode, p, st);
    }
    return (int)cudaErrorInvalidValue;
}

}  // namespace xfb

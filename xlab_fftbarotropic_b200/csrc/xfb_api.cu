// xfb_api.cu -- the C ABI declared in include/xfb.h: handle, tables, operator tier, stepper.
// No CPU fallback lives here: every entry point needs a CUDA device and says so when it fails.
#include <cfloat>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <vector>

#include "xfb_handle.h"

using namespace xfb;

// ------------------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";

int xfb::fail(int code, const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

extern "C" const char *xfb_last_error(void) { return g_err; }

cudaEvent_t xfb::next_event(std::vector<cudaEvent_t> *pool, size_t &used)
{
    if (used == pool->size()) {
        cudaEvent_t e;
        cudaEventCreate(&e);
        pool->push_back(e);
    }
    return (*pool)[used++];
}

int xfb::dev_alloc(void **p, size_t bytes)
{
    cudaError_t e = cudaMalloc(p, bytes);
    if (e != cudaSuccess) return fail(XFB_E_CUDA, "cudaMalloc(%zu): %s", bytes, cudaGetErrorString(e));
    return 0;
}

bool xfb::is_device_ptr(const void *p)
{
    cudaPointerAttributes a;
    cudaError_t e = cudaPointerGetAttributes(&a, p);
    if (e != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

extern "C" int xfb_size_supported(int nx, int ny)
{
    if (col_tile_width(nx) > 0 && row_size_ok(ny)) return 1;
    if (generic_size_ok(nx, ny)) return 2;
    return 0;
}

// ------------------------------------------------------------------------------------------------
// pointwise kernels (operator tier, layout conversion, physical-space helpers)
// ------------------------------------------------------------------------------------------------

struct PwParams {
    const cpx *in;
    cpx *out;
    int nx, in_pitch, out_pitch, ncols;   // ncols columns are processed; the rest of out's pitch is zeroed
    int in_tw, out_tw;                    // > 0: that side is in the stepper's tile-major layout, tile width tw
    int j_base;                           // global index of column 0 (slab runs)
    const float *kx, *ky;
    const double *kx2, *ky2;
    double mask_kd;
    int op;
};

// One thread per spectral element.  Same float expressions as fftwfop.cpp:87-124.
__global__ void pointwise_kernel(const PwParams p)
{
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long total = (long long)p.nx * p.out_pitch;
    if (idx >= total) return;
    const int i = (int)(idx / p.out_pitch), j = (int)(idx % p.out_pitch);
    const int jg = p.j_base + j;
    const size_t oidx = p.out_tw ? ((size_t)(j / p.out_tw) * p.nx + i) * p.out_tw + (j % p.out_tw) : (size_t)idx;
    if (j >= p.ncols) { p.out[oidx] = mk(0.f, 0.f); return; }
    const cpx z = p.in_tw ? p.in[((size_t)(j / p.in_tw) * p.nx + i) * p.in_tw + (j % p.in_tw)]
                          : p.in[(size_t)i * p.in_pitch + j];
    cpx r = z;
    switch (p.op) {
    case OP_GRADX: { const float k = p.kx[i]; r = mk(__fmul_rn(-z.y, k), __fmul_rn(z.x, k)); break; }
    case OP_GRADY: { const float k = p.ky[jg]; r = mk(__fmul_rn(-z.y, k), __fmul_rn(z.x, k)); break; }
    case OP_LAP: { const float l = lap_coe(p.kx2[i], p.ky2[jg]); r = mk(__fmul_rn(z.x, l), __fmul_rn(z.y, l)); break; }
    case OP_INVLAP: {
        const float l = (i == 0 && jg == 0) ? 1.0f : lap_coe(p.kx2[i], p.ky2[jg]);
        r = mk(__fdiv_rn(z.x, l), __fdiv_rn(z.y, l));
        break;
    }
    case OP_DEALIAS: {
        const long long ii = (i <= p.nx / 2) ? i : p.nx - i;
        const float m = ((double)(ii * ii + (long long)jg * jg) >= p.mask_kd) ? 0.0f : 1.0f;
        r = mk(__fmul_rn(z.x, m), __fmul_rn(z.y, m));
        break;
    }
    default: break;
    }
    p.out[oidx] = r;
}

// tables in the reference's H-sized form, for xfb_get_table (parity tests of fftwfop.cpp:40-68)
__global__ void table_kernel(float *out, int which, int nx, int hy, const double *kx2, const double *ky2, double kd)
{
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)nx * hy) return;
    const int i = (int)(idx / hy), j = (int)(idx % hy);
    if (which == XFB_TAB_MASK) {
        const long long ii = (i <= nx / 2) ? i : nx - i;
        out[idx] = ((double)(ii * ii + (long long)j * j) >= kd) ? 0.0f : 1.0f;
    } else {
        const float l = lap_coe(kx2[i], ky2[j]);
        out[idx] = (which == XFB_TAB_LAPINV && i == 0 && j == 0) ? 1.0f : l;
    }
}

int xfb::launch_pw(xfb_handle h, int op, const cpx *in, int in_pitch, cpx *out, int out_pitch, int ncols, int in_tw, int out_tw,
                   int chunk)
{
    PwParams p;
    p.in = in; p.out = out; p.nx = h->nx; p.in_pitch = in_pitch; p.out_pitch = out_pitch; p.ncols = ncols;
    p.in_tw = in_tw; p.out_tw = out_tw; p.j_base = h->col0 + chunk * h->pitch;
    p.kx = h->kx; p.ky = h->ky; p.kx2 = h->kx2; p.ky2 = h->ky2; p.mask_kd = h->mask_kd; p.op = op;
    const long long total = (long long)h->nx * out_pitch;
    const int threads = 256;
    pointwise_kernel<<<(unsigned)((total + threads - 1) / threads), threads, 0, h->stream>>>(p);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(XFB_E_CUDA, "pointwise_kernel: %s", cudaGetErrorString(e));
    h->launches++;
    return 0;
}

// ------------------------------------------------------------------------------------------------
// create / destroy
// ------------------------------------------------------------------------------------------------
extern "C" int xfb_slab_partition(int nx, int ny, int nranks, int nchunks, int rank, int *row0, int *rows, int *col0,
                                  int *cols, int *chunk_cols, int *pitch_global)
{
    if (nranks < 1 || rank < 0 || rank >= nranks) return fail(XFB_E_ARG, "xfb_slab_partition: bad rank %d of %d", rank, nranks);
    if (nchunks < 1 || nchunks > 16) return fail(XFB_E_ARG, "xfb_slab_partition: nchunks %d not in 1..16", nchunks);
    if (nx % (2 * nranks) != 0)
        return fail(XFB_E_SIZE, "xfb_slab_partition: nx=%d is not a multiple of 2 x %d ranks (row pairs stay on one rank)", nx, nranks);
    const int hy = ny / 2 + 1, panels = nranks * nchunks;
    int cw = (hy + panels - 1) / panels;
    cw = (cw + 3) / 4 * 4;                                  // whole column tiles, 32-byte aligned panels
    if (panels == 1) cw = ny / 2 + 4;
    if (row0) *row0 = rank * (nx / nranks);
    if (rows) *rows = nx / nranks;
    if (col0) *col0 = rank * nchunks * cw;
    if (cols) *cols = nchunks * cw;
    if (chunk_cols) *chunk_cols = cw;
    if (pitch_global) *pitch_global = cw * panels;
    return 0;
}

static int create_body(xfb_handle h, int size_class, int nx, int ny, float lx, float ly, float nu, int batch, int device, int rank,
                       int nranks, int nchunks);

int xfb::create_impl(xfb_handle *out, int nx, int ny, float lx, float ly, float nu, int batch, int device, int rank, int nranks,
                     int nchunks)
{
    if (!out) return fail(XFB_E_ARG, "xfb_create: null handle pointer");
    *out = nullptr;
    if (batch < 1) return fail(XFB_E_ARG, "xfb_create: batch must be >= 1");
    if (nranks > 1 && batch != 1) return fail(XFB_E_ARG, "slab handles hold one member");
    const int size_class = xfb_size_supported(nx, ny);
    if (!size_class)
        return fail(XFB_E_SIZE, "xfb_create: grid %dx%d not supported (fused kernels: powers of two 256..16384; generic path: "
                                "even sizes 2^a 3^b 5^c up to 4096)", nx, ny);
    if (size_class == 2 && nranks > 1) return fail(XFB_E_SIZE, "slab decomposition needs a power-of-two grid");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(XFB_E_CUDA, "xfb_create: no CUDA device (%s); this library has no CPU path",
                    e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
    if (device < 0 || device >= ndev) return fail(XFB_E_ARG, "xfb_create: device %d out of range (%d devices)", device, ndev);
    CK(cudaSetDevice(device));

    xfb_handle h = new (std::nothrow) xfb_handle_s();
    if (!h) return fail(XFB_E_ARG, "xfb_create: out of host memory");
    memset(h, 0, sizeof(*h));
    // every failure below releases what has been allocated so far (streams, events, device memory, the handle itself)
    if (int e2 = create_body(h, size_class, nx, ny, lx, ly, nu, batch, device, rank, nranks, nchunks)) {
        destroy_impl(h);
        return e2;
    }
    *out = h;
    return 0;
}

static int create_body(xfb_handle h, int size_class, int nx, int ny, float lx, float ly, float nu, int batch, int device, int rank,
                       int nranks, int nchunks)
{
    h->nx = nx; h->ny = ny; h->hy = ny / 2 + 1; h->batch = batch; h->device = device;
    h->lx = lx; h->ly = ly; h->nu = nu;
    h->tw_state = col_tile_width(nx);
    h->rank = rank; h->nranks = nranks; h->nchunks = nchunks;
    {
        int row0, cols;
        if (xfb_slab_partition(nx, ny, nranks, nchunks, rank, &row0, &h->rows, &h->col0, &cols, &h->pitch, &h->pitch_g))
            return XFB_E_SIZE;
        // k / cw by multiply-high: verified for every column index the kernels can form
        h->cw_magic = (unsigned)(((1ull << 32) + h->pitch - 1) / h->pitch);
        for (unsigned k = 0; k < (unsigned)h->pitch_g; ++k)
            if ((unsigned)(((unsigned long long)k * h->cw_magic) >> 32) != k / (unsigned)h->pitch)
                return fail(XFB_E_SIZE, "internal: magic division fails for k=%u cw=%d", k, h->pitch);
    }
    if (size_class == 2) {
        // generic path: reference layout everywhere -- no padding, and the state arrays are ROW-major (tw_state = 0):
        // a mixed grid such as 1024 x 768 has a fused-size nx but must not use the fused kernels' tile-major indexing
        h->pitch = h->pitch_g = h->hy;
        h->tw_state = 0;
    }
    // `pitch` is the pitch of the column-side arrays (one chunk of this rank's columns; all columns on one GPU)
    h->grids = (size_t)h->rows * ny; h->hgrids = (size_t)nx * h->hy; h->hpad = (size_t)nx * h->pitch * nchunks;
    CK(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));

    // master twiddle table exp(-2 pi i k / twn), float64 -> float32 once
    h->twn = nx > ny ? nx : ny;
    {
        std::vector<float2> tw(h->twn);
        for (int k = 0; k < h->twn; ++k) {
            const double a = -2.0 * M_PI * (double)k / (double)h->twn;
            tw[k] = make_float2((float)cos(a), (float)sin(a));
        }
        if (dev_alloc((void **)&h->tw, sizeof(float2) * h->twn)) return XFB_E_CUDA;
        CK(cudaMemcpy(h->tw, tw.data(), sizeof(float2) * h->twn, cudaMemcpyHostToDevice));
    }
    // wavenumber tables with the reference's float expressions (fftwfop.cpp:15-24, fftwfop.hpp:7)
    {
        const float TWOPI = acosf(-1.0f) * 2.0f;
        const int nky = h->pitch_g;
        std::vector<float> kx(nx), ky(nky);
        std::vector<double> kx2(nx), ky2(nky);
        for (int i = 0; i <= nx / 2; ++i) kx[i] = TWOPI * ((float)i) / lx;
        for (int i = nx / 2 + 1; i < nx; ++i) kx[i] = -kx[nx - i];
        for (int j = 0; j < nky; ++j) ky[j] = TWOPI * ((float)j) / ly;
        for (int i = 0; i < nx; ++i) kx2[i] = (double)kx[i] * (double)kx[i];
        for (int j = 0; j < nky; ++j) ky2[j] = (double)ky[j] * (double)ky[j];
        if (dev_alloc((void **)&h->kx, sizeof(float) * nx) || dev_alloc((void **)&h->ky, sizeof(float) * nky) ||
            dev_alloc((void **)&h->kx2, sizeof(double) * nx) || dev_alloc((void **)&h->ky2, sizeof(double) * nky))
            return XFB_E_CUDA;
        CK(cudaMemcpy(h->kx, kx.data(), sizeof(float) * nx, cudaMemcpyHostToDevice));
        CK(cudaMemcpy(h->ky, ky.data(), sizeof(float) * nky, cudaMemcpyHostToDevice));
        CK(cudaMemcpy(h->kx2, kx2.data(), sizeof(double) * nx, cudaMemcpyHostToDevice));
        CK(cudaMemcpy(h->ky2, ky2.data(), sizeof(double) * nky, cudaMemcpyHostToDevice));
        // fftwfop.cpp:11-12,57: ceil(((float)N)/3.0) squared and summed in double, stored as float
        const int dkx = (int)ceil(((float)nx) / 3.0), dky = (int)ceil(((float)ny) / 3.0);
        h->mask_kd = (double)(float)((double)dkx * dkx + (double)dky * dky);
    }
    const size_t sb = sizeof(cpx) * h->hpad * batch;
    cpx **state[] = {&h->z0, &h->zk, &h->acc, &h->jint};
    for (auto pp : state) {
        if (dev_alloc((void **)pp, sb)) return XFB_E_CUDA;
        CK(cudaMemsetAsync(*pp, 0, sb, h->stream));
    }
    // the four product arrays back to back (one 2-D copy moves a block of all four in the slab exchange)
    if (dev_alloc((void **)&h->t_block, 4 * sb)) return XFB_E_CUDA;
    CK(cudaMemsetAsync(h->t_block, 0, 4 * sb, h->stream));
    for (int f = 0; f < 4; ++f) h->t[f] = h->t_block + (size_t)f * h->hpad * batch;
    if (dev_alloc((void **)&h->real_a, sizeof(float) * h->grids) || dev_alloc((void **)&h->real_b, sizeof(float) * h->grids) ||
        dev_alloc((void **)&h->real_c, sizeof(float) * h->grids) ||
        dev_alloc((void **)&h->spec_a, sizeof(cpx) * h->hpad) || dev_alloc((void **)&h->spec_b, sizeof(cpx) * h->hpad))
        return XFB_E_CUDA;
    if (nranks == 1) {
        if (dev_alloc((void **)&h->ref_a, sizeof(cpx) * h->hgrids) || dev_alloc((void **)&h->ref_b, sizeof(cpx) * h->hgrids))
            return XFB_E_CUDA;
    }
    CK(cudaMemsetAsync(h->spec_a, 0, sizeof(cpx) * h->hpad, h->stream));
    CK(cudaMemsetAsync(h->spec_b, 0, sizeof(cpx) * h->hpad, h->stream));
    if (nranks > 1) {
        // receive arrays of both transposes in ONE allocation (one CUDA-IPC mapping per peer): the tendency, the four
        // products, and the same three arrays of the passive tracer (384 MB more per rank at 16384^2 on 8 GPUs)
        if (dev_alloc((void **)&h->recv_block, 8 * sb)) return XFB_E_CUDA;
        CK(cudaMemsetAsync(h->recv_block, 0, 8 * sb, h->stream));
        h->jint_recv = h->recv_block;
        for (int f = 0; f < 4; ++f) h->tr[f] = h->recv_block + (size_t)(1 + f) * h->hpad;
        h->cjint_recv = h->recv_block + (size_t)5 * h->hpad;
        for (int f = 0; f < 2; ++f) h->trc[f] = h->recv_block + (size_t)(6 + f) * h->hpad;
        if (dev_alloc((void **)&h->sync_buf, sizeof(float))) return XFB_E_CUDA;
        CK(cudaMemsetAsync(h->sync_buf, 0, sizeof(float), h->stream));
        {
            int lo = 0, hi = 0;
            CK(cudaDeviceGetStreamPriorityRange(&lo, &hi));
            CK(cudaStreamCreateWithPriority(&h->comm_stream, cudaStreamNonBlocking, hi));     // exchange work jumps the queue
        }
        h->ncopy = 1;     // measured: several copy streams are SLOWER when the SMs keep HBM busy (tools/probes/probe_p2p_copy.cu)
        if (const char *e = getenv("XFB_SLAB_COPY_STREAMS")) h->ncopy = atoi(e) < 1 ? 1 : (atoi(e) > 4 ? 4 : atoi(e));
        for (int i = 0; i < 4; ++i) {
            CK(cudaStreamCreateWithFlags(&h->copy_stream[i], cudaStreamNonBlocking));
            CK(cudaEventCreateWithFlags(&h->ev_copy[i], cudaEventDisableTiming));
        }
        CK(cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming));
        for (auto &ev : h->ev_chunk) CK(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
        for (auto &ev : h->ev_comm) CK(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    }
    if (size_class == 2 && generic_create(h)) return XFB_E_CUDA;
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

extern "C" int xfb_create(xfb_handle *out, int nx, int ny, float lx, float ly, float nu, int batch, int device)
{
    return create_impl(out, nx, ny, lx, ly, nu, batch, device, 0, 1, 1);
}

// the captured step bakes in dt, the source pointer, the tracer and the linear terms: a change of the last two drops it
static void drop_step_graph(xfb_handle h)
{
    if (h->step_graph) cudaGraphExecDestroy((cudaGraphExec_t)h->step_graph);
    h->step_graph = nullptr;
}

int xfb::destroy_impl(xfb_handle h)
{
    if (!h) return 0;
    cudaSetDevice(h->device);
    cudaStreamSynchronize(h->stream);
    if (h->comm_stream) cudaStreamSynchronize(h->comm_stream);
    generic_destroy(h);
    drop_step_graph(h);
    if (h->rec_stream) {
        cudaStreamSynchronize(h->rec_stream);
        for (int i = 0; i < XFB_NREC; ++i) {
            cudaEventDestroy(h->rec_ready[i]);
            cudaEventDestroy(h->rec_done[i]);
            if (h->rec_buf[i]) cudaFree(h->rec_buf[i]);
        }
        cudaStreamDestroy(h->rec_stream);
    }
    void *ptrs[] = {h->tw, h->kx, h->ky, h->kx2, h->ky2, h->z0, h->zk, h->acc, h->jint, h->t_block, h->src, h->dg, h->real_a,
                    h->real_b, h->real_c, h->spec_a, h->spec_b, h->ref_a, h->ref_b, h->recv_block, h->sync_buf, h->espec, h->bspec, h->c0, h->ck, h->cacc, h->cjint, h->tc[0], h->panel_base, h->panel_base_c};
    for (void *p : ptrs)
        if (p) cudaFree(p);
    for (auto pool : {h->ev_row, h->ev_col, h->ev_a2a})
        if (pool) {
            for (cudaEvent_t e : *pool) cudaEventDestroy(e);
            delete pool;
        }
    if (h->comm_stream) {
        for (auto ev : h->ev_chunk) cudaEventDestroy(ev);
        for (auto ev : h->ev_comm) cudaEventDestroy(ev);
        for (int i = 0; i < 4; ++i) {
            cudaStreamSynchronize(h->copy_stream[i]);
            cudaStreamDestroy(h->copy_stream[i]);
            cudaEventDestroy(h->ev_copy[i]);
        }
        cudaEventDestroy(h->ev_fork);
        cudaStreamDestroy(h->comm_stream);
    }
    if (h->stream) cudaStreamDestroy(h->stream);
    cudaGetLastError();          // a partially created handle (create failure) may have left harmless errors behind
    delete h;
    return 0;
}

extern "C" int xfb_destroy(xfb_handle h)
{
    if (!h) return 0;
    if (h->team) { dist_release(h); return 0; }
    return destroy_impl(h);
}

extern "C" int xfb_sync(xfb_handle h)
{
    if (!h) return fail(XFB_E_ARG, "null handle");
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

extern "C" int xfb_profile(xfb_handle h, int enable)
{
    if (!h) return fail(XFB_E_ARG, "null handle");
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    if (!h->ev_row) h->ev_row = new std::vector<cudaEvent_t>();
    if (!h->ev_col) h->ev_col = new std::vector<cudaEvent_t>();
    h->ev_row_used = h->ev_col_used = h->ev_a2a_used = 0;
    h->profiling = enable != 0;
    return 0;
}

extern "C" int xfb_profile_read(xfb_handle h, double *row_ms, long long *row_launches, double *col_ms, long long *col_launches)
{
    if (!h || !row_ms || !row_launches || !col_ms || !col_launches) return fail(XFB_E_ARG, "null argument");
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    *row_ms = *col_ms = 0.0;
    *row_launches = (long long)(h->ev_row_used / 2);
    *col_launches = (long long)(h->ev_col_used / 2);
    for (size_t i = 0; i + 1 < h->ev_row_used; i += 2) {
        float ms = 0.f;
        CK(cudaEventElapsedTime(&ms, (*h->ev_row)[i], (*h->ev_row)[i + 1]));
        *row_ms += ms;
    }
    for (size_t i = 0; i + 1 < h->ev_col_used; i += 2) {
        float ms = 0.f;
        CK(cudaEventElapsedTime(&ms, (*h->ev_col)[i], (*h->ev_col)[i + 1]));
        *col_ms += ms;
    }
    return 0;
}

extern "C" long long xfb_launch_count(xfb_handle h) { return h ? h->launches : 0; }
extern "C" void *xfb_stream(xfb_handle h) { return h ? (void *)h->stream : nullptr; }

// ------------------------------------------------------------------------------------------------
// staging helpers: bring a caller buffer to the device / back
// ------------------------------------------------------------------------------------------------
int xfb::stage_in(xfb_handle h, const void *user, void *dev_scratch, size_t bytes, const void **dev)
{
    if (is_device_ptr(user)) { *dev = user; return 0; }
    CK(cudaMemcpyAsync(dev_scratch, user, bytes, cudaMemcpyHostToDevice, h->stream));
    *dev = dev_scratch;
    return 0;
}

void *xfb::stage_out_target(const void *user, void *dev_scratch) { return is_device_ptr(user) ? (void *)user : dev_scratch; }

int xfb::stage_out(xfb_handle h, void *user, const void *dev, size_t bytes, bool wait)
{
    if ((const void *)user != dev) {
        CK(cudaMemcpyAsync(user, dev, bytes, cudaMemcpyDeviceToHost, h->stream));
        if (wait) CK(cudaStreamSynchronize(h->stream));
    }
    return 0;
}

// ------------------------------------------------------------------------------------------------
// operator tier
// ------------------------------------------------------------------------------------------------
#define NO_SLAB(h, what)                                                                                        \
    do {                                                                                                         \
        if ((h)->nranks > 1) return fail(XFB_E_STATE, what ": not available on a slab-decomposed handle");       \
    } while (0)

static int spectral_op(xfb_handle h, int op, const float *in, float *out)
{
    if (!h || !in || !out) return fail(XFB_E_ARG, "null argument");
    NO_SLAB(h, "spectral operator");
    CK(cudaSetDevice(h->device));
    const size_t bytes = sizeof(cpx) * h->hgrids;
    const void *din;
    if (stage_in(h, in, h->ref_a, bytes, &din)) return XFB_E_CUDA;
    void *dout = stage_out_target(out, h->ref_b);
    if (launch_pw(h, op, (const cpx *)din, h->hy, (cpx *)dout, h->hy, h->hy)) return XFB_E_CUDA;
    return stage_out(h, out, dout, bytes);
}

extern "C" int xfb_gradx(xfb_handle h, const float *in, float *out) { return spectral_op(h, OP_GRADX, in, out); }
extern "C" int xfb_grady(xfb_handle h, const float *in, float *out) { return spectral_op(h, OP_GRADY, in, out); }
extern "C" int xfb_laplacian(xfb_handle h, const float *in, float *out) { return spectral_op(h, OP_LAP, in, out); }
extern "C" int xfb_invert_laplacian(xfb_handle h, const float *in, float *out) { return spectral_op(h, OP_INVLAP, in, out); }
extern "C" int xfb_dealias(xfb_handle h, const float *in, float *out) { return spectral_op(h, OP_DEALIAS, in, out); }

extern "C" int xfb_get_table(xfb_handle h, int which, float *out)
{
    if (!h || !out) return fail(XFB_E_ARG, "null argument");
    NO_SLAB(h, "xfb_get_table");
    CK(cudaSetDevice(h->device));
    if (which == XFB_TAB_GRADX) { CK(cudaMemcpy(out, h->kx, sizeof(float) * h->nx, cudaMemcpyDeviceToHost)); return 0; }
    if (which == XFB_TAB_GRADY) { CK(cudaMemcpy(out, h->ky, sizeof(float) * h->hy, cudaMemcpyDeviceToHost)); return 0; }
    if (which < XFB_TAB_LAP || which > XFB_TAB_MASK) return fail(XFB_E_ARG, "xfb_get_table: bad table id %d", which);
    float *d = (float *)h->ref_a;
    const long long total = (long long)h->hgrids;
    table_kernel<<<(unsigned)((total + 255) / 256), 256, 0, h->stream>>>(d, which, h->nx, h->hy, h->kx2, h->ky2, h->mask_kd);
    CK(cudaGetLastError());
    h->launches++;
    CK(cudaMemcpyAsync(out, d, sizeof(float) * h->hgrids, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

// ---- 2-D transforms on device buffers ---------------------------------------------------------
void xfb::fill_row(xfb_handle h, RowParams &p, int nrows)
{
    memset(&p, 0, sizeof(p));
    p.tw = h->tw; p.twn = h->twn; p.nrows = nrows; p.pitch = h->pitch_g;
    p.scale = 1.0f / (float)((double)h->nx * (double)h->ny);
    if (h->nranks > 1) {
        p.cw = h->pitch; p.panel_stride = (long long)h->rows * h->pitch; p.cw_magic = h->cw_magic;
    }
}

void xfb::fill_col(xfb_handle h, ColParams &p, int chunk)
{
    memset(&p, 0, sizeof(p));
    p.tw = h->tw; p.twn = h->twn; p.kx = h->kx; p.ky = h->ky; p.kx2 = h->kx2; p.ky2 = h->ky2;
    p.pitch = h->pitch; p.member_stride = (long long)h->hpad; p.ny = h->ny; p.mask_kd = h->mask_kd; p.nu = h->nu;
    p.j_base = h->col0 + chunk * h->pitch;
    p.mask_kd_i = (int)h->mask_kd;
    p.st_tile_stride = col_tile_width(h->nx); p.st_row_stride = h->pitch;      // row-major unless the stepper says otherwise
    p.kxscale = (acosf(-1.0f) * 2.0f) / h->lx;
    p.lin = h->lin;
}

// real [nx][ny] (device) -> padded spectrum (device), via `tmp` (padded)
static int fwd2d(xfb_handle h, const float *real_in, cpx *tmp, cpx *spec_out)
{
    if (h->generic) return generic_fwd2d(h, real_in, tmp, spec_out);
    RowParams r; fill_row(h, r, h->nx);
    r.real_in = real_in; r.spec_out = tmp;
    CKL(h, launch_row(h->ny, ROW_R2C, r, h->stream));
    ColParams c; fill_col(h, c);
    c.jint = tmp; c.z0 = spec_out;
    CKL(h, launch_col(h->nx, COL_FWD, c, 1, h->stream));
    return 0;
}

// padded spectrum (device) -> real [nx][ny] (device), scaled by `scale`; spec_in is preserved
static int inv2d(xfb_handle h, const cpx *spec_in, cpx *tmp, float *real_out, float scale, int negate)
{
    if (h->generic) return generic_inv2d(h, spec_in, tmp, real_out, scale, negate);
    ColParams c; fill_col(h, c);
    c.inv_in = spec_in; c.t_out[0] = tmp;
    CKL(h, launch_col(h->nx, COL_INV, c, 1, h->stream));
    RowParams r; fill_row(h, r, h->nx);
    r.spec_in[0] = tmp; r.real_out = real_out; r.scale = scale; r.negate = negate;
    CKL(h, launch_row(h->ny, ROW_C2R, r, h->stream));
    return 0;
}

extern "C" int xfb_r2c(xfb_handle h, const float *real_in, float *spec_out)
{
    if (!h || !real_in || !spec_out) return fail(XFB_E_ARG, "null argument");
    NO_SLAB(h, "xfb_r2c");
    CK(cudaSetDevice(h->device));
    const void *din;
    if (stage_in(h, real_in, h->real_a, sizeof(float) * h->grids, &din)) return XFB_E_CUDA;
    if (fwd2d(h, (const float *)din, h->spec_a, h->spec_b)) return XFB_E_CUDA;
    void *dout = stage_out_target(spec_out, h->ref_a);
    if (launch_pw(h, OP_COPY, h->spec_b, h->pitch, (cpx *)dout, h->hy, h->hy)) return XFB_E_CUDA;
    return stage_out(h, spec_out, dout, sizeof(cpx) * h->hgrids);
}

extern "C" int xfb_c2r(xfb_handle h, const float *spec_in, float *real_out)
{
    if (!h || !spec_in || !real_out) return fail(XFB_E_ARG, "null argument");
    NO_SLAB(h, "xfb_c2r");
    CK(cudaSetDevice(h->device));
    const void *din;
    if (stage_in(h, spec_in, h->ref_a, sizeof(cpx) * h->hgrids, &din)) return XFB_E_CUDA;
    if (launch_pw(h, OP_COPY, (const cpx *)din, h->hy, h->spec_a, h->pitch, h->hy)) return XFB_E_CUDA;
    void *dout = stage_out_target(real_out, h->real_a);
    if (inv2d(h, h->spec_a, h->spec_b, (float *)dout, 1.0f, 0)) return XFB_E_CUDA;
    return stage_out(h, real_out, dout, sizeof(float) * h->grids);
}

// ------------------------------------------------------------------------------------------------
// stepper tier
// ------------------------------------------------------------------------------------------------
static bool fused_diag_ok(xfb_handle h);
static int fused_products(xfb_handle h, int member, int kind, int nfields, const cpx *state = nullptr);
static int fused_diag(xfb_handle h, int member, int kind, float *out0, float *out1, const cpx *state = nullptr);

static int check_member(xfb_handle h, int member)
{
    if (!h) return fail(XFB_E_ARG, "null handle");
    if (member < 0 || member >= h->batch) return fail(XFB_E_ARG, "member %d out of range [0,%d)", member, h->batch);
    return 0;
}

// physical field (device) -> tile-major spectral state array of one member: y pass (pair kernel) then the TMA-staged
// x pass straight into the state (main.cpp:256)
static int fused_forward_to_state(xfb_handle h, const float *din, cpx *state_member)
{
    RowParams r; fill_row(h, r, h->nx);
    r.real_in = din; r.spec_out = h->spec_a;
    CKL(h, launch_row(h->ny, ROW_R2C, r, h->stream));
    ColParams c; fill_col(h, c);
    c.jint = h->spec_a; c.z0 = state_member; c.zk = c.z0; c.acc = c.z0;
    c.st_tile_stride = (long long)h->nx * h->tw_state; c.st_row_stride = h->tw_state;
    CKL(h, launch_col(h->nx, COL_FWDT, c, 1, h->stream));
    return 0;
}

extern "C" int xfb_set_vorticity(xfb_handle h, int member, const float *vort)
{
    if (check_member(h, member)) return XFB_E_ARG;
    if (!vort) return fail(XFB_E_ARG, "null vorticity");
    CK(cudaSetDevice(h->device));
    if (h->nranks > 1) return dist_set_vorticity(h, vort);
    const void *din;
    if (stage_in(h, vort, h->real_a, sizeof(float) * h->grids, &din)) return XFB_E_CUDA;
    if (fused_diag_ok(h)) {
        if (fused_forward_to_state(h, (const float *)din, h->z0 + (size_t)member * h->hpad)) return XFB_E_CUDA;
    } else {
        if (fwd2d(h, (const float *)din, h->spec_a, h->spec_b)) return XFB_E_CUDA;
        if (launch_pw(h, OP_COPY, h->spec_b, h->pitch, h->z0 + (size_t)member * h->hpad, h->pitch, h->pitch, 0, h->tw_state))
            return XFB_E_CUDA;
    }
    h->have_state = true;
    h->tf_valid = false;
    if (!is_device_ptr(vort)) CK(cudaStreamSynchronize(h->stream));
    return 0;
}

extern "C" int xfb_set_spectrum(xfb_handle h, int member, const float *spec)
{
    if (check_member(h, member)) return XFB_E_ARG;
    if (!spec) return fail(XFB_E_ARG, "null spectrum");
    NO_SLAB(h, "xfb_set_spectrum");
    CK(cudaSetDevice(h->device));
    const void *din;
    if (stage_in(h, spec, h->ref_a, sizeof(cpx) * h->hgrids, &din)) return XFB_E_CUDA;
    if (launch_pw(h, OP_COPY, (const cpx *)din, h->hy, h->z0 + (size_t)member * h->hpad, h->pitch, h->hy, 0, h->tw_state))
        return XFB_E_CUDA;
    h->have_state = true;
    h->tf_valid = false;
    if (!is_device_ptr(spec)) CK(cudaStreamSynchronize(h->stream));
    return 0;
}

extern "C" int xfb_get_spectrum(xfb_handle h, int member, float *spec)
{
    if (check_member(h, member)) return XFB_E_ARG;
    if (!spec) return fail(XFB_E_ARG, "null spectrum");
    if (!h->have_state) return fail(XFB_E_STATE, "xfb_get_spectrum before xfb_set_vorticity");
    NO_SLAB(h, "xfb_get_spectrum");
    CK(cudaSetDevice(h->device));
    void *dout = stage_out_target(spec, h->ref_a);
    if (launch_pw(h, OP_COPY, h->z0 + (size_t)member * h->hpad, h->pitch, (cpx *)dout, h->hy, h->hy, h->tw_state, 0))
        return XFB_E_CUDA;
    return stage_out(h, spec, dout, sizeof(cpx) * h->hgrids);
}

extern "C" int xfb_set_source(xfb_handle h, int member, const float *src)
{
    if (check_member(h, member)) return XFB_E_ARG;
    CK(cudaSetDevice(h->device));
    if (!h->src) {
        if (!src) return 0;
        if (dev_alloc((void **)&h->src, sizeof(float) * h->grids * h->batch)) return XFB_E_CUDA;
        CK(cudaMemsetAsync(h->src, 0, sizeof(float) * h->grids * h->batch, h->stream));
    }
    float *dst = h->src + (size_t)member * h->grids;
    if (!src) {
        CK(cudaMemsetAsync(dst, 0, sizeof(float) * h->grids, h->stream));
    } else {
        CK(cudaMemcpyAsync(dst, src, sizeof(float) * h->grids,
                           is_device_ptr(src) ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, h->stream));
        h->has_src = true;
        if (!is_device_ptr(src)) CK(cudaStreamSynchronize(h->stream));
    }
    return 0;
}

int xfb::tracer_state_alloc(xfb_handle h)
{
    if (h->c0) return 0;
    const size_t sb = sizeof(cpx) * h->hpad * h->batch;
    cpx **state[] = {&h->c0, &h->ck, &h->cacc, &h->cjint};
    for (auto pp : state) {
        if (dev_alloc((void **)pp, sb)) return XFB_E_CUDA;
        CK(cudaMemsetAsync(*pp, 0, sb, h->stream));
    }
    if (!h->generic) {
        if (dev_alloc((void **)&h->tc[0], 2 * sb)) return XFB_E_CUDA;
        CK(cudaMemsetAsync(h->tc[0], 0, 2 * sb, h->stream));
        h->tc[1] = h->tc[0] + h->hpad * h->batch;
    }
    return 0;
}

// Passive tracer (SURVEY.md section 8 (f-4)): dc/dt = -u c_x - v c_y + kappa lap(c), advanced inside xfb_step by the
// velocity of the same Runge-Kutta stage with the vorticity equation's own operation order (dealiased tendency, same
// evolve / final combine).  The reference has no tracer; the definition is the oracle's (barotropic_oracle.c
// get_dtrcdt).  Per stage it costs one more K-ROW launch (the Jacobian kernel on T_u, T_cx, T_v, T_cy -- u and v are
// read from the vorticity stage's product arrays) and one K-COL launch (COL_TSTEP: 2 products instead of 4).
extern "C" int xfb_set_tracer(xfb_handle h, int member, const float *tracer, float kappa)
{
    if (check_member(h, member)) return XFB_E_ARG;
    if (!tracer) return fail(XFB_E_ARG, "null tracer");
    if (!fused_diag_ok(h) && !h->generic && h->nranks == 1 && h->nx != 16384)
        return fail(XFB_E_SIZE, "the passive tracer needs the fused kernels (power-of-two grids), a generic mixed-radix grid, or a slab-decomposed handle");
    CK(cudaSetDevice(h->device));
    if (tracer_state_alloc(h)) return XFB_E_CUDA;
    const void *din;
    if (stage_in(h, tracer, h->real_a, sizeof(float) * h->grids, &din)) return XFB_E_CUDA;
    if (h->nranks > 1) {
        if (int e = dist_set_tracer(h, (const float *)din)) return e;          // local rows; collective
    } else if (h->generic) {
        if (fwd2d(h, (const float *)din, h->spec_a, h->spec_b)) return XFB_E_CUDA;
        if (launch_pw(h, OP_COPY, h->spec_b, h->pitch, h->c0 + (size_t)member * h->hpad, h->pitch, h->pitch, 0, h->tw_state))
            return XFB_E_CUDA;
    } else if (fused_diag_ok(h)) {
        if (fused_forward_to_state(h, (const float *)din, h->c0 + (size_t)member * h->hpad)) return XFB_E_CUDA;
    } else {
        // 16384-point lines: plain transforms, then the layout conversion into the tile-major state
        if (fwd2d(h, (const float *)din, h->spec_a, h->spec_b)) return XFB_E_CUDA;
        if (launch_pw(h, OP_COPY, h->spec_b, h->pitch, h->c0 + (size_t)member * h->hpad, h->pitch, h->pitch, 0, h->tw_state))
            return XFB_E_CUDA;
    }
    if (!h->has_tracer || h->kappa != kappa) drop_step_graph(h);     // it has no tracer launches / another diffusivity baked in
    h->has_tracer = true;
    h->kappa = kappa;
    h->tcf_valid = false;
    if (!is_device_ptr(tracer)) CK(cudaStreamSynchronize(h->stream));
    return 0;
}

// Linear terms of the vorticity equation (DESIGN.md section 3): -beta v - mu zeta - nu_h (-lap)^order zeta, added per mode as
// L(k) Z_k next to the nu term inside the dealiasing mask of every Runge-Kutta stage.  The passive tracer keeps its kappa
// lap(c) only.  With a non-zero term the stepper runs the LIN instances of its K-COL kernels (and of gen_stage on the
// generic grids); all zeros switches back to the default kernels.  A change drops the captured step graph, which bakes
// the kernel parameters in.
extern "C" int xfb_set_linear_terms(xfb_handle h, float beta, float mu, float nu_h, int order)
{
    if (!h) return fail(XFB_E_ARG, "null handle");
    if (!std::isfinite(beta) || !std::isfinite(mu) || !std::isfinite(nu_h))
        return fail(XFB_E_ARG, "xfb_set_linear_terms: beta, mu and nu_h must be finite");
    if (mu < 0.0f || nu_h < 0.0f) return fail(XFB_E_ARG, "xfb_set_linear_terms: mu and nu_h must be >= 0");
    if (order < 1 || order > 8) return fail(XFB_E_ARG, "xfb_set_linear_terms: order %d not in 1..8", order);
    LinCoef L;
    memset(&L, 0, sizeof(L));
    if (beta != 0.0f || mu != 0.0f || nu_h != 0.0f) {
        // hyperviscosity as ch (k^2 / k_c^2)^order with the largest wavenumber of the grid, k_c^2 = kx(nx/2)^2 + ky(ny/2)^2
        // (the float expressions of the wavenumber tables): (k^2 / k_c^2)^order <= 1 never overflows, whatever the size
        // and domain length; ch = nu_h k_c^(2 order) is formed in float64 and must be a normal float
        const float TWOPI = acosf(-1.0f) * 2.0f;
        const double kxc = (double)(TWOPI * ((float)(h->nx / 2)) / h->lx), kyc = (double)(TWOPI * ((float)(h->ny / 2)) / h->ly);
        const double kc2 = kxc * kxc + kyc * kyc;
        const double ch = (double)nu_h * std::pow(kc2, (double)order);
        if (!std::isfinite(ch) || ch > (double)FLT_MAX || (nu_h != 0.0f && ch < (double)FLT_MIN))
            return fail(XFB_E_ARG, "xfb_set_linear_terms: nu_h * k_c^%d = %g is out of float range", 2 * order, ch);
        L.beta = beta; L.mu = mu; L.ch = (float)ch; L.inv_kc2 = (float)(1.0 / kc2); L.order = order; L.on = 1;
    }
    if (memcmp(&L, &h->lin, sizeof(L)) != 0) {
        // the captured step (fused or generic path) has the old coefficients baked in
        if (h->step_graph) CK(cudaSetDevice(h->device));
        drop_step_graph(h);
        h->lin = L;
    }
    return 0;
}

// K-COL parameters of the fused stepper: every member's state (tile-major), tendency and product arrays
static void stepper_col(xfb_handle h, ColParams &c)
{
    fill_col(h, c);
    c.jint = h->jint; c.z0 = h->z0; c.zk = h->zk; c.acc = h->acc;
    c.st_tile_stride = (long long)h->nx * h->tw_state; c.st_row_stride = h->tw_state;     // tile-major state
    for (int f = 0; f < 4; ++f) c.t_out[f] = h->t[f];
}

extern "C" int xfb_step(xfb_handle h, int nsteps, float dt)
{
    if (!h) return fail(XFB_E_ARG, "null handle");
    if (nsteps < 0) return fail(XFB_E_ARG, "negative step count");
    if (!h->have_state) return fail(XFB_E_STATE, "xfb_step before xfb_set_vorticity");
    CK(cudaSetDevice(h->device));
    if (h->nranks > 1) return dist_step(h, nsteps, dt);
    if (h->generic) return step_replay(h, nsteps, dt, false, [&]() { return generic_one_step(h, dt); });
    ColParams c; stepper_col(h, c);
    c.dt = dt;
    RowParams r; fill_row(h, r, h->nx * h->batch);
    for (int f = 0; f < 4; ++f) r.spec_in[f] = h->t[f];
    r.real_in = h->has_src ? h->src : nullptr;
    r.spec_out = h->jint;
    if (nsteps > 0 && !h->tf_valid) {
        CKL(h, launch_col(h->nx, COL_PRO, c, h->batch, h->stream));
        h->tf_valid = true;
    }
    // passive tracer: its own state and Jacobian arrays, the vorticity stage's velocity products
    const bool tracer = h->has_tracer;
    ColParams ct = c;
    RowParams rt = r;
    if (tracer) {
        ct.jint = h->cjint; ct.z0 = h->c0; ct.zk = h->ck; ct.acc = h->cacc; ct.nu = h->kappa;
        ct.t_out[0] = h->tc[0]; ct.t_out[1] = h->tc[1]; ct.t_out[2] = h->tc[0]; ct.t_out[3] = h->tc[1];
        rt.spec_in[0] = h->tc[0]; rt.spec_in[1] = h->tc[1];           // c_x, c_y ; [2], [3] stay u, v
        rt.real_in = nullptr; rt.spec_out = h->cjint;
        if (nsteps > 0 && !h->tcf_valid) {
            CKL(h, launch_col(h->nx, COL_TPRO, ct, h->batch, h->stream));
            h->tcf_valid = true;
        }
    }
    return step_replay(h, nsteps, dt, true, [&]() -> int {
        for (int k = 1; k <= 4; ++k) {
            if (h->profiling) cudaEventRecord(next_event(h->ev_row, h->ev_row_used), h->stream);
            CKL(h, launch_row(h->ny, ROW_JAC, r, h->stream));
            if (tracer) CKL(h, launch_row(h->ny, ROW_JAC, rt, h->stream));     // before K-COL overwrites u, v
            if (h->profiling) {
                cudaEventRecord(next_event(h->ev_row, h->ev_row_used), h->stream);
                cudaEventRecord(next_event(h->ev_col, h->ev_col_used), h->stream);
            }
            c.stage = k;
            c.dt_stage = (k == 3) ? dt : dt / 2.0f;          // main.cpp:296,299,302
            CKL(h, launch_col(h->nx, COL_STEP, c, h->batch, h->stream));
            if (tracer) {
                ct.stage = k; ct.dt_stage = c.dt_stage;
                CKL(h, launch_col(h->nx, COL_TSTEP, ct, h->batch, h->stream));
            }
            if (h->profiling) cudaEventRecord(next_event(h->ev_col, h->ev_col_used), h->stream);
        }
        return 0;
    });
}

// The launches of a step are captured once into a CUDA graph and replayed: on small grids (one launch is 15-25 us at
// 512^2 / 1024^2 on the fused path; the generic path issues 72 short launches per member) the launch gaps are a large
// part of the step.  The first step of a handle runs eagerly (it also configures the kernels); XFB_NO_GRAPH=1, and
// per-kernel profiling of the fused step (its events), keep the eager path.  The graph is captured again when dt or
// the source pointer changes; xfb_set_tracer and xfb_set_linear_terms drop it.
int xfb::step_replay(xfb_handle h, int nsteps, float dt, bool eager_if_profiling, const std::function<int()> &one_step)
{
    static const bool no_graph = getenv("XFB_NO_GRAPH") && atoi(getenv("XFB_NO_GRAPH")) != 0;
    const bool eager_all = no_graph || (eager_if_profiling && h->profiling);
    int s = 0;
    if (nsteps > 0 && (!h->warmed || eager_all)) {
        const int eager = eager_all ? nsteps : 1;
        for (; s < eager; ++s)
            if (int e = one_step()) return e;
        h->warmed = true;
    }
    if (s < nsteps) {
        const void *src_now = h->has_src ? (const void *)h->src : nullptr;
        if (!h->step_graph || h->graph_dt != dt || h->graph_src != src_now) {
            drop_step_graph(h);
            cudaGraph_t g = nullptr;
            CK(cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeRelaxed));
            const long long l0 = h->launches;
            const int e = one_step();
            const int per_step = (int)(h->launches - l0);
            h->launches = l0;
            cudaError_t ce = cudaStreamEndCapture(h->stream, &g);
            if (e) { if (g) cudaGraphDestroy(g); return e; }
            if (ce != cudaSuccess) return fail(XFB_E_CUDA, "cudaStreamEndCapture: %s", cudaGetErrorString(ce));
            cudaGraphExec_t ge = nullptr;
            ce = cudaGraphInstantiate(&ge, g, 0);
            cudaGraphDestroy(g);
            if (ce != cudaSuccess) return fail(XFB_E_CUDA, "cudaGraphInstantiate: %s", cudaGetErrorString(ce));
            h->step_graph = ge; h->graph_dt = dt; h->graph_src = src_now; h->graph_launches = per_step;
        }
        for (; s < nsteps; ++s) {
            CK(cudaGraphLaunch((cudaGraphExec_t)h->step_graph, h->stream));
            h->launches += h->graph_launches;
        }
    }
    return 0;
}

const FieldOps *xfb::field_ops(int which)
{
    static const FieldOps table[] = {
        {1, {OP_COPY}, 0},                          // XFB_VORT
        {1, {OP_INVLAP}, 0},                        // XFB_PSI
        {2, {OP_INVLAP, OP_GRADY}, 1},              // XFB_U = -psi_y
        {2, {OP_INVLAP, OP_GRADX}, 0},              // XFB_V = psi_x
        {0}, {0}, {0},                              // XFB_SRC, XFB_TFIL, XFB_DEFORM
        {1, {OP_GRADX}, 0},                         // XFB_DVORTDX
        {1, {OP_GRADY}, 0},                         // XFB_DVORTDY
        {1, {OP_COPY}, 0},                          // XFB_TRACER (of the tracer's state)
    };
    static_assert(sizeof(table) / sizeof(table[0]) == XFB_TRACER + 1, "one entry per field id");
    if (which < 0 || which > XFB_TRACER || table[which].nops == 0) return nullptr;
    return &table[which];
}

const FieldOps xfb::psi_second_ops[3] = {
    {3, {OP_INVLAP, OP_GRADX, OP_GRADY}, 0},    // psi_xy
    {3, {OP_INVLAP, OP_GRADX, OP_GRADX}, 0},    // psi_xx
    {3, {OP_INVLAP, OP_GRADY, OP_GRADY}, 0},    // psi_yy
};

// operator chain `f` of one member's state array z (tile-major, or row-major on generic grids) -> physical field in
// `dout` (device), reference normalisation; spec_a and spec_b are the scratch
static int chain_to_device(xfb_handle h, const cpx *z, const FieldOps &f, float *dout)
{
    const float scale = 1.0f / (float)((double)h->nx * (double)h->ny);
    const int P = h->pitch;
    if (launch_pw(h, f.ops[0], z, P, h->spec_a, P, P, h->tw_state, 0)) return XFB_E_CUDA;
    for (int o = 1; o < f.nops; ++o)
        if (launch_pw(h, f.ops[o], h->spec_a, P, h->spec_a, P, P)) return XFB_E_CUDA;
    return inv2d(h, h->spec_a, h->spec_b, dout, scale, f.negate);
}

// derived spectral field of member -> physical field in `dout` (device), reference normalisation
static int derived_field(xfb_handle h, int member, int which, float *dout, const cpx *state = nullptr)
{
    if (which == XFB_TRACER) {
        if (!h->has_tracer) return fail(XFB_E_STATE, "XFB_TRACER before xfb_set_tracer");
        return derived_field(h, member, XFB_VORT, dout, h->c0);
    }
    const cpx *z = (state ? state : h->z0) + (size_t)member * h->hpad;
    const float scale = 1.0f / (float)((double)h->nx * (double)h->ny);
    if (fused_diag_ok(h)) {
        // record fields on the stepper's kernels: one K-COL launch (spectral multiplier + x pass, TMA-staged) and one
        // K-ROW launch (y pass, normalisation, sign); multipliers in float32 (<= 2 ulp from the operator tier's tables)
        if (fused_products(h, member, 2 + which, 1, state)) return XFB_E_CUDA;
        RowParams r; fill_row(h, r, h->nx);
        r.spec_in[0] = h->dg; r.real_out = dout; r.scale = scale; r.negate = (which == XFB_U) ? 1 : 0;
        CKL(h, launch_row(h->ny, ROW_C2R, r, h->stream));
        return 0;
    }
    const FieldOps *f = field_ops(which);
    if (!f) return fail(XFB_E_ARG, "bad field id %d", which);
    return chain_to_device(h, z, *f, dout);
}

// filamentation time and deformation factor from psi_xy, psi_xx, psi_yy
__global__ void diag_kernel(const float *pxy, const float *pxx, const float *pyy, float *out, long long n, int which)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float s1 = __fmul_rn(-2.0f, pxy[i]), s2 = __fsub_rn(pxx[i], pyy[i]), z = __fadd_rn(pxx[i], pyy[i]);
    const float ss = __fadd_rn(__fmul_rn(s1, s1), __fmul_rn(s2, s2)), zz = __fmul_rn(z, z);
    const float q = __fsub_rn(ss, zz), den = __fadd_rn(ss, zz);
    if (which == XFB_TFIL) out[i] = (q > 0.0f) ? __fdiv_rn(2.0f, __fsqrt_rn(q)) : 0.0f;
    else out[i] = (den > 0.0f) ? __fdiv_rn(q, den) : 0.0f;
}

int xfb::launch_strain(xfb_handle h, const float *pxy, const float *pxx, const float *pyy, float *out, long long n, int which)
{
    diag_kernel<<<(unsigned)((n + 255) / 256), 256, 0, h->stream>>>(pxy, pxx, pyy, out, n, which);
    CK(cudaGetLastError());
    h->launches++;
    return 0;
}

// Both strain diagnostics of member from ONE set of the three second derivatives of psi, into device buffers; either
// may be null.  Filamentation time (Rozoff et al. 2006) and deformation factor, README.md:5,7.  The fused pair writes
// both outputs, so a missing one goes to scratch.  Otherwise psi_xy -> real_b, psi_xx -> real_c, psi_yy -> real_a; an
// output may be real_a only when it is the sole output (the strain kernel then runs in place).
static int strain_to_device(xfb_handle h, int member, float *tfil, float *deform)
{
    if (fused_diag_ok(h)) return fused_diag(h, member, 0, tfil ? tfil : h->real_c, deform ? deform : h->real_b);
    const cpx *z = h->z0 + (size_t)member * h->hpad;
    if (chain_to_device(h, z, psi_second_ops[0], h->real_b) || chain_to_device(h, z, psi_second_ops[1], h->real_c) ||
        chain_to_device(h, z, psi_second_ops[2], h->real_a))
        return XFB_E_CUDA;
    const long long n = (long long)h->grids;
    if (tfil && launch_strain(h, h->real_b, h->real_c, h->real_a, tfil, n, XFB_TFIL)) return XFB_E_CUDA;
    if (deform && launch_strain(h, h->real_b, h->real_c, h->real_a, deform, n, XFB_DEFORM)) return XFB_E_CUDA;
    return 0;
}

// field `which` of member into the DEVICE buffer dout (grids floats), on the handle's stream
static int field_to_device(xfb_handle h, int member, int which, float *dout)
{
    const size_t bytes = sizeof(float) * h->grids;
    if (which == XFB_SRC) {
        if (!h->src) { CK(cudaMemsetAsync(dout, 0, bytes, h->stream)); return 0; }
        CK(cudaMemcpyAsync(dout, h->src + (size_t)member * h->grids, bytes, cudaMemcpyDeviceToDevice, h->stream));
        return 0;
    }
    if (which == XFB_TFIL || which == XFB_DEFORM)      // dout may be real_a
        return strain_to_device(h, member, which == XFB_TFIL ? dout : nullptr, which == XFB_DEFORM ? dout : nullptr);
    return derived_field(h, member, which, dout);
}

extern "C" int xfb_get_field(xfb_handle h, int member, int which, float *out)
{
    if (check_member(h, member)) return XFB_E_ARG;
    if (!out) return fail(XFB_E_ARG, "null output");
    if (!h->have_state) return fail(XFB_E_STATE, "xfb_get_field before xfb_set_vorticity");
    CK(cudaSetDevice(h->device));
    if (h->nranks > 1 && which != XFB_SRC) return dist_get_field(h, which, out);
    const size_t bytes = sizeof(float) * h->grids;
    if (which == XFB_SRC && !h->src && !is_device_ptr(out)) { memset(out, 0, bytes); return 0; }
    float *dout = (float *)stage_out_target(out, h->real_a);
    if (field_to_device(h, member, which, dout)) return XFB_E_CUDA;
    if (which == XFB_SRC && dout == out) { CK(cudaStreamSynchronize(h->stream)); return 0; }
    return stage_out(h, out, dout, bytes);
}

// ---- asynchronous record output: the fields of the current state travel to pinned host buffers on a second stream
// while the caller goes on stepping (src/main.cpp:266-282,183-222 overlapped with the following steps) --------------
extern "C" int xfb_host_alloc(float **p, size_t nfloats)
{
    if (!p) return fail(XFB_E_ARG, "null pointer");
    CK(cudaMallocHost((void **)p, sizeof(float) * nfloats));
    return 0;
}

extern "C" int xfb_host_free(float *p)
{
    if (p) CK(cudaFreeHost(p));
    return 0;
}

extern "C" int xfb_get_field_async(xfb_handle h, int member, int which, float *pinned_out, int *ticket)
{
    if (check_member(h, member)) return XFB_E_ARG;
    if (!pinned_out || !ticket) return fail(XFB_E_ARG, "null argument");
    if (!h->have_state) return fail(XFB_E_STATE, "xfb_get_field_async before xfb_set_vorticity");
    NO_SLAB(h, "xfb_get_field_async");
    CK(cudaSetDevice(h->device));
    if (!h->rec_stream) {
        CK(cudaStreamCreateWithFlags(&h->rec_stream, cudaStreamNonBlocking));
        for (int i = 0; i < XFB_NREC; ++i) {
            CK(cudaEventCreateWithFlags(&h->rec_ready[i], cudaEventDisableTiming));
            CK(cudaEventCreateWithFlags(&h->rec_done[i], cudaEventDisableTiming));
        }
    }
    // rec_next is read by xfb_wait_field from another host thread (main.out's writer): atomic accesses, and the slot's
    // events are recorded BEFORE the ticket is published
    const int next = __atomic_load_n(&h->rec_next, __ATOMIC_RELAXED);
    const int slot = next % XFB_NREC;
    if (next >= XFB_NREC) CK(cudaEventSynchronize(h->rec_done[slot]));        // the slot's previous copy has left
    if (!h->rec_buf[slot] && dev_alloc((void **)&h->rec_buf[slot], sizeof(float) * h->grids)) return XFB_E_CUDA;
    if (field_to_device(h, member, which, h->rec_buf[slot])) return XFB_E_CUDA;
    CK(cudaEventRecord(h->rec_ready[slot], h->stream));
    CK(cudaStreamWaitEvent(h->rec_stream, h->rec_ready[slot], 0));
    CK(cudaMemcpyAsync(pinned_out, h->rec_buf[slot], sizeof(float) * h->grids, cudaMemcpyDeviceToHost, h->rec_stream));
    CK(cudaEventRecord(h->rec_done[slot], h->rec_stream));
    *ticket = next;
    __atomic_store_n(&h->rec_next, next + 1, __ATOMIC_RELEASE);
    return 0;
}

extern "C" int xfb_wait_field(xfb_handle h, int ticket)
{
    if (!h) return fail(XFB_E_ARG, "null handle");
    // thread-safe against a concurrent xfb_get_field_async on the same handle (one producer, one waiter)
    const int next = __atomic_load_n(&h->rec_next, __ATOMIC_ACQUIRE);
    if (ticket < 0 || ticket >= next) return fail(XFB_E_ARG, "bad ticket %d", ticket);
    if (next - ticket > XFB_NREC) return 0;                     // its slot has been reused: that copy completed long ago
    CK(cudaSetDevice(h->device));
    CK(cudaEventSynchronize(h->rec_done[ticket % XFB_NREC]));
    return 0;
}

// Fused diagnostics (north_star item 4): ONE K-COL launch forms the three spectral products of the current state and
// transforms them along x (COL_DIAG: psi_xy, psi_xx, psi_yy or zeta, zeta_x, zeta_y), ONE K-ROW launch transforms them
// along y and combines them pointwise (ROW_DIAG) -- the stepper's TMA-staged persistent kernels with other
// multipliers.  Replaces 6-9 pointwise passes, 3 column and 3 row transforms of the record path.
static bool fused_diag_ok(xfb_handle h)
{
    // XFB_DIAG_UNFUSED=1: every grid takes the unfused record path that 16384 and generic grids take (A/B knob)
    static const bool off = getenv("XFB_DIAG_UNFUSED") && atoi(getenv("XFB_DIAG_UNFUSED")) != 0;
    return !off && !h->generic && h->nranks == 1 && h->nx <= 8192 && h->ny <= 8192;
}

// K-COL half: `nfields` spectral products of member's state, x-inverse-transformed into h->dg[0 .. nfields-1]
static int fused_products(xfb_handle h, int member, int kind, int nfields, const cpx *state)
{
    if (!h->dg) {
        if (dev_alloc((void **)&h->dg, 3 * sizeof(cpx) * h->hpad)) return XFB_E_CUDA;
        CK(cudaMemsetAsync(h->dg, 0, 3 * sizeof(cpx) * h->hpad, h->stream));
    }
    ColParams c; fill_col(h, c);
    c.z0 = const_cast<cpx *>(state ? state : h->z0) + (size_t)member * h->hpad; c.zk = c.z0; c.acc = c.z0; c.jint = h->jint;
    c.st_tile_stride = (long long)h->nx * h->tw_state; c.st_row_stride = h->tw_state;
    for (int f = 0; f < 4; ++f) c.t_out[f] = h->dg + (size_t)(f < 3 ? f : 2) * h->hpad;
    c.stage = kind;
    c.nfields = nfields;
    CKL(h, launch_col(h->nx, COL_DIAG, c, 1, h->stream));
    return 0;
}

static int fused_diag(xfb_handle h, int member, int kind, float *out0, float *out1, const cpx *state)
{
    if (fused_products(h, member, kind, 3, state)) return XFB_E_CUDA;
    RowParams r; fill_row(h, r, h->nx);
    for (int f = 0; f < 3; ++f) r.spec_in[f] = h->dg + (size_t)f * h->hpad;
    r.real_out = out0; r.real_out2 = out1; r.diag_kind = kind;
    CKL(h, launch_row(h->ny, ROW_DIAG, r, h->stream));
    return 0;
}

// both strain diagnostics of one member (xfb_get_field recomputes the second derivatives of psi per field); either
// output may be NULL.  Host or device pointers.
extern "C" int xfb_get_diagnostics(xfb_handle h, int member, float *tfil, float *deform)
{
    if (check_member(h, member)) return XFB_E_ARG;
    if (!tfil && !deform) return fail(XFB_E_ARG, "no output requested");
    if (!h->have_state) return fail(XFB_E_STATE, "xfb_get_diagnostics before xfb_set_vorticity");
    CK(cudaSetDevice(h->device));
    if (h->nranks > 1) return dist_diagnostics(h, tfil, deform);          // local rows; collective
    const size_t bytes = sizeof(float) * h->grids;
    // host outputs are produced in the reference-layout scratch arrays (2 * hgrids floats >= grids floats)
    float *dt = tfil ? (float *)stage_out_target(tfil, h->ref_a) : nullptr;
    float *dd = deform ? (float *)stage_out_target(deform, h->ref_b) : nullptr;
    if (strain_to_device(h, member, dt, dd)) return XFB_E_CUDA;
    if (tfil && stage_out(h, tfil, dt, bytes, false)) return XFB_E_CUDA;
    if (deform && stage_out(h, deform, dd, bytes, false)) return XFB_E_CUDA;
    if (dt != tfil || dd != deform) CK(cudaStreamSynchronize(h->stream));      // one wait for the host copies
    return 0;
}

// histogram of area and |grad zeta|^2 over tracer bins
__global__ void keff_hist_kernel(const float *c, const float *gx, const float *gy, long long n, int nbins, float cmin,
                                 float scale, double da, double *area, double *grad2)
{
    // Most of the domain sits in one bin (zeta ~ 0 away from the vortex): a naive shared-memory atomicAdd per point
    // serialises on that address (measured 2.6 ms at 4096^2).  Each thread therefore runs over its elements with a
    // private (bin, count, sum) accumulator and only touches shared memory when the bin changes.
    extern __shared__ double sh[];
    double *sg = sh;                                                   // [nbins] sum of |grad c|^2
    unsigned long long *sc = reinterpret_cast<unsigned long long *>(sh + nbins);   // [nbins] point counts
    for (int b = threadIdx.x; b < nbins; b += blockDim.x) { sg[b] = 0.0; sc[b] = 0ull; }
    __syncthreads();
    int cur = -1;
    unsigned long long cnt = 0;
    double acc = 0.0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        int b = (int)floorf(__fmul_rn(__fsub_rn(c[i], cmin), scale));
        b = b < 0 ? 0 : (b >= nbins ? nbins - 1 : b);
        const float g2 = gy ? __fadd_rn(__fmul_rn(gx[i], gx[i]), __fmul_rn(gy[i], gy[i])) : gx[i];   // gy == null: gx holds |grad c|^2
        if (b != cur) {
            if (cur >= 0) { atomicAdd(&sc[cur], cnt); atomicAdd(&sg[cur], acc); }
            cur = b; cnt = 0; acc = 0.0;
        }
        ++cnt;
        acc += (double)g2;
    }
    if (cur >= 0) { atomicAdd(&sc[cur], cnt); atomicAdd(&sg[cur], acc); }
    __syncthreads();
    for (int b = threadIdx.x; b < nbins; b += blockDim.x) {
        if (sc[b] != 0ull) {
            atomicAdd(&area[b], (double)sc[b] * da);
            atomicAdd(&grad2[b], sg[b] * da);
        }
    }
}

int xfb::launch_keff_hist(xfb_handle h, const float *c, const float *gx, const float *gy, long long n, int nbins, float cmin,
                          float cmax, double *d_area, double *d_grad2)
{
    const double da = ((double)h->lx / h->nx) * ((double)h->ly / h->ny);
    const float scale = (float)nbins / (cmax - cmin);
    keff_hist_kernel<<<296, 256, sizeof(double) * 2 * nbins, h->stream>>>(c, gx, gy, n, nbins, cmin, scale, da, d_area, d_grad2);
    CK(cudaGetLastError());
    h->launches++;
    return 0;
}

int xfb::keff_hist_args(int nbins, float cmin, float cmax, const double *area, const double *grad2)
{
    if (!area || !grad2 || nbins < 1 || nbins > 2048 || !(cmax > cmin)) return fail(XFB_E_ARG, "bad histogram arguments");
    return 0;
}

int xfb::keff_hist_finish(xfb_handle h, const double *d, int nbins, double *area, double *grad2)
{
    std::vector<double> host(2 * (size_t)nbins);
    CK(cudaMemcpyAsync(host.data(), d, sizeof(double) * 2 * nbins, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    memcpy(area, host.data(), sizeof(double) * nbins);
    memcpy(grad2, host.data() + nbins, sizeof(double) * nbins);
    return 0;
}

static int keff_hist_impl(xfb_handle h, int member, int nbins, float cmin, float cmax, double *area, double *grad2,
                          const cpx *state)
{
    const bool fused = fused_diag_ok(h);
    if (fused) {
        if (fused_diag(h, member, 1, h->real_a, h->real_b, state)) return XFB_E_CUDA;       // c, |grad c|^2
    } else {
        if (derived_field(h, member, XFB_VORT, h->real_a, state)) return XFB_E_CUDA;
        if (derived_field(h, member, XFB_DVORTDX, h->real_b, state)) return XFB_E_CUDA;
        if (derived_field(h, member, XFB_DVORTDY, h->real_c, state)) return XFB_E_CUDA;
    }
    double *d = (double *)h->ref_a;
    CK(cudaMemsetAsync(d, 0, sizeof(double) * 2 * nbins, h->stream));
    if (launch_keff_hist(h, h->real_a, h->real_b, fused ? nullptr : h->real_c, (long long)h->grids, nbins, cmin, cmax, d, d + nbins))
        return XFB_E_CUDA;
    return keff_hist_finish(h, d, nbins, area, grad2);
}

// slab handles: every rank bins its own rows, one all-reduce of the 2 * nbins sums (SURVEY.md 8e); collective
extern "C" int xfb_get_keff_hist(xfb_handle h, int member, int nbins, float cmin, float cmax, double *area, double *grad2)
{
    if (check_member(h, member)) return XFB_E_ARG;
    if (!h->have_state) return fail(XFB_E_STATE, "xfb_get_keff_hist before xfb_set_vorticity");
    if (int e = keff_hist_args(nbins, cmin, cmax, area, grad2)) return e;
    CK(cudaSetDevice(h->device));
    if (h->nranks > 1) return dist_keff_hist(h, nbins, cmin, cmax, area, grad2, false);
    return keff_hist_impl(h, member, nbins, cmin, cmax, area, grad2, nullptr);
}

// the same histograms over the passive tracer (Hendricks & Schubert 2009 use a tracer distinct from the vorticity)
extern "C" int xfb_get_tracer_keff_hist(xfb_handle h, int member, int nbins, float cmin, float cmax, double *area,
                                        double *grad2)
{
    if (check_member(h, member)) return XFB_E_ARG;
    if (!h->has_tracer) return fail(XFB_E_STATE, "xfb_get_tracer_keff_hist before xfb_set_tracer");
    if (int e = keff_hist_args(nbins, cmin, cmax, area, grad2)) return e;
    CK(cudaSetDevice(h->device));
    if (h->nranks > 1) return dist_keff_hist(h, nbins, cmin, cmax, area, grad2, true);
    return keff_hist_impl(h, member, nbins, cmin, cmax, area, grad2, h->c0);
}

// Quadratic invariants E, Z, P of the state (vorticity or tracer) and their isotropic shell spectra, reduced on the device
// from the tile-major (or generic row-major) state in one launch (xfb_spectra.cu); definitions in DESIGN.md section 3.
int xfb::energy_spectrum_args(xfb_handle h, int member, int which, int nshells, const double *totals, const double *e,
                              const double *z, const char *api)
{
    if (check_member(h, member)) return XFB_E_ARG;
    if (which != XFB_VORT && which != XFB_TRACER)
        return fail(XFB_E_ARG, "%sget_energy_spectrum: which must be XFB_VORT or XFB_TRACER", api);
    if (nshells < 0 || nshells > XFB_SPECTRUM_MAX_SHELLS)
        return fail(XFB_E_ARG, "%sget_energy_spectrum: nshells %d not in 0..%d", api, nshells, XFB_SPECTRUM_MAX_SHELLS);
    if (!totals || (nshells > 0 && (!e || !z))) return fail(XFB_E_ARG, "%sget_energy_spectrum: null output", api);
    if (!h->have_state) return fail(XFB_E_STATE, "%sget_energy_spectrum before %sset_vorticity", api, api);
    if (which == XFB_TRACER && !h->has_tracer)
        return fail(XFB_E_STATE, "%sget_energy_spectrum: XFB_TRACER before %sset_tracer", api, api);
    return 0;
}

extern "C" int xfb_get_energy_spectrum(xfb_handle h, int member, int which, int nshells, double *totals, double *e, double *z)
{
    if (int r = energy_spectrum_args(h, member, which, nshells, totals, e, z, "xfb_")) return r;
    CK(cudaSetDevice(h->device));
    if (h->nranks > 1) return dist_energy_spectrum(h, which, nshells, totals, e, z);     // collective
    if (energy_spectrum_scratch(h)) return XFB_E_CUDA;
    const cpx *state = (which == XFB_TRACER ? h->c0 : h->z0) + (size_t)member * h->hpad;
    CK(cudaMemsetAsync(h->espec, 0, sizeof(double) * (3 + 2 * (size_t)nshells), h->stream));
    if (launch_energy_spectrum(h, state, nshells, h->espec)) return XFB_E_CUDA;
    return energy_spectrum_finish(h, h->espec, nshells, totals, e, z);
}

// Spectral budget of the vorticity (DESIGN.md section 3): the tendency N = r2c(-u.grad(zeta)) and the source's spectrum S
// of one member are formed with the stepper's own transforms into scratch arrays in the state's layout, then one
// reduction (xfb_spectra.cu) reads state, N and S once.  Scratch: spec_a, spec_b and jint, which the next stage
// overwrites before reading; the products t[0..3] of the current state are formed as the next step would form them.
int xfb::spectral_budget_args(xfb_handle h, int member, int nshells, const double *totals, const double *budget, const char *api)
{
    if (check_member(h, member)) return XFB_E_ARG;
    if (nshells < 0 || nshells > XFB_SPECTRUM_MAX_SHELLS)
        return fail(XFB_E_ARG, "%sget_spectral_budget: nshells %d not in 0..%d", api, nshells, XFB_SPECTRUM_MAX_SHELLS);
    if (!totals || (nshells > 0 && !budget)) return fail(XFB_E_ARG, "%sget_spectral_budget: null output", api);
    if (!h->have_state) return fail(XFB_E_STATE, "%sget_spectral_budget before %sset_vorticity", api, api);
    return 0;
}

// tendency and source spectrum of one member on one GPU, tile-major (row-major on generic grids); *n, *s name the arrays
// (*s null without a source)
static int budget_terms(xfb_handle h, int member, const cpx **n, const cpx **s)
{
    const float *src = h->has_src ? h->src + (size_t)member * h->grids : nullptr;
    *s = nullptr;
    if (h->generic) {
        // generic_one_step's stage body without the source, stopping before gen_stage
        if (generic_tendency(h, h->z0 + (size_t)member * h->hpad, nullptr, h->jint)) return XFB_E_CUDA;
        *n = h->jint;
        if (src) {
            if (fwd2d(h, src, h->spec_a, h->spec_b)) return XFB_E_CUDA;
            *s = h->spec_b;
        }
        return 0;
    }
    if (!h->tf_valid) {
        ColParams c; stepper_col(h, c);
        CKL(h, launch_col(h->nx, COL_PRO, c, h->batch, h->stream));
        h->tf_valid = true;
    }
    RowParams r; fill_row(h, r, h->nx);
    for (int f = 0; f < 4; ++f) r.spec_in[f] = h->t[f] + (size_t)member * h->hpad;
    r.real_in = nullptr;
    r.spec_out = h->spec_a;
    CKL(h, launch_row(h->ny, ROW_JAC, r, h->stream));
    if (h->nx <= 8192 && h->ny <= 8192) {
        // x pass of the pair-layout tendency straight into tile-major scratch, then the source the way set_vorticity goes
        ColParams c; fill_col(h, c);
        c.jint = h->spec_a; c.z0 = h->spec_b; c.zk = c.z0; c.acc = c.z0;
        c.st_tile_stride = (long long)h->nx * h->tw_state; c.st_row_stride = h->tw_state;
        CKL(h, launch_col(h->nx, COL_FWDT, c, 1, h->stream));
        *n = h->spec_b;
        if (src) {
            if (fused_forward_to_state(h, src, h->jint)) return XFB_E_CUDA;
            *s = h->jint;
        }
        return 0;
    }
    // 16384-point lines: plain x pass into row-major scratch, then the layout conversion (as xfb_set_tracer does)
    ColParams c; fill_col(h, c);
    c.jint = h->spec_a; c.z0 = h->spec_b;
    CKL(h, launch_col(h->nx, COL_FWD, c, 1, h->stream));
    if (launch_pw(h, OP_COPY, h->spec_b, h->pitch, h->jint, h->pitch, h->pitch, 0, h->tw_state)) return XFB_E_CUDA;
    *n = h->jint;
    if (src) {
        if (fwd2d(h, src, h->spec_a, h->spec_b)) return XFB_E_CUDA;
        if (launch_pw(h, OP_COPY, h->spec_b, h->pitch, h->spec_a, h->pitch, h->pitch, 0, h->tw_state)) return XFB_E_CUDA;
        *s = h->spec_a;
    }
    return 0;
}

extern "C" int xfb_get_spectral_budget(xfb_handle h, int member, int nshells, double *totals, double *budget)
{
    if (int r = spectral_budget_args(h, member, nshells, totals, budget, "xfb_")) return r;
    CK(cudaSetDevice(h->device));
    if (h->nranks > 1) return dist_spectral_budget(h, nshells, totals, budget);      // collective
    if (spectral_budget_scratch(h)) return XFB_E_CUDA;
    const cpx *n, *s;
    if (budget_terms(h, member, &n, &s)) return XFB_E_CUDA;
    CK(cudaMemsetAsync(h->bspec, 0, sizeof(double) * XFB_BUDGET_N * (1 + (size_t)nshells), h->stream));
    if (launch_spectral_budget(h, h->z0 + (size_t)member * h->hpad, n, s, nshells, h->bspec)) return XFB_E_CUDA;
    return spectral_budget_finish(h, h->bspec, nshells, totals, budget);
}

// ------------------------------------------------------------------------------------------------
// pressure inversion (invert_pres.cpp:132-187)
// ------------------------------------------------------------------------------------------------
__global__ void gauss_curv_kernel(const float *dx2, const float *dy2, const float *dxdy, float *out, long long n)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    // invert_pres.cpp:159: float product, then `pow(float, 2.0f)` = ::pow(double,double) and a double subtraction
    out[i] = (float)((double)__fmul_rn(dx2[i], dy2[i]) - (double)dxdy[i] * (double)dxdy[i]);
}

// lap_pres_c = rho * (f * tmp_c + 2.0 * lap_pres_c), float64 intermediates        (invert_pres.cpp:166-169)
__global__ void pres_source_kernel(const cpx *lap_psi, cpx *lap_pres, long long n, float rho, float f)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const cpx a = lap_psi[i], b = lap_pres[i];
    const float fa_x = __fmul_rn(f, a.x), fa_y = __fmul_rn(f, a.y);
    lap_pres[i] = mk((float)((double)rho * ((double)fa_x + 2.0 * (double)b.x)),
                     (float)((double)rho * ((double)fa_y + 2.0 * (double)b.y)));
}

__global__ void sub_ref_kernel(float *p, long long n, size_t ref)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    __shared__ float r;
    if (threadIdx.x == 0) r = p[ref];
    __syncthreads();
    // all blocks read p[ref] before any block can overwrite it only if it is excluded here;
    // the reference element itself is handled by a second launch
    if (i < n && (size_t)i != ref) p[i] = __fsub_rn(p[i], r);
}

__global__ void zero_one_kernel(float *p, size_t ref) { p[ref] = __fsub_rn(p[ref], p[ref]); }

extern "C" int xfb_invert_pres(xfb_handle h, const float *psi, float *pres, size_t ref_x, size_t ref_y, float rho, float f)
{
    if (!h || !psi || !pres) return fail(XFB_E_ARG, "null argument");
    NO_SLAB(h, "xfb_invert_pres");
    const size_t ref = ref_x + (size_t)h->nx * ref_y;     // invert_pres.cpp:182 (x + XPTS*y, as written there)
    if (ref >= h->grids) return fail(XFB_E_ARG, "reference point out of range");
    CK(cudaSetDevice(h->device));
    const int P = h->pitch;
    const long long n = (long long)h->grids, hn = (long long)h->hpad;
    const float scale = 1.0f / (float)((double)h->nx * (double)h->ny);
    const void *din;
    if (stage_in(h, psi, h->real_a, sizeof(float) * h->grids, &din)) return XFB_E_CUDA;
    // psi_c lives in t[0]; t[1..3] and jint are scratch (the stepper's prologue is invalidated)
    h->tf_valid = false;
    cpx *psi_c = h->t[0], *w1 = h->t[1], *w2 = h->t[2], *lap_pres = h->t[3];
    if (fwd2d(h, (const float *)din, h->spec_a, psi_c)) return XFB_E_CUDA;                       // :135
    // d2/dx2                                                                                      :139-140,148,153
    if (launch_pw(h, OP_GRADX, psi_c, P, w1, P, P) || launch_pw(h, OP_GRADX, w1, P, w1, P, P) ||
        launch_pw(h, OP_DEALIAS, w1, P, w1, P, P) || inv2d(h, w1, h->spec_b, h->real_a, scale, 0))
        return XFB_E_CUDA;
    // d2/dy2                                                                                      :142-143,149,154
    if (launch_pw(h, OP_GRADY, psi_c, P, w2, P, P) || launch_pw(h, OP_GRADY, w2, P, w1, P, P) ||
        launch_pw(h, OP_DEALIAS, w1, P, w1, P, P) || inv2d(h, w1, h->spec_b, h->real_b, scale, 0))
        return XFB_E_CUDA;
    // d2/dxdy = gradx(grady(psi))                                                                 :145,150,155
    if (launch_pw(h, OP_GRADX, w2, P, w1, P, P) || launch_pw(h, OP_DEALIAS, w1, P, w1, P, P) ||
        inv2d(h, w1, h->spec_b, h->real_c, scale, 0))
        return XFB_E_CUDA;
    gauss_curv_kernel<<<(unsigned)((n + 255) / 256), 256, 0, h->stream>>>(h->real_a, h->real_b, h->real_c, h->real_a, n);
    CK(cudaGetLastError()); h->launches++;
    if (fwd2d(h, h->real_a, h->spec_a, lap_pres)) return XFB_E_CUDA;                               // :161
    if (launch_pw(h, OP_LAP, psi_c, P, w1, P, P)) return XFB_E_CUDA;                               // :164
    pres_source_kernel<<<(unsigned)((hn + 255) / 256), 256, 0, h->stream>>>(w1, lap_pres, hn, rho, f);
    CK(cudaGetLastError()); h->launches++;
    if (launch_pw(h, OP_INVLAP, lap_pres, P, w1, P, P)) return XFB_E_CUDA;                         // :171
    float *dout = (float *)stage_out_target(pres, h->real_b);
    if (inv2d(h, w1, h->spec_b, dout, scale, 0)) return XFB_E_CUDA;                                // :172
    sub_ref_kernel<<<(unsigned)((n + 255) / 256), 256, 0, h->stream>>>(dout, n, ref);              // :182-185
    CK(cudaGetLastError()); h->launches++;
    zero_one_kernel<<<1, 1, 0, h->stream>>>(dout, ref);
    CK(cudaGetLastError()); h->launches++;
    return stage_out(h, pres, dout, sizeof(float) * h->grids);
}

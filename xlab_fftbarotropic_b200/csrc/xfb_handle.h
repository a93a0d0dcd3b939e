// xfb_handle.h -- the handle behind the C ABI and the helpers shared by xfb_api.cu (single GPU) and
// xfb_dist.cu (slab decomposition).
#pragma once
#include <cstdarg>
#include <cstddef>
#include <cstdio>
#include <functional>
#include <vector>

#include "../../include/xfb.h"
#include "xfb_internal.h"

namespace xfb {

int fail(int code, const char *fmt, ...);

#define CK(call)                                                                                        \
    do {                                                                                                \
        cudaError_t e__ = (call);                                                                       \
        if (e__ != cudaSuccess) return xfb::fail(XFB_E_CUDA, "%s: %s", #call, cudaGetErrorString(e__)); \
    } while (0)

#define CKL(h, call)                                                                                         \
    do {                                                                                                     \
        int e__ = (call);                                                                                    \
        if (e__ != 0) return xfb::fail(XFB_E_CUDA, "%s: %s", #call, cudaGetErrorString((cudaError_t)e__));   \
        (h)->launches++;                                                                                     \
    } while (0)

struct Team;

}  // namespace xfb

#define XFB_NREC 8          // record fields in flight (xfb_get_field_async)
#define XFB_SPECTRUM_MAX_SHELLS 65536   // nshells limit of xfb_get_energy_spectrum

struct xfb_handle_s {
    int nx, ny, hy, pitch, batch, device;
    int tw_state;        // column tile width = tile-major layout of z0/zk/acc
    float lx, ly, nu;
    // per member: real points held (rows * ny), reference half spectrum nx*(ny/2+1), padded spectral array
    size_t grids, hgrids, hpad;
    cudaStream_t stream;
    // tables
    xfb::cpx *tw;
    int twn;
    float *kx, *ky;
    double *kx2, *ky2;
    double mask_kd;
    // stepper state (per member one padded array)
    xfb::cpx *z0, *zk, *acc, *jint, *t[4];
    float *src;          // [batch][rows][ny], allocated on first use
    bool has_src;
    bool have_state;     // a vorticity/spectrum has been set
    bool tf_valid;       // t[0..3] hold the prologue of the current z0
    // scratch for the operator tier / record path (one member)
    float *real_a, *real_b, *real_c;
    xfb::cpx *spec_a, *spec_b;      // padded layout
    float *ref_a, *ref_b;           // reference layout half spectra (2*hgrids floats)
    long long launches;
    cudaStream_t rec_stream;                     // device -> pinned host copies of xfb_get_field_async
    float *rec_buf[XFB_NREC];
    cudaEvent_t rec_ready[XFB_NREC], rec_done[XFB_NREC];
    int rec_next;
    xfb::cpx *dg;        // 3 exchange arrays of the fused diagnostics path, allocated on first use
    double *espec;       // xfb_get_energy_spectrum sums: 3 + 2 * XFB_SPECTRUM_MAX_SHELLS doubles, allocated on first use
    double *bspec;       // xfb_get_spectral_budget sums: 6 + 6 * XFB_SPECTRUM_MAX_SHELLS doubles, allocated on first use
    bool warmed;         // one eager step has run (kernels configured)
    void *step_graph;    // cudaGraphExec_t of one RK4 step (step_replay), valid for graph_dt / graph_src
    float graph_dt;
    const void *graph_src;
    int graph_launches;  // launches one replay of step_graph stands for (counted while it was captured)
    // passive tracer (xfb_set_tracer), allocated on first use: state like z0/zk/acc/jint, two gradient product arrays
    xfb::cpx *c0, *ck, *cacc, *cjint, *tc[2];
    float kappa;
    bool has_tracer, tcf_valid;     // tcf_valid: tc[0..1] hold the gradient products of the current c0
    xfb::LinCoef lin;    // beta-plane, linear drag, hyperviscosity (xfb_set_linear_terms); all zero: off
    void *generic;       // non-null: grid served by the generic mixed-radix path (xfb_generic.cu), reference layout everywhere
    // ---- slab decomposition (xfb_dist.cu); nranks == 1 otherwise ------------------------------------
    // rank r holds physical rows [r*rows, (r+1)*rows) and the spectral columns of panels r*nchunks ..
    // (r+1)*nchunks-1; a panel is `pitch` (= cw) columns wide, pitch_g = pitch * nranks * nchunks.
    int rank, nranks, rows, nchunks, pitch_g, col0;
    unsigned cw_magic;
    xfb::Team *team;
    xfb::cpx *jint_recv, *tr[4];    // receive sides of the two transposes: ONE allocation (recv_block), exported over CUDA IPC
    xfb::cpx *cjint_recv, *trc[2];  // the same for the passive tracer (arrays 5, 6, 7 of recv_block)
    xfb::cpx *t_block, *recv_block; // t[0..3] back to back ; jint_recv, tr[0..3], cjint_recv, trc[0..1] back to back
    xfb::cpx *peer_recv[16];        // recv_block of every rank mapped into this process (peer-to-peer over NVLink)
    float *sync_buf;                // 1 float, reduced over all ranks as the phase barrier
    bool p2p;                       // exchange by pushes into peer_recv (else ncclSend/ncclRecv)
    bool push_sm;                   // p2p: pushes by an SM kernel (plain stores on the peer mappings) instead of the copy engines
    int push_blocks;                // CTAs per segment of the push kernel
    xfb::cpx **panel_base;          // fused row->column exchange: device table [nranks * nchunks] of the places in the ranks'
                                    // receive arrays where K-ROW writes its output panels directly (null: exchange by pushes)
    bool self_direct;               // two-level K-COL stores this rank's own row pairs straight into its tr[] arrays (no self-copy in the push)
    xfb::cpx **panel_base_c;        // the same table for the tracer's tendency (array 5 of the receive blocks)
    cudaStream_t comm_stream;
    cudaStream_t copy_stream[4];    // p2p transport: the pushes of one exchange are spread over several copy engines
    cudaEvent_t ev_copy[4], ev_fork;
    int ncopy;
    cudaEvent_t ev_chunk[16], ev_comm[2];
    // optional per-kernel timing (xfb_profile)
    bool profiling;
    std::vector<cudaEvent_t> *ev_row, *ev_col, *ev_a2a;   // pairs (begin, end)
    size_t ev_row_used, ev_col_used, ev_a2a_used;
};

namespace xfb {

cudaEvent_t next_event(std::vector<cudaEvent_t> *pool, size_t &used);
int dev_alloc(void **p, size_t bytes);
bool is_device_ptr(const void *p);

enum { OP_GRADX = 0, OP_GRADY = 1, OP_LAP = 2, OP_INVLAP = 3, OP_DEALIAS = 4, OP_COPY = 5 };

// Spectral operator chain of a record field (xfb_api.cu): ops[0] reads the state, the others run in place, then the
// inverse 2-D transform with sign `negate`.  field_ops(which) takes the field ids of include/xfb.h and returns null for
// one that is not such a chain (XFB_SRC, XFB_TFIL, XFB_DEFORM) and for any other value.  psi_second_ops are psi_xy,
// psi_xx and psi_yy, the second derivatives the strain diagnostics combine; they are not field ids a caller can ask for.
struct FieldOps {
    int nops, ops[3], negate;
};
const FieldOps *field_ops(int which);
extern const FieldOps psi_second_ops[3];

// caller buffers (xfb_api.cu): a device pointer is used in place, a host pointer goes through `dev_scratch`.
// stage_in copies host input in; stage_out_target names the buffer a result is produced in; stage_out copies it to the
// host unless it was produced in place, and then waits for the copy unless `wait` is false (the caller synchronises).
int stage_in(xfb_handle h, const void *user, void *dev_scratch, size_t bytes, const void **dev);
void *stage_out_target(const void *user, void *dev_scratch);
int stage_out(xfb_handle h, void *user, const void *dev, size_t bytes, bool wait = true);

// pointwise spectral operator on one chunk of K-COL-side columns (chunk 0 on one GPU)
int launch_pw(xfb_handle h, int op, const cpx *in, int in_pitch, cpx *out, int out_pitch, int ncols, int in_tw = 0,
              int out_tw = 0, int chunk = 0);
void fill_row(xfb_handle h, RowParams &p, int nrows);
void fill_col(xfb_handle h, ColParams &p, int chunk = 0);

// common part of xfb_create / xfb_create_dist / the loopback team
int create_impl(xfb_handle *out, int nx, int ny, float lx, float ly, float nu, int batch, int device, int rank, int nranks,
                int nchunks);
int destroy_impl(xfb_handle h);

// generic mixed-radix path (xfb_generic.cu): sizes 2^a 3^b 5^c the fused kernels do not serve, e.g. the reference's 768
bool generic_size_ok(int nx, int ny);
int generic_create(xfb_handle h);
void generic_destroy(xfb_handle h);
int generic_fwd2d(xfb_handle h, const float *real_in, cpx *tmp, cpx *spec_out);
int generic_inv2d(xfb_handle h, const cpx *spec_in, cpx *tmp, float *real_out, float scale, int negate);
int generic_one_step(xfb_handle h, float dt);
// the nonlinear tendency r2c(-u.grad(zeta) [+ src]) of the spectral state z (row-major), as one Runge-Kutta stage of
// generic_one_step forms it, into T; uses real_a, real_b, real_c, t[0], t[1], spec_a and spec_b
int generic_tendency(xfb_handle h, const cpx *z, const float *src, cpx *T);

// nsteps calls of `one_step` (one RK4 step, xfb_api.cu): the first step of a handle runs eagerly, later ones replay a
// CUDA graph captured from one call; XFB_NO_GRAPH=1, and profiling when `eager_if_profiling`, keep the eager path
int step_replay(xfb_handle h, int nsteps, float dt, bool eager_if_profiling, const std::function<int()> &one_step);

// passive tracer state (c0, ck, cacc, cjint; tc[0..1] except on generic grids), allocated and zeroed on first use
int tracer_state_alloc(xfb_handle h);

// histogram of area and |grad c|^2 over tracer bins of `n` points (xfb_api.cu); accumulates into d_area[nbins], d_grad2[nbins]
// (device, float64, zeroed by the caller); gy == nullptr: gx holds |grad c|^2
int launch_keff_hist(xfb_handle h, const float *c, const float *gx, const float *gy, long long n, int nbins, float cmin, float cmax,
                     double *d_area, double *d_grad2);
// the argument check of every histogram entry point, and the copy of the 2 * nbins device sums d to area / grad2 (host)
int keff_hist_args(int nbins, float cmin, float cmax, const double *area, const double *grad2);
int keff_hist_finish(xfb_handle h, const double *d, int nbins, double *area, double *grad2);

// filamentation time (which = XFB_TFIL) or deformation factor (XFB_DEFORM) of `n` points from psi_xy, psi_xx, psi_yy
// (xfb_api.cu); `out` may be any of the inputs: each element is read before it is written
int launch_strain(xfb_handle h, const float *pxy, const float *pxx, const float *pyy, float *out, long long n, int which);

// quadratic invariants and shell spectra (xfb_spectra.cu): one launch adds the raw sums of one state array into
// d_out[3 + 2 * nshells] (device, zeroed by the caller); _finish copies them to the host and scales them to domain means
long long shells_all(int nx, int ny, float lx, float ly);
int energy_spectrum_scratch(xfb_handle h);
int launch_energy_spectrum(xfb_handle h, const cpx *state, int nshells, double *d_out);
int energy_spectrum_finish(xfb_handle h, const double *d, int nshells, double *totals, double *e, double *z);
// argument and state checks of xfb_get_energy_spectrum (xfb_api.cu); `api` ("xfb_" or "xfb_loopback_") prefixes the entry
// points the messages name
int energy_spectrum_args(xfb_handle h, int member, int which, int nshells, const double *totals, const double *e, const double *z,
                         const char *api);
// spectral budget (xfb_spectra.cu): one launch adds the raw sums of one member into d_out[6 + 6 * nshells] (device, zeroed by
// the caller) from its state, its nonlinear tendency and its source (null: none), all three in the state's layout; _finish
// copies them to the host and scales them to rates of domain means; _args checks as energy_spectrum_args does
int spectral_budget_scratch(xfb_handle h);
int launch_spectral_budget(xfb_handle h, const cpx *state, const cpx *tend, const cpx *src, int nshells, double *d_out);
int spectral_budget_finish(xfb_handle h, const double *d, int nshells, double *totals, double *budget);
int spectral_budget_args(xfb_handle h, int member, int nshells, const double *totals, const double *budget, const char *api);

// slab paths (xfb_dist.cu)
int dist_keff_hist(xfb_handle h, int nbins, float cmin, float cmax, double *area, double *grad2, bool tracer_state);
int dist_diagnostics(xfb_handle h, float *tfil_rows, float *deform_rows);
int dist_set_vorticity(xfb_handle h, const float *vort_rows);
int dist_set_tracer(xfb_handle h, const float *tracer_rows);
int dist_step(xfb_handle h, int nsteps, float dt);
int dist_get_field(xfb_handle h, int which, float *out_rows);
int dist_energy_spectrum(xfb_handle h, int which, int nshells, double *totals, double *e, double *z);
int dist_spectral_budget(xfb_handle h, int nshells, double *totals, double *budget);
void dist_release(xfb_handle h);

}  // namespace xfb

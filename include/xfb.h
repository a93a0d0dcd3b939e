/* xfb.h -- C ABI of the B200-native backend for XLab-FFTBarotropic's pseudospectral RK4 step.
 *
 * This is the drop-in boundary: plain pointers and sizes, no C++/torch types.  Every entry point
 * names the reference interface it replaces (paths under the reference tree, file:line).
 *
 * Conventions
 *   - every function returns 0 on success, a negative XFB_E_* code on failure;
 *     xfb_last_error() returns a thread-local message for the last failure.
 *   - the library never calls exit()/abort() and has NO CPU fallback: without a CUDA device
 *     xfb_create fails with XFB_E_CUDA.
 *   - data pointers may be HOST or DEVICE pointers (detected with cudaPointerGetAttributes);
 *     host pointers imply a copy on the handle's stream and a synchronisation before return.
 *   - layouts are the reference's (src/configuration.hpp:31-32):
 *       real field   : float[nx*ny],  IDX(i,j)  = ny*i + j         (i = x slow, j = y fast)
 *       half spectrum: float[2*nx*(ny/2+1)] interleaved re,im, HIDX(i,j) = (ny/2+1)*i + j
 *   - one handle per host thread; calls on one handle are ordered on its CUDA stream.
 */
#ifndef XFB_H
#define XFB_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct xfb_handle_s *xfb_handle;

enum {
    XFB_OK = 0,
    XFB_E_ARG = -1,      /* bad argument (null pointer, member out of range, ...) */
    XFB_E_SIZE = -2,     /* grid size not supported by the kernels */
    XFB_E_CUDA = -3,     /* CUDA runtime error (message in xfb_last_error) */
    XFB_E_STATE = -4,    /* call order (e.g. step before set_vorticity) */
    XFB_E_NCCL = -5      /* NCCL error or libnccl.so.2 not loadable (slab-decomposed handles only) */
};

/* fields of xfb_get_field */
enum {
    XFB_VORT = 0,        /* vort_step_N.bin      src/main.cpp:273-281 */
    XFB_PSI = 1,         /* psi_step_N.bin       src/main.cpp:183-192 */
    XFB_U = 2,           /* u_step_N.bin         src/main.cpp:198-209 */
    XFB_V = 3,           /* v_step_N.bin         src/main.cpp:212-222 */
    XFB_SRC = 4,         /* vort_src_input_step_N.bin  src/main.cpp:268-270 */
    XFB_TFIL = 5,        /* filamentation time   README.md:5 (Rozoff et al. 2006) */
    XFB_DEFORM = 6,      /* deformation factor   README.md:7 */
    XFB_DVORTDX = 7,     /* dvortdx_step_N.bin   src/main.cpp:156-162 (OUTPUT_GRAD_VORT) */
    XFB_DVORTDY = 8,     /* dvortdy_step_N.bin   src/main.cpp:170-176 */
    XFB_TRACER = 9       /* passive tracer of xfb_set_tracer (no reference counterpart) */
};

/* tables of xfb_get_table (src/fftwfop.cpp:5-79) */
enum {
    XFB_TAB_GRADX = 0,   /* gradx_coe[nx]                     fftwfop.cpp:15-20 */
    XFB_TAB_GRADY = 1,   /* grady_coe[ny/2+1]                 fftwfop.cpp:22-24 */
    XFB_TAB_LAP = 2,     /* laplacian_coe[nx*(ny/2+1)]        fftwfop.cpp:40-54 */
    XFB_TAB_LAPINV = 3,  /* laplacian_coe_inverse[...]        fftwfop.cpp:40-54, (0,0) = 1 */
    XFB_TAB_MASK = 4     /* dealiasing_mask[...]              fftwfop.cpp:57-68 */
};

const char *xfb_last_error(void);

/* ---- lifetime: replaces the global `fftwf_operation<XPTS,YPTS> fop(LX, LY)` (src/main.cpp:33,
 * src/invert_pres.cpp:39; constructor src/fftwfop.cpp:5-79), the fftwf_malloc block and the eight
 * fftwf_plan_dft_{r2c,c2r}_2d plans of src/main.cpp:103-135.  `batch` ensemble members share the
 * tables; `device` is the CUDA device ordinal. */
int xfb_create(xfb_handle *h, int nx, int ny, float lx, float ly, float nu, int batch, int device);
int xfb_destroy(xfb_handle h);
int xfb_sync(xfb_handle h);

/* ---- operator tier: the five methods of class fftwf_operation (src/fftwfop.hpp:20-24) ---------
 * in/out: half spectra of ONE field.  out may equal in for laplacian / invert_laplacian /
 * dealias (the reference calls dealiase in place, src/invert_pres.cpp:148-150); gradx/grady
 * also allow it here (the reference's do not). */
int xfb_gradx(xfb_handle h, const float *in, float *out);            /* src/fftwfop.cpp:87-94   */
int xfb_grady(xfb_handle h, const float *in, float *out);            /* src/fftwfop.cpp:96-103  */
int xfb_laplacian(xfb_handle h, const float *in, float *out);        /* src/fftwfop.cpp:105-110 */
int xfb_invert_laplacian(xfb_handle h, const float *in, float *out); /* src/fftwfop.cpp:112-117 */
int xfb_dealias(xfb_handle h, const float *in, float *out);          /* src/fftwfop.cpp:119-124 */
int xfb_get_table(xfb_handle h, int which, float *out);              /* src/fftwfop.cpp:5-79 (host pointer only) */

/* ---- 2-D real transforms: replace fftwf_execute on the raw FFTW plans (src/main.cpp:126-135,
 * 154,168,186,200,214,237,256,275; src/invert_pres.cpp:100-107,135,153-155,161,172).
 * Unnormalised like FFTW.  Unlike FFTW's c2r, the input is never destroyed. */
int xfb_r2c(xfb_handle h, const float *real_in, float *spec_out);
int xfb_c2r(xfb_handle h, const float *spec_in, float *real_out);

/* ---- stepper tier: device-resident state, replaces the RK4 loop of src/main.cpp:260-317 -------*/
/* readField + step 01 forward transform (src/main.cpp:143-144,256) */
int xfb_set_vorticity(xfb_handle h, int member, const float *vort);
/* raw spectral state, reference layout (exact restart; no reference equivalent) */
int xfb_set_spectrum(xfb_handle h, int member, const float *spec);
int xfb_get_spectrum(xfb_handle h, int member, float *spec);
/* vort_src (src/main.cpp:110,226; src/vorticity_source.cpp:112-133). NULL clears it. */
int xfb_set_source(xfb_handle h, int member, const float *src);
/* nsteps RK4 steps of all members: getDvortdt x4, dealiase, evolve, final combine
 * (src/main.cpp:286-317).  Asynchronous; no record I/O. */
int xfb_step(xfb_handle h, int nsteps, float dt);
/* record-step fields of the current state (src/main.cpp:266-282,183-222) and diagnostics */
int xfb_get_field(xfb_handle h, int member, int which, float *out);
/* asynchronous record output: the field is formed on the handle's stream and copied to a PINNED host buffer
 * (xfb_host_alloc) on a second stream; the call returns at once and later xfb_step calls overlap the copy.
 * xfb_wait_field(ticket) blocks until that buffer is complete.  Up to 8 fields in flight. */
int xfb_host_alloc(float **p, size_t nfloats);
int xfb_host_free(float *p);
int xfb_get_field_async(xfb_handle h, int member, int which, float *pinned_out, int *ticket);
int xfb_wait_field(xfb_handle h, int ticket);
/* filamentation time and deformation factor together, from one set of second derivatives of psi (the two
 * XFB_TFIL / XFB_DEFORM calls of xfb_get_field recompute them); either output may be NULL.  Slab-decomposed handles:
 * the LOCAL rows, collective. */
int xfb_get_diagnostics(xfb_handle h, int member, float *tfil, float *deform);
/* effective-diffusivity histograms (README.md:6, Hendricks & Schubert 2009): per bin of the
 * tracer zeta in [cmin,cmax): area and integral of |grad zeta|^2 (float64[nbins] each, host).  Slab-decomposed
 * handles: every rank bins its rows, ONE ncclAllReduce sums the 2 * nbins values, every rank receives the whole-domain
 * histograms; collective. */
int xfb_get_keff_hist(xfb_handle h, int member, int nbins, float cmin, float cmax, double *area, double *grad2);
/* quadratic invariants of the current state and their isotropic shell spectra (no reference counterpart;
 * definitions in DESIGN.md).  which = XFB_VORT (vorticity) or XFB_TRACER (the passive tracer, same forms).
 * totals[3] = {E, Z, P}: domain means, float64.  nshells == 0: totals only (e, z may be NULL); else e[nshells],
 * z[nshells] = shell sums of E and Z.  Host pointers only.  Reads the state only: later steps are unaffected.
 * Slab-decomposed handles: collective, every rank receives the whole-domain result. */
int xfb_get_energy_spectrum(xfb_handle h, int member, int which, int nshells, double *totals, double *e, double *z);
/* spectral budget of the vorticity (no reference counterpart; definitions in DESIGN.md section 3): the rates that the
 * nonlinear transfer T, the forcing F (xfb_set_source; zero without one) and the dissipation D (nu, mu and the
 * hyperviscosity of xfb_set_linear_terms) give the energy E and the enstrophy Z of xfb_get_energy_spectrum, per mode
 * w_j M Re(conj(Z_k) X_k) / Np^2 (over k^2 for E) inside the dealiasing mask M, with X = the r2c of -u.grad(zeta) formed as
 * the stepper's first Runge-Kutta stage forms it, the r2c of the source, and (-nu k^2 - mu - nu_h k^(2 order)) Z_k.  The
 * beta term rotates the phase of each mode and adds nothing to E or Z: it is no term of the budget.  totals[6] = domain
 * sums over all modes, in XFB_BUDGET_* order; nshells == 0: totals only (budget may be NULL), else
 * budget[q * nshells + s] = the sum of quantity q over shell s (the shells of xfb_get_energy_spectrum, modes beyond
 * nshells count in the totals only).  Host pointers only.  Vorticity only.  Reads the state and leaves later steps
 * bit-identical (it may form the products the next step would form first).  Slab-decomposed handles: collective,
 * every rank receives the whole-domain result. */
enum { XFB_BUDGET_TE = 0, XFB_BUDGET_FE = 1, XFB_BUDGET_DE = 2, XFB_BUDGET_TZ = 3, XFB_BUDGET_FZ = 4, XFB_BUDGET_DZ = 5,
       XFB_BUDGET_N = 6 };
int xfb_get_spectral_budget(xfb_handle h, int member, int nshells, double *totals, double *budget);

/* ---- passive tracer (SURVEY.md section 8 (f-4); the reference has none) -------------------------
 * dc/dt = -u c_x - v c_y + kappa lap(c), advanced by xfb_step together with the vorticity: every Runge-Kutta stage
 * uses that stage's velocity, the tendency is dealiased and combined exactly like the vorticity's
 * (src/main.cpp:225-251,286-312 with c for vort and kappa for NU), so a tracer equal to the vorticity with
 * kappa == nu and no forcing stays bit-identical to it.  `tracer` is nx*ny floats, host or device; kappa is one value
 * per handle (the last call's).  Power-of-two grids 256 .. 16384 (fused kernels), the generic mixed-radix sizes (e.g. 768) and
 * slab-decomposed handles (`tracer` = the LOCAL rows, collective; the tracer's tendency and its two gradient products
 * travel through three more receive arrays of the same CUDA-IPC block).
 * Read back with xfb_get_field(..., XFB_TRACER, ...); effective-diffusivity histograms over the tracer: */
int xfb_set_tracer(xfb_handle h, int member, const float *tracer, float kappa);
int xfb_get_tracer_keff_hist(xfb_handle h, int member, int nbins, float cmin, float cmax, double *area, double *grad2);

/* ---- linear terms (the reference has only nu lap(zeta)) -------------------------------------------
 * d(zeta)/dt = -u.grad(zeta) + src + nu lap(zeta) - beta v - mu zeta - nu_h (-lap)^order zeta, v = d(psi)/dx, x the slow
 * index: beta-plane (beta > 0: f grows with y; Rossby waves propagate westward), linear drag, hyperviscosity.  Per mode
 * the step adds L(k) Z_k inside the dealiasing mask, L(k) = -mu - nu_h k^(2 order) + i beta kx / k^2 (DESIGN.md section 3).
 * Acts on every member of the handle; the passive tracer keeps kappa lap(c) only.  order 1..8, mu >= 0, nu_h >= 0, all
 * finite (beta may be negative), and nu_h k_c^(2 order) must be a normal float (k_c: the grid's largest wavenumber), else
 * XFB_E_ARG.  All zeros switches the terms off.  Slab-decomposed handles: per rank, no communication -- every rank must
 * pass the same values. */
int xfb_set_linear_terms(xfb_handle h, float beta, float mu, float nu_h, int order);

/* ---- pressure inversion: replaces the loop body of src/invert_pres.cpp:132-187 ---------------*/
int xfb_invert_pres(xfb_handle h, const float *psi, float *pres, size_t ref_x, size_t ref_y, float rho, float f);

/* ---- slab decomposition of one large grid over the GPUs of a node ------------------------------
 * No reference equivalent (src/main.cpp is single-threaded); SURVEY.md section 8(e).
 * Rank r of `nranks` holds the physical rows [row0, row0+rows) and, in spectral space, `cols`
 * columns starting at col0, cut into `nchunks` chunks of chunk_cols columns (the unit of the
 * compute/communication overlap); every 2-D transform is a local 1-D pass, an all-to-all over
 * NVLink and the other local 1-D pass.  xfb_slab_partition is pure host arithmetic. */
int xfb_slab_partition(int nx, int ny, int nranks, int nchunks, int rank, int *row0, int *rows, int *col0, int *cols,
                       int *chunk_cols, int *pitch_global);
/* one process per GPU: rank 0 calls xfb_nccl_unique_id and hands the 128 bytes to the other ranks
 * (MPI, torch.distributed, a file ...); all ranks then call xfb_create_dist collectively.
 * On such a handle xfb_set_vorticity / xfb_set_source / xfb_get_field take and return the LOCAL
 * rows [rows][ny] and are collective, like xfb_step; the operator tier is not available. */
int xfb_nccl_unique_id(char *id128);
int xfb_create_dist(xfb_handle *h, int nx, int ny, float lx, float ly, float nu, int device, int rank, int nranks,
                    int nchunks, const char *id128);
/* transport of a slab handle: 0 none (one rank), 1 grouped ncclSend/ncclRecv (XFB_SLAB_NCCL=1), 2 copy-engine
 * pushes / 3 SM push kernel into the peers' receive arrays mapped over CUDA IPC (XFB_SLAB_PUSH=ce|sm) */
int xfb_slab_transport(xfb_handle h);
/* 1 if K-ROW stores its output panels straight into the peers' receive arrays (fused row -> column transpose; P2P
 * transports only, XFB_SLAB_FUSED=0 turns it off), else 0 */
int xfb_slab_fused(xfb_handle h);
/* summed milliseconds of the all-to-all exchanges since xfb_profile(h, 1) (NCCL handles) */
int xfb_profile_read_a2a(xfb_handle h, double *a2a_ms, long long *exchanges);
/* loopback team: all ranks of a slab decomposition in ONE process on ONE device, exchanging by
 * device copies.  Same kernels and indexing as the NCCL path; exists so the decomposition can be
 * verified on a single GPU.  Fields are full [nx][ny] host arrays. */
typedef struct xfb_loopback_s *xfb_loopback;
int xfb_loopback_create(xfb_loopback *t, int nx, int ny, float lx, float ly, float nu, int device, int nranks, int nchunks);
int xfb_loopback_destroy(xfb_loopback t);
int xfb_loopback_set_vorticity(xfb_loopback t, const float *vort);
int xfb_loopback_set_source(xfb_loopback t, const float *src);
int xfb_loopback_set_tracer(xfb_loopback t, const float *tracer, float kappa);
int xfb_loopback_set_linear_terms(xfb_loopback t, float beta, float mu, float nu_h, int order);
int xfb_loopback_step(xfb_loopback t, int nsteps, float dt);
int xfb_loopback_get_field(xfb_loopback t, int which, float *out);
int xfb_loopback_get_diagnostics(xfb_loopback t, float *tfil, float *deform);
int xfb_loopback_get_keff_hist(xfb_loopback t, int nbins, float cmin, float cmax, double *area, double *grad2);
int xfb_loopback_get_energy_spectrum(xfb_loopback t, int which, int nshells, double *totals, double *e, double *z);
int xfb_loopback_get_spectral_budget(xfb_loopback t, int nshells, double *totals, double *budget);
long long xfb_loopback_launch_count(xfb_loopback t);

/* ---- introspection --------------------------------------------------------------------------*/
/* number of CUDA kernels this handle has launched so far */
long long xfb_launch_count(xfb_handle h);
/* cudaStream_t of the handle, as void* (for event timing by the caller) */
void *xfb_stream(xfb_handle h);
/* per-kernel CUDA-event timing of the stepper's two kernels (K-ROW = ROW_JAC, K-COL = COL_STEP):
 * xfb_profile(h, 1) resets the counters and brackets every stepper launch with events on the
 * handle's stream; xfb_profile_read synchronises and returns summed milliseconds and launch counts. */
int xfb_profile(xfb_handle h, int enable);
int xfb_profile_read(xfb_handle h, double *row_ms, long long *row_launches, double *col_ms, long long *col_launches);
/* 1 if (nx, ny) is served by the fused power-of-two kernels, 2 if by the generic mixed-radix
 * path, 0 if unsupported */
int xfb_size_supported(int nx, int ny);

#ifdef __cplusplus
}
#endif
#endif

// xfb_generic.cu -- grids the fused kernels do not serve (any NX, NY = 2^a 3^b 5^c up to 4096, NY even): the
// reference's own default NPTS = 768 = 3 * 256 (src/configuration.hpp:18) lands here.
//
// This path keeps the reference's structure (src/main.cpp:146-317) one kernel per loop: pointwise spectral
// operators (the bit-exact ones of xfb_api.cu), a mixed-radix Stockham line FFT in shared memory for the two
// directions of the 2-D transforms, the Jacobian loop, the RK updates.  It is a completeness path -- small
// grids that live in L2 -- not the roofline path; xfb_size_supported() reports 2 for it.
// Spectral arrays are in the reference layout [NX][NY/2+1] (pitch = NY/2+1, no pair interleave, no tiling).
#include <cstring>
#include <vector>

#include "xfb_handle.h"

namespace xfb {

// ---- mixed-radix Stockham FFT of `nl` lines of length n held in shared memory ---------------------------------
// a: input lines [nl][n], b: scratch of the same size; returns the buffer that holds the result.
// tw[k] = exp(-2 pi i k / n).  SIGN = +1: forward (e^{-i}), -1: inverse (e^{+i}), unnormalised.
template <int SIGN>
__device__ cpx *gen_fft(cpx *a, cpx *b, const int n, const int nl, const int *__restrict__ fac, const int nfac,
                        const cpx *__restrict__ tw, const int tpl)
{
    // tpl threads work on one line (tpl divides blockDim.x): no per-butterfly integer division
    const int line0 = threadIdx.x / tpl, lane = threadIdx.x - line0 * tpl, lpb = blockDim.x / tpl;
    int ns = 1;
    for (int f = 0; f < nfac; ++f) {
        const int r = fac[f], m = n / r;              // m butterflies per line
        const int tstep = n / (ns * r);               // twiddle exp(-2 pi i s k / (ns r)) = tw[s * k * tstep], index < n
        const bool pow2 = (ns & (ns - 1)) == 0;       // radices 4 and 2 come first: ns stays a power of two for them
        for (int line = line0; line < nl; line += lpb) {
            const cpx *src = a + (size_t)line * n;
            cpx *dl = b + (size_t)line * n;
            for (int j = lane; j < m; j += tpl) {
                const int k = pow2 ? (j & (ns - 1)) : (j % ns);
                cpx *dst = dl + (j - k) * r + k;
                cpx x[5];
                x[0] = src[j];
                for (int s = 1; s < r; ++s) {
                    cpx v = src[j + s * m];
                    if (k > 0) {
                        cpx w = tw[s * k * tstep];
                        if (SIGN < 0) w.y = -w.y;
                        v = cmul(v, w);
                    }
                    x[s] = v;
                }
                if (r == 2) {
                    dst[0] = cadd(x[0], x[1]);
                    dst[ns] = csub(x[0], x[1]);
                } else if (r == 4) {
                    const cpx t0 = cadd(x[0], x[2]), t1 = csub(x[0], x[2]), t2 = cadd(x[1], x[3]);
                    cpx t3 = csub(x[1], x[3]);
                    t3 = (SIGN > 0) ? mul_negi(t3) : mul_i(t3);
                    dst[0] = cadd(t0, t2);
                    dst[ns] = cadd(t1, t3);
                    dst[2 * ns] = csub(t0, t2);
                    dst[3 * ns] = csub(t1, t3);
                } else if (r == 3) {
                    // y0 = x0 + x1 + x2 ; y1,2 = x0 - (x1 + x2)/2 -+ i (sqrt(3)/2)(x1 - x2)   (forward; inverse swaps)
                    const cpx t1 = cadd(x[1], x[2]);
                    const cpx t2 = mk(x[0].x - 0.5f * t1.x, x[0].y - 0.5f * t1.y);
                    const cpx d = csub(x[1], x[2]);
                    cpx t3 = mk(0.86602540378443864676f * d.x, 0.86602540378443864676f * d.y);
                    t3 = (SIGN > 0) ? mul_negi(t3) : mul_i(t3);
                    dst[0] = cadd(x[0], t1);
                    dst[ns] = cadd(t2, t3);
                    dst[2 * ns] = csub(t2, t3);
                } else {
                    // radix 5: c1 = cos(2 pi/5), c2 = cos(4 pi/5), s1 = sin(2 pi/5), s2 = sin(4 pi/5)
                    const float c1 = 0.30901699437494742410f, c2 = -0.80901699437494742410f;
                    const float s1 = 0.95105651629515357212f, s2 = 0.58778525229247312917f;
                    const cpx a1 = cadd(x[1], x[4]), a2 = cadd(x[2], x[3]), b1 = csub(x[1], x[4]), b2 = csub(x[2], x[3]);
                    const cpx p1 = mk(x[0].x + c1 * a1.x + c2 * a2.x, x[0].y + c1 * a1.y + c2 * a2.y);
                    const cpx p2 = mk(x[0].x + c2 * a1.x + c1 * a2.x, x[0].y + c2 * a1.y + c1 * a2.y);
                    cpx q1 = mk(s1 * b1.x + s2 * b2.x, s1 * b1.y + s2 * b2.y);
                    cpx q2 = mk(s2 * b1.x - s1 * b2.x, s2 * b1.y - s1 * b2.y);
                    q1 = (SIGN > 0) ? mul_negi(q1) : mul_i(q1);
                    q2 = (SIGN > 0) ? mul_negi(q2) : mul_i(q2);
                    dst[0] = mk(x[0].x + a1.x + a2.x, x[0].y + a1.y + a2.y);
                    dst[ns] = cadd(p1, q1);
                    dst[2 * ns] = cadd(p2, q2);
                    dst[3 * ns] = csub(p2, q2);
                    dst[4 * ns] = csub(p1, q1);
                }
            }
        }
        __syncthreads();
        cpx *t = a; a = b; b = t;
        ns *= r;
    }
    return a;
}

struct GenParams {
    int nx, ny, hy;
    int nfx, nfy;
    int facx[24], facy[24];
    const cpx *twx, *twy;
};

// rows: real line -> half spectrum (complex transform of the real line, bins 0 .. NY/2 kept)   main.cpp:126-127,237,256
__global__ void gen_rows_r2c(const GenParams g, const float *__restrict__ in, cpx *__restrict__ out)
{
    extern __shared__ __align__(16) unsigned char smem[];
    cpx *a = reinterpret_cast<cpx *>(smem), *b = a + g.ny;
    const size_t row = blockIdx.x;
    for (int j = threadIdx.x; j < g.ny; j += blockDim.x) a[j] = mk(in[row * g.ny + j], 0.f);
    __syncthreads();
    const cpx *r = gen_fft<1>(a, b, g.ny, 1, g.facy, g.nfy, g.twy, blockDim.x);
    for (int j = threadIdx.x; j < g.hy; j += blockDim.x) out[row * g.hy + j] = r[j];
}

// rows: half spectrum -> real line, unnormalised * scale; Im of the DC and Nyquist bins ignored like FFTW's c2r
// div != 0: the result is DIVIDED by div = (float)GRIDS like fftwf_backward_normalize (main.cpp:37-41) -- a multiplication
// by 1/GRIDS differs by 1 ulp on grids that are not powers of two (768^2) --, then multiplied by scale (+-1)
__global__ void gen_rows_c2r(const GenParams g, const cpx *__restrict__ in, float *__restrict__ out, const float scale,
                             const float div)
{
    extern __shared__ __align__(16) unsigned char smem[];
    cpx *a = reinterpret_cast<cpx *>(smem), *b = a + g.ny;
    const size_t row = blockIdx.x;
    for (int j = threadIdx.x; j < g.hy; j += blockDim.x) {
        cpx v = in[row * g.hy + j];
        if (j == 0 || j == g.ny / 2) v.y = 0.f;
        a[j] = v;
        if (j > 0 && j < g.ny / 2) a[g.ny - j] = cconj(v);
    }
    __syncthreads();
    const cpx *r = gen_fft<-1>(a, b, g.ny, 1, g.facy, g.nfy, g.twy, blockDim.x);
    for (int j = threadIdx.x; j < g.ny; j += blockDim.x) {
        const float x = (div != 0.0f) ? __fdiv_rn(r[j].x, div) : r[j].x;
        out[row * g.ny + j] = __fmul_rn(x, scale);
    }
}

// columns: complex transform along x for a tile of w adjacent columns
template <int SIGN>
__global__ void gen_cols(const GenParams g, const cpx *__restrict__ in, cpx *__restrict__ out, const int w)
{
    extern __shared__ __align__(16) unsigned char smem[];
    cpx *a = reinterpret_cast<cpx *>(smem), *b = a + (size_t)w * g.nx;
    const int j0 = blockIdx.x * w;
    const int wl = (g.hy - j0 < w) ? g.hy - j0 : w;
    for (int idx = threadIdx.x; idx < g.nx * wl; idx += blockDim.x) {
        const int i = idx / wl, c = idx - i * wl;
        a[(size_t)c * g.nx + i] = in[(size_t)i * g.hy + j0 + c];
    }
    __syncthreads();
    const cpx *r = gen_fft<SIGN>(a, b, g.nx, wl, g.facx, g.nfx, g.twx, blockDim.x / w);
    for (int idx = threadIdx.x; idx < g.nx * wl; idx += blockDim.x) {
        const int i = idx / wl, c = idx - i * wl;
        out[(size_t)i * g.hy + j0 + c] = r[(size_t)c * g.nx + i];
    }
}

// dvortdt = -u dvortdx - v dvortdy + vort_src with u already negated                              main.cpp:201,225-227
__global__ void gen_jacobian(const float *mu, const float *zx, const float *v, const float *zy, const float *src, float *out,
                             const long long n)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    // reference: u[i] = -u[i]; then  - u*dvortdx - v*dvortdy + src, evaluated left to right in float
    const float u = mu[i];                        // c2r result already multiplied by -1 (negate flag)
    float r = __fsub_rn(__fmul_rn(-u, zx[i]), __fmul_rn(v[i], zy[i]));
    if (src) r = __fadd_rn(r, src[i]);
    out[i] = r;
}

// rk = mask * (T + nu * lap * Z_k); RK bookkeeping exactly as the fused epilogue (xfb_colt.cuh)   main.cpp:240-251,296-312
// LIN: + L(k) Z_k inside the mask (xfb_set_linear_terms; kx from the gradx table, k^2 = -lap)
template <bool LIN>
__global__ void gen_stage(const cpx *T, cpx *z0, cpx *zk, cpx *acc, const int nx, const int hy, const double *kx2, const double *ky2,
                          const double mask_kd, const float nu, const float dt, const float dt_stage, const int stage,
                          const float *kx, const LinCoef lin)
{
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)nx * hy) return;
    const int i = (int)(idx / hy), j = (int)(idx % hy);
    const cpx zkv = (stage == 1) ? z0[idx] : zk[idx];
    const float lap = lap_coe(kx2[i], ky2[j]);
    float tx = __fadd_rn(T[idx].x, __fmul_rn(__fmul_rn(zkv.x, lap), nu));
    float ty = __fadd_rn(T[idx].y, __fmul_rn(__fmul_rn(zkv.y, lap), nu));
    if constexpr (LIN) {
        const cpx l = lin_term(lin, kx[i], -lap, zkv);
        tx = __fadd_rn(tx, l.x);
        ty = __fadd_rn(ty, l.y);
    }
    const long long ii = (i <= nx / 2) ? i : nx - i;
    const float m = ((double)(ii * ii + (long long)j * j) >= mask_kd) ? 0.0f : 1.0f;
    const float rx = __fmul_rn(tx, m), ry = __fmul_rn(ty, m);
    const cpx z0v = z0[idx];
    if (stage == 4) {
        const cpx av = acc[idx];
        z0[idx] = mk(__fadd_rn(z0v.x, __fdiv_rn(__fmul_rn(__fadd_rn(av.x, rx), dt), 6.0f)),
                     __fadd_rn(z0v.y, __fdiv_rn(__fmul_rn(__fadd_rn(av.y, ry), dt), 6.0f)));
    } else {
        if (stage == 1) acc[idx] = mk(rx, ry);
        else {
            const cpx av = acc[idx];
            acc[idx] = mk(__fadd_rn(av.x, __fmul_rn(2.0f, rx)), __fadd_rn(av.y, __fmul_rn(2.0f, ry)));
        }
        zk[idx] = mk(__fadd_rn(z0v.x, __fmul_rn(rx, dt_stage)), __fadd_rn(z0v.y, __fmul_rn(ry, dt_stage)));
    }
}

// ---- host side ------------------------------------------------------------------------------------------------
struct GenericPlan {
    GenParams g;
    cpx *twx, *twy;
    int cols_w, row_threads;
    size_t smem_rows, smem_cols;
};

static bool factor(int n, int *fac, int *nfac)
{
    int k = 0;
    while (n % 4 == 0) { fac[k++] = 4; n /= 4; }
    while (n % 2 == 0) { fac[k++] = 2; n /= 2; }
    while (n % 3 == 0) { fac[k++] = 3; n /= 3; }
    while (n % 5 == 0) { fac[k++] = 5; n /= 5; }
    *nfac = k;
    return n == 1 && k <= 24;
}

bool generic_size_ok(int nx, int ny)
{
    int f[24], nf;
    if (nx < 8 || ny < 8 || nx > 4096 || ny > 4096 || (ny & 1) || (nx & 1)) return false;
    return factor(nx, f, &nf) && factor(ny, f, &nf);
}

static int make_table(cpx **dev, int n)
{
    std::vector<float2> tw(n);
    for (int k = 0; k < n; ++k) {
        const double a = -2.0 * M_PI * (double)k / (double)n;
        tw[k] = make_float2((float)cos(a), (float)sin(a));
    }
    if (dev_alloc((void **)dev, sizeof(float2) * n)) return XFB_E_CUDA;
    CK(cudaMemcpy(*dev, tw.data(), sizeof(float2) * n, cudaMemcpyHostToDevice));
    return 0;
}

int generic_create(xfb_handle h)
{
    GenericPlan *P = new GenericPlan();
    memset(P, 0, sizeof(*P));
    P->g.nx = h->nx; P->g.ny = h->ny; P->g.hy = h->hy;
    if (!factor(h->nx, P->g.facx, &P->g.nfx) || !factor(h->ny, P->g.facy, &P->g.nfy)) { delete P; return fail(XFB_E_SIZE, "bad generic size"); }
    if (make_table(&P->twx, h->nx) || make_table(&P->twy, h->ny)) return XFB_E_CUDA;
    P->g.twx = P->twx; P->g.twy = P->twy;
    P->smem_rows = 2 * sizeof(cpx) * h->ny;
    // column tile width: 4 columns (32-byte rows) unless that leaves fewer than two CTAs per SM -- these grids live in
    // L2, parallelism matters more than sector efficiency; always a power of two so that it divides the block size
    int w = 4;
    while (w > 1 && (2 * sizeof(cpx) * (size_t)w * h->nx > 100 * 1024 || (h->hy + w - 1) / w < 2 * 148)) w /= 2;
    P->cols_w = w;
    P->row_threads = (h->ny >= 512) ? 256 : 128;
    P->smem_cols = 2 * sizeof(cpx) * (size_t)w * h->nx;
    CK(cudaFuncSetAttribute(gen_rows_r2c, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)P->smem_rows));
    CK(cudaFuncSetAttribute(gen_rows_c2r, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)P->smem_rows));
    CK(cudaFuncSetAttribute(gen_cols<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)P->smem_cols));
    CK(cudaFuncSetAttribute(gen_cols<-1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)P->smem_cols));
    h->generic = P;
    return 0;
}

void generic_destroy(xfb_handle h)
{
    GenericPlan *P = (GenericPlan *)h->generic;
    if (!P) return;
    cudaFree(P->twx);
    cudaFree(P->twy);
    delete P;
    h->generic = nullptr;
}

#define GLAUNCH(h, expr)                                                                          \
    do {                                                                                          \
        expr;                                                                                     \
        cudaError_t e__ = cudaGetLastError();                                                     \
        if (e__ != cudaSuccess) return fail(XFB_E_CUDA, "%s: %s", #expr, cudaGetErrorString(e__)); \
        (h)->launches++;                                                                          \
    } while (0)

int generic_fwd2d(xfb_handle h, const float *real_in, cpx *tmp, cpx *spec_out)
{
    GenericPlan *P = (GenericPlan *)h->generic;
    const int tiles = (h->hy + P->cols_w - 1) / P->cols_w;
    GLAUNCH(h, (gen_rows_r2c<<<h->nx, P->row_threads, P->smem_rows, h->stream>>>(P->g, real_in, tmp)));
    GLAUNCH(h, (gen_cols<1><<<tiles, 256, P->smem_cols, h->stream>>>(P->g, tmp, spec_out, P->cols_w)));
    return 0;
}

int generic_inv2d(xfb_handle h, const cpx *spec_in, cpx *tmp, float *real_out, float scale, int negate)
{
    GenericPlan *P = (GenericPlan *)h->generic;
    const int tiles = (h->hy + P->cols_w - 1) / P->cols_w;
    GLAUNCH(h, (gen_cols<-1><<<tiles, 256, P->smem_cols, h->stream>>>(P->g, spec_in, tmp, P->cols_w)));
    // the reference normalisation is a division by (float)GRIDS: keep that expression when the caller asks for 1/GRIDS
    const float grids = (float)((double)h->nx * (double)h->ny);
    const bool norm = (scale == 1.0f / grids);
    const float mul = norm ? 1.0f : scale;
    GLAUNCH(h, (gen_rows_c2r<<<h->nx, P->row_threads, P->smem_rows, h->stream>>>(P->g, tmp, real_out, negate ? -mul : mul,
                                                                                  norm ? grids : 0.0f)));
    return 0;
}

int generic_tendency(xfb_handle h, const cpx *z, const float *src, cpx *T)
{
    const int P = h->hy;
    const long long n = (long long)h->grids;
    const float scale = 1.0f / (float)((double)h->nx * (double)h->ny);
    const unsigned gb = (unsigned)((n + 255) / 256);
    float *fa = h->real_a, *fb = h->real_b, *fc = h->real_c, *fd = (float *)h->t[0];      // dvortdx, dvortdy, -u, v
    cpx *tmp = h->spec_a, *tmp2 = h->spec_b, *psi = h->t[1];
    if (launch_pw(h, OP_GRADX, z, P, tmp, P, P) || generic_inv2d(h, tmp, tmp2, fa, scale, 0)) return XFB_E_CUDA;       // :151-154
    if (launch_pw(h, OP_GRADY, z, P, tmp, P, P) || generic_inv2d(h, tmp, tmp2, fb, scale, 0)) return XFB_E_CUDA;       // :165-168
    if (launch_pw(h, OP_INVLAP, z, P, psi, P, P)) return XFB_E_CUDA;                                                    // :179
    if (launch_pw(h, OP_GRADY, psi, P, tmp, P, P) || generic_inv2d(h, tmp, tmp2, fc, scale, 1)) return XFB_E_CUDA;     // :198-201
    if (launch_pw(h, OP_GRADX, psi, P, tmp, P, P) || generic_inv2d(h, tmp, tmp2, fd, scale, 0)) return XFB_E_CUDA;     // :212-214
    GLAUNCH(h, (gen_jacobian<<<gb, 256, 0, h->stream>>>(fc, fa, fd, fb, src, fa, n)));                                  // :225-227
    return generic_fwd2d(h, fa, tmp2, T);                                                                                // :237
}

// one RK4 step of every member, one kernel per loop of src/main.cpp:286-317.  A step is 72 short launches per member
// (124 with the tracer) on grids that live in L2 -- launch gaps, not kernels, bound it --, so xfb_step replays it from a
// CUDA graph (step_replay) like the fused step.
int generic_one_step(xfb_handle h, float dt)
{
    const int P = h->hy;
    const long long n = (long long)h->grids, hn = (long long)h->nx * h->hy;
    const float scale = 1.0f / (float)((double)h->nx * (double)h->ny);
    const unsigned gb = (unsigned)((n + 255) / 256), hb = (unsigned)((hn + 255) / 256);
    for (int m = 0; m < h->batch; ++m) {
        cpx *z0 = h->z0 + (size_t)m * h->hpad, *zk = h->zk + (size_t)m * h->hpad, *acc = h->acc + (size_t)m * h->hpad;
        const float *src = h->has_src ? h->src + (size_t)m * h->grids : nullptr;
        float *fa = h->real_a, *fb = h->real_b, *fc = h->real_c, *fd = (float *)h->t[0];      // dvortdx, dvortdy, -u, v
        cpx *tmp = h->spec_a, *tmp2 = h->spec_b, *T = h->jint;
        for (int k = 1; k <= 4; ++k) {
            const cpx *z = (k == 1) ? z0 : zk;
            if (generic_tendency(h, z, src, T)) return XFB_E_CUDA;
            if (h->lin.on)
                GLAUNCH(h, (gen_stage<true><<<hb, 256, 0, h->stream>>>(T, z0, zk, acc, h->nx, h->hy, h->kx2, h->ky2, h->mask_kd, h->nu,
                                                                        dt, (k == 3) ? dt : dt / 2.0f, k, h->kx, h->lin)));
            else
                GLAUNCH(h, (gen_stage<false><<<hb, 256, 0, h->stream>>>(T, z0, zk, acc, h->nx, h->hy, h->kx2, h->ky2, h->mask_kd, h->nu,
                                                                         dt, (k == 3) ? dt : dt / 2.0f, k, h->kx, h->lin)));
            if (h->has_tracer) {
                // passive tracer (xfb_set_tracer): the same loops with c for vort and kappa for NU; -u, v of this
                // stage are still in fc, fd
                cpx *c0 = h->c0 + (size_t)m * h->hpad, *ck = h->ck + (size_t)m * h->hpad, *cacc = h->cacc + (size_t)m * h->hpad;
                const cpx *c = (k == 1) ? c0 : ck;
                if (launch_pw(h, OP_GRADX, c, P, tmp, P, P) || generic_inv2d(h, tmp, tmp2, fa, scale, 0)) return XFB_E_CUDA;
                if (launch_pw(h, OP_GRADY, c, P, tmp, P, P) || generic_inv2d(h, tmp, tmp2, fb, scale, 0)) return XFB_E_CUDA;
                GLAUNCH(h, (gen_jacobian<<<gb, 256, 0, h->stream>>>(fc, fa, fd, fb, nullptr, fa, n)));
                if (generic_fwd2d(h, fa, tmp2, h->cjint)) return XFB_E_CUDA;
                GLAUNCH(h, (gen_stage<false><<<hb, 256, 0, h->stream>>>(h->cjint, c0, ck, cacc, h->nx, h->hy, h->kx2, h->ky2, h->mask_kd,
                                                                         h->kappa, dt, (k == 3) ? dt : dt / 2.0f, k, h->kx, LinCoef())));
            }
        }
    }
    return 0;
}

}  // namespace xfb

// xfb_row.cuh -- K-ROW: the line transforms along y (the contiguous direction) shared by every K-ROW kernel,
// and row_kernel, one line per group of NY/32 threads, which replaces for one row i of the grid:
//   R2C : the last-dimension half of fftwf_plan_dft_r2c_2d   (/root/reference/src/main.cpp:126-127,237,256)
//   C2R : the last-dimension half of fftwf_plan_dft_c2r_2d + fftwf_backward_normalize
//         (main.cpp:129-135,37-41)
// row_kernel serves 16384-point lines only (operator tier, record path, slab handles); shorter lines run on the pair
// kernels (xfb_rowpair.cuh), and the stepper's JAC at 16384 on the two-level kernel (xfb_rowpair2l.cuh).
// A real line of NY points is transformed as a complex line of L = NY/2 points plus the
// standard split/merge step of a half-length real transform.
//
// Layout of the spectral lines exchanged with K-COL ("pair layout"): rows 2m and 2m+1 are interleaved
// element by element, element (i, k) lives at ((i >> 1) * pitch + k) * 2 + (i & 1).  K-COL reads and writes
// these arrays in tiles of W columns x all rows; with the rows paired a W = 2 tile touches whole 32-byte
// sectors (2 columns x 2 rows) instead of half sectors -- measured 4.8 TB/s against 1.9 TB/s for a plain
// strided tile copy on B200 (tools/probes/probe_tma_tile.cu).  The two lines of a pair are transformed by
// the same CTA whenever a CTA holds more than one line, so the half-used sectors of one line are L1 hits
// of the other.
#pragma once
#include "xfb_fft.cuh"

namespace xfb {

enum { ROW_R2C = 0, ROW_C2R = 1, ROW_JAC = 2, ROW_DIAG = 3 };

struct RowParams {
    const cpx *spec_in[4];   // JAC: T_zx, T_zy, T_u, T_v ; C2R: [0]
    const float *real_in;    // R2C input ; JAC: optional source term (may be null)
    cpx *spec_out;           // R2C / JAC output (y-transformed lines)
    float *real_out;         // C2R output ; DIAG: first output field
    float *real_out2;        // DIAG: second output field
    int diag_kind;           // DIAG: 0 strain diagnostics (tfil, deform) of psi_xy, psi_xx, psi_yy ; 1 tracer (zeta, |grad zeta|^2)
    const cpx *tw;           // exp(-2 pi i k / twn)
    int twn;
    int nrows;               // NX * batch
    int pitch;               // complex elements per spectral line (>= NY/2+1)
    // slab-decomposed runs (DIST): a spectral line is cut into `pitch / cw` panels of cw columns, one per
    // (rank, column chunk); element k of local row r lives at
    //   (k / cw) * panel_stride + ((r >> 1) * cw + (k % cw)) * 2 + (r & 1)
    int cw;                  // columns per panel
    long long panel_stride;  // complex elements between panels (= local rows * cw)
    unsigned cw_magic;       // ceil(2^32 / cw): k / cw == __umulhi(k, cw_magic) for every k < pitch (checked on the host)
    // DIST, fused exchange: panel (q, c) of the OUTPUT is not written to the local array but straight into the
    // receive array of rank q (peer memory over NVLink, or the rank's own for q == me): panel_base[q * nchunks + c]
    // points at rows [me * rows, ...) of chunk c there, out_row_off = first local row of this launch * cw.
    cpx *const *panel_base;  // device array, null: local output
    long long out_row_off;
    float scale;             // 1/(NX*NY) applied after every C2R (fftwf_backward_normalize)
    int negate;              // C2R: multiply by -1 after scaling (u = -u)
};

template <int NY>
struct RowCfg {
    static constexpr int L = NY / 2;
    static constexpr int G = L / 16;                         // threads per line
    // both lines of a row pair in one CTA wherever the shared memory allows it (NY <= 8192); row_kernel is instantiated
    // at NY = 16384 only, where THREADS = G = 512 and LPC = 1
    static constexpr int THREADS = (G >= 512) ? G : (2 * G >= 128) ? 2 * G : 128;
    static constexpr int LPC = THREADS / G;                  // lines per CTA
    static constexpr int SMEM = LPC * LinePlan<L>::PADDED * (int)sizeof(cpx);
    static constexpr int MINB = (THREADS >= 512) ? 1 : (THREADS >= 256) ? 2 : 4;
};

template <bool NAMED>
struct RowBarSel {
    typedef CtaBar type;
    static __device__ __forceinline__ CtaBar make(int, int) { return CtaBar(); }
};
template <>
struct RowBarSel<true> {
    typedef NamedBar type;
    static __device__ __forceinline__ NamedBar make(int id, int n) { return NamedBar{id, n}; }
};

// position of element k of a spectral line relative to the line's base pointer (pair layout: stride 2)
template <bool DIST>
__device__ __forceinline__ long long line_pos(const RowParams &p, const int k)
{
    if (!DIST) return 2 * k;
    const int panel = (int)__umulhi((unsigned)k, p.cw_magic);
    return (long long)panel * p.panel_stride + 2 * (k - panel * p.cw);
}

// address of output element k of the line whose local base pointer is `line` (= p.spec_out + line offset)
template <bool DIST>
__device__ __forceinline__ cpx *out_addr(const RowParams &p, cpx *line, const int k)
{
    if (!DIST) return line + 2 * k;
    const int panel = (int)__umulhi((unsigned)k, p.cw_magic);
    const long long within = 2 * (k - panel * p.cw);
    if (p.panel_base == nullptr) return line + (long long)panel * p.panel_stride + within;
    cpx *base = reinterpret_cast<cpx *>(__ldg(reinterpret_cast<const unsigned long long *>(p.panel_base) + panel));
    return base + p.out_row_off + (line - p.spec_out) + within;
}

// base of the line of `row` in a pair-layout array whose rows hold `rowpitch` complex elements
__device__ __forceinline__ size_t line_base(const int row, const int rowpitch)
{
    return (size_t)(row >> 1) * (size_t)(2 * rowpitch) + (size_t)(row & 1);
}

// exp(-2 pi i q / 32), q = 0..15
__device__ __forceinline__ cpx w32(int q)
{
    const float C[16] = {1.f, 0.98078528040323044913f, XFB_C16, 0.83146961230254523708f, XFB_C8, 0.55557023301960222474f,
                         XFB_S16, 0.19509032201612826785f, 0.f, -0.19509032201612826785f, -XFB_S16,
                         -0.55557023301960222474f, -XFB_C8, -0.83146961230254523708f, -XFB_C16, -0.98078528040323044913f};
    const float S[16] = {0.f, -0.19509032201612826785f, -XFB_S16, -0.55557023301960222474f, -XFB_C8,
                         -0.83146961230254523708f, -XFB_C16, -0.98078528040323044913f, -1.f, -0.98078528040323044913f,
                         -XFB_C16, -0.83146961230254523708f, -XFB_C8, -0.55557023301960222474f, -XFB_S16,
                         -0.19509032201612826785f};
    return mk(C[q], S[q]);
}

// half-spectrum line X[0..L] -> physical pairs: on return v[q] = (x[2m+1], x[2m]) * 1 (unscaled,
// swapped), m = t + q*G.  wt = exp(-2 pi i t / NY).
template <int NY, bool DIST, typename Bar>
__device__ __forceinline__ void c2r_line(cpx (&v)[16], const cpx *X, const RowParams &p, cpx *sm, int t, cpx wt,
                                         const LineTw<NY / 2> &tw, const Bar &bar)
{
    constexpr int L = NY / 2, G = L / 16;
    wt = launder(wt);
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        cpx a[8], b[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const int k = t + (8 * h + e) * G;
            a[e] = X[line_pos<DIST>(p, k)];
            b[e] = X[line_pos<DIST>(p, L - k)];
        }
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const int q = 8 * h + e;
            const int k = t + q * G;
            cpx A = a[e], B = cconj(b[e]);
            if (k == 0) { A.y = 0.f; B.y = 0.f; }      // c2r ignores Im of the DC and Nyquist bins
            const cpx E = cadd(A, B), D = csub(A, B);
            const cpx wk = cconj((q == 0) ? wt : cmul(wt, w32(q)));   // exp(+2 pi i k / NY)
            const cpx O = cmul(D, wk);
            // Z = E + i O ; swapped for the inverse transform
            v[q] = mk(E.y + O.x, E.x - O.y);
        }
    }
    line_fft<L, 1>(v, sm, t, 0, tw, bar);
}

// physical pairs v[q] = (x[2m], x[2m+1]) -> half-spectrum line written to Xout[0..L] (+ zeroed pad)
template <int NY, bool DIST, typename Bar>
__device__ __forceinline__ void r2c_line(cpx (&v)[16], cpx *__restrict__ Xout, const RowParams &p, int pitch, cpx *sm,
                                         int t, cpx wt, const LineTw<NY / 2> &tw, const Bar &bar)
{
    constexpr int L = NY / 2, G = L / 16;
    line_fft<L, 1>(v, sm, t, 0, tw, bar);
    wt = launder(wt);
#pragma unroll
    for (int q = 0; q < 16; ++q) sm[padpos(t + q * G)] = v[q];
    bar.sync();
#pragma unroll
    for (int q = 0; q < 16; ++q) {
        const int k = t + q * G;
        const cpx Zk = v[q];
        const cpx Zm = cconj(sm[padpos((L - k) & (L - 1))]);
        const cpx E = mk(0.5f * (Zk.x + Zm.x), 0.5f * (Zk.y + Zm.y));
        const cpx D = mk(0.5f * (Zk.x - Zm.x), 0.5f * (Zk.y - Zm.y));
        const cpx wk = (q == 0) ? wt : cmul(wt, w32(q));           // exp(-2 pi i k / NY)
        const cpx O = cmul(mul_negi(D), wk);
        *out_addr<DIST>(p, Xout, k) = cadd(E, O);
        if (k == 0) *out_addr<DIST>(p, Xout, L) = mk(Zk.x - Zk.y, 0.f);
    }
    for (int k = L + 1 + t; k < pitch; k += G) *out_addr<DIST>(p, Xout, k) = mk(0.f, 0.f);
}

template <int NY, int MODE, bool DIST>
__global__ void __launch_bounds__(RowCfg<NY>::THREADS, RowCfg<NY>::MINB)
row_kernel(const RowParams p)
{
    static_assert(MODE == ROW_R2C || MODE == ROW_C2R, "row_kernel has the plain transforms only");
    typedef RowCfg<NY> C;
    constexpr int L = C::L, G = C::G;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane_line = threadIdx.x / G;
    const int t = threadIdx.x % G;
    cpx *sm = reinterpret_cast<cpx *>(smem_raw) + (size_t)lane_line * LinePlan<L>::PADDED;
    int row = blockIdx.x * C::LPC + lane_line;
    const bool live = row < p.nrows;
    if (!live) row = p.nrows - 1;

    LineTw<L> tw;
    tw.init(p.tw, p.twn, t);
    const cpx wt = __ldg(p.tw + (size_t)t * (p.twn / NY));
    // one barrier per line where a line is made of whole warps, else the CTA barrier
    typedef typename RowBarSel<(G >= 32 && C::LPC > 1)>::type Bar;
    const Bar bar = RowBarSel<(G >= 32 && C::LPC > 1)>::make(1 + lane_line, G);

    cpx v[16];
    if (MODE == ROW_R2C) {
        const float2 *x = reinterpret_cast<const float2 *>(p.real_in + (size_t)row * NY);
#pragma unroll
        for (int q = 0; q < 16; ++q) v[q] = __ldg(x + t + q * G);
        cpx *out = p.spec_out + line_base(row, DIST ? p.cw : p.pitch);
        r2c_line<NY, DIST>(v, out, p, live ? p.pitch : 0, sm, t, wt, tw, bar);   // a clamped duplicate row rewrites identical values
    } else {
        c2r_line<NY, DIST>(v, p.spec_in[0] + line_base(row, DIST ? p.cw : p.pitch), p, sm, t, wt, tw, bar);
        float2 *x = reinterpret_cast<float2 *>(p.real_out + (size_t)row * NY);
        const float s = p.negate ? -p.scale : p.scale;
#pragma unroll
        for (int q = 0; q < 16; ++q) x[t + q * G] = mk(v[q].y * s, v[q].x * s);
    }
}

}  // namespace xfb

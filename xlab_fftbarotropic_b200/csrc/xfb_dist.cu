// xfb_dist.cu -- slab decomposition of one large grid over the GPUs of a node (SURVEY.md section 8e; the
// reference has no parallel path at all, src/main.cpp is one thread).
//
// Rank r of P holds the physical rows [r*NX/P, (r+1)*NX/P) and, in spectral space, a contiguous range of
// columns.  A 2-D transform is   local 1-D pass -> all-to-all -> local 1-D pass;   per RK stage five
// spectral arrays cross (the y-transformed tendency one way, the four x-inverse-transformed products the
// other way).  K-ROW and K-COL are the single-GPU kernels: K-ROW addresses its spectral lines through
// "panels" (one per (destination rank, column chunk), each a contiguous [rows][cw] block, so every
// message of the all-to-all is one contiguous buffer), K-COL runs once per column chunk.
//
// Overlap: K-ROW is launched in row chunks and K-COL in column chunks; the exchange of chunk i runs on a
// second stream while chunk i+1 computes, so only the last chunk's exchange is exposed.
//
// Two transports:
//   NCCL     one process per GPU (xfb_create_dist): grouped ncclSend/ncclRecv over NVLink, libnccl.so.2 is
//            loaded at run time (the single-GPU path does not depend on it);
//   loopback all ranks in one process on ONE device sharing one stream (xfb_loopback_*): plain device
//            copies.  It exists so the slab indexing is testable on a single GPU.
#include <dlfcn.h>
#include <nccl.h>

#include <cstdlib>
#include <cstring>
#include <new>

#include "xfb_handle.h"

namespace xfb {

struct NcclApi {
    void *lib;
    ncclResult_t (*GetUniqueId)(ncclUniqueId *);
    ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int);
    ncclResult_t (*CommDestroy)(ncclComm_t);
    ncclResult_t (*Send)(const void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t);
    ncclResult_t (*Recv)(void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t);
    ncclResult_t (*GroupStart)();
    ncclResult_t (*GroupEnd)();
    ncclResult_t (*AllGather)(const void *, void *, size_t, ncclDataType_t, ncclComm_t, cudaStream_t);
    ncclResult_t (*AllReduce)(const void *, void *, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t);
    const char *(*GetErrorString)(ncclResult_t);
};

static NcclApi g_nccl;

static int nccl_load()
{
    if (g_nccl.lib) return 0;
    void *lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!lib) lib = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!lib) return fail(XFB_E_NCCL, "cannot load libnccl.so.2: %s", dlerror());
    NcclApi a;
    a.lib = lib;
#define SYM(field, name)                                                                   \
    do {                                                                                   \
        *(void **)(&a.field) = dlsym(lib, name);                                           \
        if (!a.field) return fail(XFB_E_NCCL, "libnccl.so.2 has no symbol %s", name);      \
    } while (0)
    SYM(GetUniqueId, "ncclGetUniqueId");
    SYM(CommInitRank, "ncclCommInitRank");
    SYM(CommDestroy, "ncclCommDestroy");
    SYM(Send, "ncclSend");
    SYM(Recv, "ncclRecv");
    SYM(GroupStart, "ncclGroupStart");
    SYM(GroupEnd, "ncclGroupEnd");
    SYM(AllGather, "ncclAllGather");
    SYM(AllReduce, "ncclAllReduce");
    SYM(GetErrorString, "ncclGetErrorString");
#undef SYM
    g_nccl = a;
    return 0;
}

#define NCK(call)                                                                                        \
    do {                                                                                                 \
        ncclResult_t r__ = (call);                                                                       \
        if (r__ != ncclSuccess) return fail(XFB_E_NCCL, "%s: %s", #call, g_nccl.GetErrorString(r__));    \
    } while (0)

struct Team {
    int nranks;
    int nlocal;               // loopback: nranks handles in this process; NCCL: 1
    xfb_handle local[16];
    ncclComm_t comm;          // NCCL transport
    bool loopback;
};

// ---- block addressing -----------------------------------------------------------------------------
// row side (K-ROW's panels): panel (q, c) = [rows][cw], rows paired ; col side (K-COL's chunks): chunk c = [NX][cw]
static inline size_t row_off(xfb_handle h, int q, int c, int r0) { return ((size_t)(q * h->nchunks + c) * h->rows + r0) * h->pitch; }
static inline size_t col_off(xfb_handle h, int q, int c, int r0) { return ((size_t)c * h->nx + (size_t)q * h->rows + r0) * h->pitch; }

enum { ROW2COL = 0, COL2ROW = 1 };

// Fused row -> column exchange (XFB_SLAB_FUSED=0 turns it off): K-ROW stores its output panels straight into the
// receive arrays of the ranks that own the columns -- plain 16-byte stores on the CUDA-IPC peer mappings, NVLink traffic
// issued by the transform kernel itself while it computes -- instead of writing them locally and having a push kernel
// or the copy engines move them afterwards.  recv_of_rank[q] = receive block of rank q as seen from this process
// (array 0 of the block = jint_recv).  Panel (q, c) of rank `me` lands at rows [me * rows, ...) of chunk c there.
static int build_panel_table(xfb_handle h, cpx *const *recv_of_rank)
{
    // two-level K-COL (16384-point columns): its own row pairs go straight into this rank's receive arrays
    static const bool self_off = getenv("XFB_SLAB_SELF_DIRECT") && atoi(getenv("XFB_SLAB_SELF_DIRECT")) == 0;
    h->self_direct = !self_off && col_two_level(h->nx) && (h->rows / 2) % (h->nx / 32) == 0;
    static const bool off = getenv("XFB_SLAB_FUSED") && atoi(getenv("XFB_SLAB_FUSED")) == 0;
    if (off) return 0;
    const int n = h->nranks * h->nchunks;
    std::vector<cpx *> tab(n);
    for (int q = 0; q < h->nranks; ++q)
        for (int c = 0; c < h->nchunks; ++c) tab[q * h->nchunks + c] = recv_of_rank[q] + col_off(h, h->rank, c, 0);
    if (dev_alloc((void **)&h->panel_base, sizeof(cpx *) * n)) return XFB_E_CUDA;
    CK(cudaMemcpy(h->panel_base, tab.data(), sizeof(cpx *) * n, cudaMemcpyHostToDevice));
    // the tracer's tendency lands in array 5 of the receive blocks (cjint_recv)
    for (int q = 0; q < h->nranks; ++q)
        for (int c = 0; c < h->nchunks; ++c) tab[q * h->nchunks + c] = recv_of_rank[q] + (size_t)5 * h->hpad + col_off(h, h->rank, c, 0);
    if (dev_alloc((void **)&h->panel_base_c, sizeof(cpx *) * n)) return XFB_E_CUDA;
    CK(cudaMemcpy(h->panel_base_c, tab.data(), sizeof(cpx *) * n, cudaMemcpyHostToDevice));
    return 0;
}

// ---- SM-driven push: one launch copies up to 64 contiguous segments into peer memory with 16-byte stores ------------
// The copy engines lose more than half of their NVLink bandwidth while the SMs keep the memory system busy
// (tools/probes/probe_p2p_copy.cu and the slab runs: 760 -> ~300 GB/s).  A few CTAs of plain ld.global / st.global on
// the peer mappings do not: their traffic is ordinary SM traffic.  Launched on the (high-priority) communication
// stream the CTAs are scheduled between the compute kernel's CTAs as SMs free up.
struct PushSegs {
    int n;
    const float4 *src[64];
    float4 *dst[64];
    unsigned long long n16[64];      // float4 elements
};

__global__ void __launch_bounds__(512) push_kernel(const PushSegs s)
{
    const int seg = blockIdx.y;
    if (seg >= s.n) return;
    const float4 *__restrict__ src = s.src[seg];
    float4 *__restrict__ dst = s.dst[seg];
    const unsigned long long n = s.n16[seg];
    const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
    unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    // four independent 16-byte loads in flight per thread
    for (; i + 3 * stride < n; i += 4 * stride) {
        const float4 a = src[i], b = src[i + stride], c = src[i + 2 * stride], d = src[i + 3 * stride];
        dst[i] = a; dst[i + stride] = b; dst[i + 2 * stride] = c; dst[i + 3 * stride] = d;
    }
    for (; i < n; i += stride) dst[i] = src[i];
}

// One all-to-all of the blocks (column chunks [c0, c1), local rows [r0, r1)) of `na` arrays.
// NCCL: issued for the single local rank on `st`.  Loopback: device copies for every rank on the shared stream.
static int exchange(Team *T, int dir, cpx *const *row_ptrs_of_rank, cpx *const *col_ptrs_of_rank, int na, int c0, int c1, int r0,
                    int r1, cudaStream_t st, bool skip_self = false, int abase = -1)
{
    // abase: index of the first destination array inside the peers' receive blocks (P2P transports): the vorticity uses
    // 0 (jint_recv) for ROW2COL and 1.. (tr[0..3]) for COL2ROW, the tracer 5 (cjint_recv) and 6.. (trc[0..1])
    if (abase < 0) abase = (dir == ROW2COL) ? 0 : 1;
    // skip_self: the producer has already put every rank's own block in place (two-level K-COL, ColParams::self_out)
    // row_ptrs_of_rank / col_ptrs_of_rank: [nlocal][na]
    xfb_handle h0 = T->local[0];
    const size_t count = (size_t)(r1 - r0) * h0->pitch;      // complex elements per block
    if (T->loopback) {
        for (int R = 0; R < T->nranks; ++R)
            for (int q = 0; q < T->nranks; ++q)
                for (int a = 0; a < na; ++a)
                    for (int c = c0; c < c1; ++c) {
                        if (skip_self && q == R) continue;
                        cpx *rowR = row_ptrs_of_rank[R * na + a], *colR = col_ptrs_of_rank[R * na + a];
                        cpx *rowq = row_ptrs_of_rank[q * na + a], *colq = col_ptrs_of_rank[q * na + a];
                        if (dir == ROW2COL)
                            CK(cudaMemcpyAsync(colR + col_off(h0, q, c, r0), rowq + row_off(h0, R, c, r0), sizeof(cpx) * count,
                                               cudaMemcpyDeviceToDevice, st));
                        else
                            CK(cudaMemcpyAsync(rowR + row_off(h0, q, c, r0), colq + col_off(h0, R, c, r0), sizeof(cpx) * count,
                                               cudaMemcpyDeviceToDevice, st));
                    }
        return 0;
    }
    const int me = h0->rank;
    if (h0->p2p) {
        // Copy-engine pushes straight into the peers' receive arrays (mapped over CUDA IPC): one 2-D copy per peer
        // and piece moves the blocks of all column chunks (ROW2COL) or of all `na` arrays (COL2ROW).  The copies
        // fork from `st` onto h->ncopy streams (several copy engines in flight) and join it again; every block is
        // cut into `pieces` column ranges when there are fewer peers than streams.  Peers are visited in a rotated
        // order so that at any moment every GPU is the target of one sender.  Completion on the RECEIVER is
        // signalled by the phase barrier (phase_barrier below), not here.
        if (h0->push_sm) {
            PushSegs segs;
            segs.n = 0;
            auto add = [&](cpx *dst, const cpx *src, size_t elems) {
                segs.src[segs.n] = reinterpret_cast<const float4 *>(src);
                segs.dst[segs.n] = reinterpret_cast<float4 *>(dst);
                segs.n16[segs.n] = elems / 2;
                ++segs.n;
            };
            auto flush = [&]() -> int {
                if (segs.n == 0) return 0;
                push_kernel<<<dim3(h0->push_blocks, segs.n), 512, 0, st>>>(segs);
                cudaError_t e = cudaGetLastError();
                if (e != cudaSuccess) return fail(XFB_E_CUDA, "push_kernel: %s", cudaGetErrorString(e));
                h0->launches++;
                segs.n = 0;
                return 0;
            };
            for (int i = skip_self ? 1 : 0; i < T->nranks; ++i) {
                const int q = (me + i) % T->nranks;
                cpx *peer = h0->peer_recv[q];
                for (int c = c0; c < c1; ++c) {
                    if (dir == ROW2COL)
                        add(peer + (size_t)abase * h0->hpad + col_off(h0, me, c, r0), row_ptrs_of_rank[0] + row_off(h0, q, c, r0), count);
                    else
                        for (int a = 0; a < na; ++a)
                            add(peer + (size_t)(abase + a) * h0->hpad + row_off(h0, me, c, r0), col_ptrs_of_rank[a] + col_off(h0, q, c, r0), count);
                    if (segs.n + 4 > 64)
                        if (int e = flush()) return e;
                }
            }
            return flush();
        }
        const int ncs = h0->ncopy;
        CK(cudaEventRecord(h0->ev_fork, st));
        for (int s = 0; s < ncs; ++s) CK(cudaStreamWaitEvent(h0->copy_stream[s], h0->ev_fork, 0));
        const int pieces = (T->nranks - 1 >= ncs) ? 1 : ncs / (T->nranks - 1);
        const size_t piece_elems = ((count + pieces - 1) / pieces + 1) & ~(size_t)1;      // even: 16-byte aligned pieces
        int slot = 0;
        for (int i = skip_self ? 1 : 0; i < T->nranks; ++i) {
            const int q = (me + i) % T->nranks;
            cpx *peer = h0->peer_recv[q];
            for (int pc = 0; pc < pieces; ++pc) {
                const size_t e0 = (size_t)pc * piece_elems;
                if (e0 >= count) break;
                const size_t wbytes = sizeof(cpx) * ((count - e0 < piece_elems) ? count - e0 : piece_elems);
                cudaStream_t cs = h0->copy_stream[slot++ % ncs];
                if (dir == ROW2COL) {
                    // array 0 of the receive block = jint_recv ; chunks c0..c1-1 are rows*cw apart here, NX*cw apart there
                    const cpx *src = row_ptrs_of_rank[0] + row_off(h0, q, c0, r0) + e0;
                    cpx *dst = peer + (size_t)abase * h0->hpad + col_off(h0, me, c0, r0) + e0;
                    CK(cudaMemcpy2DAsync(dst, sizeof(cpx) * (size_t)h0->nx * h0->pitch, src, sizeof(cpx) * (size_t)h0->rows * h0->pitch,
                                         wbytes, (size_t)(c1 - c0), cudaMemcpyDeviceToDevice, cs));
                } else {
                    // arrays 1..4 of the receive block = tr[0..3] (or tr[0] alone, na == 1)
                    for (int c = c0; c < c1; ++c) {
                        if (na == 4) {
                            const cpx *src = col_ptrs_of_rank[0] + col_off(h0, q, c, r0) + e0;     // t[0]; t[1..3] follow hpad apart
                            cpx *dst = peer + (size_t)abase * h0->hpad + row_off(h0, me, c, r0) + e0;
                            CK(cudaMemcpy2DAsync(dst, sizeof(cpx) * h0->hpad, src, sizeof(cpx) * h0->hpad, wbytes, 4,
                                                 cudaMemcpyDeviceToDevice, cs));
                        } else {
                            for (int a = 0; a < na; ++a)
                                CK(cudaMemcpyAsync(peer + (size_t)(abase + a) * h0->hpad + row_off(h0, me, c, r0) + e0,
                                                   col_ptrs_of_rank[a] + col_off(h0, q, c, r0) + e0, wbytes, cudaMemcpyDeviceToDevice, cs));
                        }
                    }
                }
            }
        }
        for (int s = 0; s < ncs; ++s) {
            CK(cudaEventRecord(h0->ev_copy[s], h0->copy_stream[s]));
            CK(cudaStreamWaitEvent(st, h0->ev_copy[s], 0));
        }
        return 0;
    }
    NCK(g_nccl.GroupStart());
    for (int a = 0; a < na; ++a)
        for (int c = c0; c < c1; ++c)
            for (int q = 0; q < T->nranks; ++q) {
                cpx *row = row_ptrs_of_rank[a] + row_off(h0, q, c, r0), *col = col_ptrs_of_rank[a] + col_off(h0, q, c, r0);
                const cpx *sendp = (dir == ROW2COL) ? row : col;
                cpx *recvp = (dir == ROW2COL) ? col : row;
                if (q == me) continue;
                NCK(g_nccl.Send(sendp, 2 * count, ncclFloat, q, T->comm, st));
                NCK(g_nccl.Recv(recvp, 2 * count, ncclFloat, q, T->comm, st));
            }
    NCK(g_nccl.GroupEnd());
    for (int a = 0; a < na && !skip_self; ++a)
        for (int c = c0; c < c1; ++c) {
            cpx *row = row_ptrs_of_rank[a] + row_off(h0, me, c, r0), *col = col_ptrs_of_rank[a] + col_off(h0, me, c, r0);
            CK(cudaMemcpyAsync((dir == ROW2COL) ? col : row, (dir == ROW2COL) ? row : col, sizeof(cpx) * count,
                               cudaMemcpyDeviceToDevice, st));
        }
    return 0;
}

// ---- per-rank launches --------------------------------------------------------------------------------
static int launch_row_chunk(xfb_handle h, int mode, const cpx *const in[4], const float *real_in, cpx *spec_out, float *real_out,
                            int negate, int r0, int r1, bool fused_out = false, bool tracer = false)
{
    RowParams r;
    fill_row(h, r, r1 - r0);
    const size_t so = (size_t)r0 * h->pitch, ro = (size_t)r0 * h->ny;
    if (fused_out && h->panel_base) { r.panel_base = tracer ? h->panel_base_c : h->panel_base; r.out_row_off = (long long)so; }
    for (int f = 0; f < 4; ++f) r.spec_in[f] = in && in[f] ? in[f] + so : nullptr;
    r.real_in = real_in ? real_in + ro : nullptr;
    r.spec_out = spec_out ? spec_out + so : nullptr;
    r.real_out = real_out ? real_out + ro : nullptr;
    r.negate = negate;
    CKL(h, launch_row(h->ny, mode, r, h->stream));
    return 0;
}

// tracer: the same launch on the passive tracer's arrays (state c0 / ck / cacc, tendency cjint_recv, two gradient
// products tc[0..1], diffusivity kappa); `mode` is then COL_TSTEP / COL_TPRO (or COL_FWD into c0).
// out: COL_INV's output; COL_FWD writes there instead of the state when it is not null
static int launch_col_chunk(xfb_handle h, int mode, int chunk, int stage, float dt, const cpx *inv_in, cpx *out, bool tracer = false)
{
    ColParams c;
    fill_col(h, c, chunk);
    const size_t off = (size_t)chunk * h->nx * h->pitch;
    c.jint = h->jint_recv + off; c.z0 = h->z0 + off; c.zk = h->zk + off; c.acc = h->acc + off;
    c.st_tile_stride = (long long)h->nx * h->tw_state; c.st_row_stride = h->tw_state;     // tile-major state
    for (int f = 0; f < 4; ++f) c.t_out[f] = h->t[f] + off;
    if (tracer) {
        c.z0 = h->c0 + off; c.zk = h->ck + off; c.acc = h->cacc + off; c.nu = h->kappa;
        if (mode != COL_FWD) c.jint = h->cjint_recv + off;       // COL_FWD: the field just travelled through jint_recv
        for (int f = 0; f < 4; ++f) c.t_out[f] = h->tc[f & 1] + off;
    }
    if (mode == COL_INV) { c.inv_in = inv_in + off; c.t_out[0] = out + off; }
    if (mode == COL_FWD && out) c.z0 = out + off;
    c.dt = dt; c.stage = stage;
    c.dt_stage = (stage == 3) ? dt : dt / 2.0f;          // main.cpp:296,299,302
    if (h->self_direct && (mode == COL_STEP || mode == COL_PRO || mode == COL_TSTEP || mode == COL_TPRO)) {
        c.self_piece0 = h->rank * (h->rows / 2);
        c.self_pieces = h->rows / 2;
        for (int f = 0; f < 4; ++f) c.self_out[f] = (tracer ? h->trc[f & 1] : h->tr[f]) + row_off(h, h->rank, chunk, 0);
    }
    CKL(h, launch_col(h->nx, mode, c, 1, h->stream));
    return 0;
}

// End of an exchange phase on the NCCL/P2P transports.  With copy-engine pushes nobody knows when the peers' data has
// landed: a one-float all-reduce on the communication stream is the barrier (every rank enters it after its own
// pushes, so leaving it means all pushes into this rank are complete -- and that every peer has finished reading
// what the NEXT phase will overwrite).  ncclSend/ncclRecv pairs synchronise by themselves.
static int phase_barrier(Team *T, cudaStream_t st)
{
    xfb_handle h0 = T->local[0];
    if (!h0->p2p) return 0;
    NCK(g_nccl.AllReduce(h0->sync_buf, h0->sync_buf, 1, ncclFloat, ncclSum, T->comm, st));
    return 0;
}

// Barrier over the ranks' COMPUTE streams: every rank has finished the work it has enqueued so far before any rank's
// later work starts.  Needed wherever a receive array (tr[], jint_recv) is read by a kernel that is NOT followed by an
// exchange phase of its own: a faster peer's next operation would otherwise push into the array while this rank is
// still reading it (the trailing ROW_C2R of team_inverse, the COL_FWD of team_set_vorticity).  Inside the RK loop the
// alternating phase barriers already give this ordering.
static int team_fence(Team *T)
{
    xfb_handle h0 = T->local[0];
    if (T->loopback || !h0->p2p) return 0;          // one stream / ncclRecv is posted by the receiver itself
    CK(cudaEventRecord(h0->ev_chunk[0], h0->stream));
    CK(cudaStreamWaitEvent(h0->comm_stream, h0->ev_chunk[0], 0));
    if (int e = phase_barrier(T, h0->comm_stream)) return e;
    CK(cudaEventRecord(h0->ev_comm[0], h0->comm_stream));
    CK(cudaStreamWaitEvent(h0->stream, h0->ev_comm[0], 0));
    return 0;
}

// events around the exchanges when profiling (NCCL transport only; the loopback shares the compute stream)
static void a2a_mark(xfb_handle h, cudaStream_t st)
{
    if (h->profiling && h->ev_a2a) cudaEventRecord(next_event(h->ev_a2a, h->ev_a2a_used), st);
}

// y pass for all local ranks (row chunks) + exchange into the column side.
//   produce(h, r0, r1) launches K-ROW on local rows [r0, r1) ; row_of(h) / col_of(h) name the two arrays
template <typename F, typename GR, typename GC>
static int rows_then_exchange(Team *T, F produce, GR row_of, GC col_of, int abase = 0)
{
    xfb_handle h0 = T->local[0];
    const int C = h0->nchunks, rc = h0->rows / C;
    cpx *rp[16], *cp[16];
    for (int l = 0; l < T->nlocal; ++l) { rp[l] = row_of(T->local[l]); cp[l] = col_of(T->local[l]); }
    if (h0->panel_base) {
        // fused exchange: the kernels have written into the receive arrays themselves; what is left is the barrier
        for (int l = 0; l < T->nlocal; ++l)
            if (int e = produce(T->local[l], 0, h0->rows)) return e;
        if (T->loopback) return 0;
        CK(cudaEventRecord(h0->ev_chunk[0], h0->stream));
        CK(cudaStreamWaitEvent(h0->comm_stream, h0->ev_chunk[0], 0));
        if (int e = phase_barrier(T, h0->comm_stream)) return e;
        CK(cudaEventRecord(h0->ev_comm[0], h0->comm_stream));
        CK(cudaStreamWaitEvent(h0->stream, h0->ev_comm[0], 0));
        return 0;
    }
    if (T->loopback) {
        for (int l = 0; l < T->nlocal; ++l)
            for (int i = 0; i < C; ++i)
                if (int e = produce(T->local[l], i * rc, (i + 1) * rc)) return e;
        return exchange(T, ROW2COL, rp, cp, 1, 0, C, 0, h0->rows, h0->stream, false, abase);
    }
    for (int i = 0; i < C; ++i) {
        if (int e = produce(h0, i * rc, (i + 1) * rc)) return e;
        CK(cudaEventRecord(h0->ev_chunk[i], h0->stream));
        CK(cudaStreamWaitEvent(h0->comm_stream, h0->ev_chunk[i], 0));
        a2a_mark(h0, h0->comm_stream);
        if (int e = exchange(T, ROW2COL, rp, cp, 1, 0, C, i * rc, (i + 1) * rc, h0->comm_stream, false, abase)) return e;
        a2a_mark(h0, h0->comm_stream);
    }
    if (int e = phase_barrier(T, h0->comm_stream)) return e;
    CK(cudaEventRecord(h0->ev_comm[0], h0->comm_stream));
    CK(cudaStreamWaitEvent(h0->stream, h0->ev_comm[0], 0));
    return 0;
}

// x pass for all local ranks (column chunks) + exchange of `na` arrays back to the row side.
//   produce(h, chunk) launches K-COL ; col_of(h, a) / row_of(h, a) name array a on the two sides
template <typename F, typename GC, typename GR>
static int cols_then_exchange(Team *T, F produce, GC col_of, GR row_of, int na, bool skip_self = false, int abase = 1)
{
    xfb_handle h0 = T->local[0];
    const int C = h0->nchunks;
    cpx *rp[16 * 4], *cp[16 * 4];
    for (int l = 0; l < T->nlocal; ++l)
        for (int a = 0; a < na; ++a) { rp[l * na + a] = row_of(T->local[l], a); cp[l * na + a] = col_of(T->local[l], a); }
    if (T->loopback) {
        for (int l = 0; l < T->nlocal; ++l)
            for (int c = 0; c < C; ++c)
                if (int e = produce(T->local[l], c)) return e;
        return exchange(T, COL2ROW, rp, cp, na, 0, C, 0, h0->rows, h0->stream, skip_self, abase);
    }
    for (int c = 0; c < C; ++c) {
        if (int e = produce(h0, c)) return e;
        CK(cudaEventRecord(h0->ev_chunk[c], h0->stream));
        CK(cudaStreamWaitEvent(h0->comm_stream, h0->ev_chunk[c], 0));
        a2a_mark(h0, h0->comm_stream);
        if (int e = exchange(T, COL2ROW, rp, cp, na, c, c + 1, 0, h0->rows, h0->comm_stream, skip_self, abase)) return e;
        a2a_mark(h0, h0->comm_stream);
    }
    if (int e = phase_barrier(T, h0->comm_stream)) return e;
    CK(cudaEventRecord(h0->ev_comm[1], h0->comm_stream));
    CK(cudaStreamWaitEvent(h0->stream, h0->ev_comm[1], 0));
    return 0;
}

// ---- team-level operations ------------------------------------------------------------------------------
// vort[l]: device pointer to the local rows of rank local[l]; tracer: the field becomes the passive tracer's state c0
static int team_set_vorticity(Team *T, const float *const *vort, bool tracer = false)
{
    int e = rows_then_exchange(
        T,
        [&](xfb_handle h, int r0, int r1) {
            int l = 0;
            while (T->local[l] != h) ++l;
            return launch_row_chunk(h, ROW_R2C, nullptr, vort[l], h->jint, nullptr, 0, r0, r1, true);
        },
        [](xfb_handle h) { return h->jint; }, [](xfb_handle h) { return h->jint_recv; });
    if (e) return e;
    for (int l = 0; l < T->nlocal; ++l) {
        xfb_handle h = T->local[l];
        for (int c = 0; c < h->nchunks; ++c)
            if (int e2 = launch_col_chunk(h, COL_FWD, c, 0, 0.f, nullptr, nullptr, tracer)) return e2;
        if (tracer) {
            h->tcf_valid = false;
        } else {
            h->have_state = true;
            h->tf_valid = false;
        }
    }
    return team_fence(T);       // jint_recv has been consumed everywhere before anybody's next K-ROW stores into it
}

static int team_products(Team *T, int mode, int stage, float dt)
{
    return cols_then_exchange(
        T, [&](xfb_handle h, int c) { return launch_col_chunk(h, mode, c, stage, dt, nullptr, nullptr); },
        [](xfb_handle h, int a) { return h->t[a]; }, [](xfb_handle h, int a) { return h->tr[a]; }, 4, T->local[0]->self_direct);
}

// the tracer's two gradient products (i kx C, i ky C), x-inverse-transformed and sent to the row side (trc[0..1])
static int team_tracer_products(Team *T, int mode, int stage, float dt)
{
    return cols_then_exchange(
        T, [&](xfb_handle h, int c) { return launch_col_chunk(h, mode, c, stage, dt, nullptr, nullptr, true); },
        [](xfb_handle h, int a) { return h->tc[a]; }, [](xfb_handle h, int a) { return h->trc[a]; }, 2, T->local[0]->self_direct, 6);
}

static int team_step(Team *T, int nsteps, float dt)
{
    xfb_handle h0 = T->local[0];
    const bool tracer = h0->has_tracer;
    if (nsteps > 0 && !h0->tf_valid) {
        if (int e = team_products(T, COL_PRO, 0, dt)) return e;
        for (int l = 0; l < T->nlocal; ++l) T->local[l]->tf_valid = true;
    }
    if (nsteps > 0 && tracer && !h0->tcf_valid) {
        if (int e = team_tracer_products(T, COL_TPRO, 0, dt)) return e;
        for (int l = 0; l < T->nlocal; ++l) T->local[l]->tcf_valid = true;
    }
    for (int s = 0; s < nsteps; ++s)
        for (int k = 1; k <= 4; ++k) {
            if (h0->profiling && !T->loopback) cudaEventRecord(next_event(h0->ev_row, h0->ev_row_used), h0->stream);
            int e = rows_then_exchange(
                T,
                [&](xfb_handle h, int r0, int r1) {
                    return launch_row_chunk(h, ROW_JAC, h->tr, h->has_src ? h->src : nullptr, h->jint, nullptr, 0, r0, r1, true);
                },
                [](xfb_handle h) { return h->jint; }, [](xfb_handle h) { return h->jint_recv; });
            if (e) return e;
            if (tracer) {
                // the tracer's Jacobian with the velocity of this stage: (T_cx, T_cy) from trc[], (T_u, T_v) from tr[2..3]
                // -- before K-COL's exchange overwrites them (xfb_api.cu: xfb_step does the same on one GPU)
                e = rows_then_exchange(
                    T,
                    [&](xfb_handle h, int r0, int r1) {
                        const cpx *in[4] = {h->trc[0], h->trc[1], h->tr[2], h->tr[3]};
                        return launch_row_chunk(h, ROW_JAC, in, nullptr, h->cjint, nullptr, 0, r0, r1, true, true);
                    },
                    [](xfb_handle h) { return h->cjint; }, [](xfb_handle h) { return h->cjint_recv; }, 5);
                if (e) return e;
            }
            if (h0->profiling && !T->loopback) {
                cudaEventRecord(next_event(h0->ev_row, h0->ev_row_used), h0->stream);
                cudaEventRecord(next_event(h0->ev_col, h0->ev_col_used), h0->stream);
            }
            if (int e2 = team_products(T, COL_STEP, k, dt)) return e2;
            if (tracer)
                if (int e3 = team_tracer_products(T, COL_TSTEP, k, dt)) return e3;
            if (h0->profiling && !T->loopback) cudaEventRecord(next_event(h0->ev_col, h0->ev_col_used), h0->stream);
        }
    return 0;
}

// Spectral budget terms of every local rank, tile-major chunks like the state: the tendency r2c(-u.grad(zeta)) into
// spec_a (the stepper's K-ROW without the source, its exchange, a plain x pass per chunk) and, when `with_src`, the
// source's spectrum into spec_b (as team_set_vorticity forms a state; a rank without a source contributes zero rows).
// The products t[0..3] / tr[0..3] of the current state are formed first if the next step would have to form them.
static int team_budget_terms(Team *T, bool with_src)
{
    xfb_handle h0 = T->local[0];
    if (!h0->tf_valid) {
        if (int e = team_products(T, COL_PRO, 0, 0.f)) return e;
        for (int l = 0; l < T->nlocal; ++l) T->local[l]->tf_valid = true;
    }
    for (int pass = 0; pass < (with_src ? 2 : 1); ++pass) {
        if (pass == 1) {
            // jint_recv has been read everywhere before the source's rows land in it
            if (int e = team_fence(T)) return e;
            for (int l = 0; l < T->nlocal; ++l) {
                xfb_handle h = T->local[l];
                if (!h->has_src) CK(cudaMemsetAsync(h->real_a, 0, sizeof(float) * h->grids, h->stream));
            }
        }
        int e = rows_then_exchange(
            T,
            [&](xfb_handle h, int r0, int r1) {
                if (pass == 0) return launch_row_chunk(h, ROW_JAC, h->tr, nullptr, h->jint, nullptr, 0, r0, r1, true);
                return launch_row_chunk(h, ROW_R2C, nullptr, h->has_src ? h->src : h->real_a, h->jint, nullptr, 0, r0, r1, true);
            },
            [](xfb_handle h) { return h->jint; }, [](xfb_handle h) { return h->jint_recv; });
        if (e) return e;
        for (int l = 0; l < T->nlocal; ++l) {
            xfb_handle h = T->local[l];
            for (int c = 0; c < h->nchunks; ++c)
                if (int e2 = launch_col_chunk(h, COL_FWD, c, 0, 0.f, nullptr, pass == 0 ? h->spec_a : h->spec_b)) return e2;
        }
    }
    return team_fence(T);       // jint_recv has been consumed everywhere before anybody's next K-ROW stores into it
}

// operator chain `f` applied to the state (tracer_state: the passive tracer's), inverse 2-D transform, into dout[l]
// (device, local rows)
static int team_inverse(Team *T, const FieldOps &f, float *const *dout, bool tracer_state = false)
{
    int e = cols_then_exchange(
        T,
        [&](xfb_handle h, int c) {
            const size_t off = (size_t)c * h->nx * h->pitch;
            const int P = h->pitch;
            if (launch_pw(h, f.ops[0], (tracer_state ? h->c0 : h->z0) + off, P, h->spec_a + off, P, P, h->tw_state, 0, c)) return (int)XFB_E_CUDA;
            for (int o = 1; o < f.nops; ++o)
                if (launch_pw(h, f.ops[o], h->spec_a + off, P, h->spec_a + off, P, P, 0, 0, c)) return (int)XFB_E_CUDA;
            return launch_col_chunk(h, COL_INV, c, 0, 0.f, h->spec_a, h->spec_b);
        },
        [](xfb_handle h, int) { return h->spec_b; }, [](xfb_handle h, int) { return h->tr[0]; }, 1);
    if (e) return e;
    for (int l = 0; l < T->nlocal; ++l) {
        xfb_handle h = T->local[l];
        const cpx *in[4] = {h->tr[0], nullptr, nullptr, nullptr};
        if (int e2 = launch_row_chunk(h, ROW_C2R, in, nullptr, nullptr, dout[l], f.negate, 0, h->rows)) return e2;
        h->tf_valid = false;                      // tr[0] was scratch
    }
    return team_fence(T);       // tr[0] has been consumed everywhere before anybody's next exchange pushes into it
}

// both strain diagnostics from ONE set of the three second derivatives of psi (psi_xy -> real_b, psi_xx -> real_c,
// psi_yy -> real_a); either output list may be null, and an output may be real_a only when it is the sole output
static int team_diagnostics(Team *T, float *const *tfil, float *const *deform)
{
    float *a[16], *b[16], *c[16];
    for (int l = 0; l < T->nlocal; ++l) { a[l] = T->local[l]->real_a; b[l] = T->local[l]->real_b; c[l] = T->local[l]->real_c; }
    if (int e = team_inverse(T, psi_second_ops[0], b)) return e;
    if (int e = team_inverse(T, psi_second_ops[1], c)) return e;
    if (int e = team_inverse(T, psi_second_ops[2], a)) return e;
    for (int l = 0; l < T->nlocal; ++l) {
        xfb_handle h = T->local[l];
        const long long n = (long long)h->grids;
        if (tfil && launch_strain(h, b[l], c[l], a[l], tfil[l], n, XFB_TFIL)) return XFB_E_CUDA;
        if (deform && launch_strain(h, b[l], c[l], a[l], deform[l], n, XFB_DEFORM)) return XFB_E_CUDA;
    }
    return 0;
}

static int team_get_field(Team *T, int which, float *const *dout)
{
    if (which == XFB_TRACER && !T->local[0]->has_tracer) return fail(XFB_E_STATE, "XFB_TRACER before xfb_set_tracer");
    if (which == XFB_TFIL) return team_diagnostics(T, dout, nullptr);
    if (which == XFB_DEFORM) return team_diagnostics(T, nullptr, dout);
    const FieldOps *f = field_ops(which);
    if (!f) return fail(XFB_E_ARG, "bad field id %d", which);
    return team_inverse(T, *f, dout, which == XFB_TRACER);
}

// effective-diffusivity histograms: zeta, zeta_x, zeta_y of the local rows, binned per rank into `d[l]` (2 * nbins doubles,
// device); the caller reduces over the ranks
static int team_keff_hist(Team *T, int nbins, float cmin, float cmax, double *const *d, bool tracer_state = false)
{
    float *a[16], *b[16], *c[16];
    for (int l = 0; l < T->nlocal; ++l) { a[l] = T->local[l]->real_a; b[l] = T->local[l]->real_b; c[l] = T->local[l]->real_c; }
    if (int e = team_inverse(T, *field_ops(XFB_VORT), a, tracer_state)) return e;
    if (int e = team_inverse(T, *field_ops(XFB_DVORTDX), b, tracer_state)) return e;
    if (int e = team_inverse(T, *field_ops(XFB_DVORTDY), c, tracer_state)) return e;
    // the inverses above use the spectral scratch arrays the caller may have taken `d` from: zero it only now
    CK(cudaMemsetAsync(d[0], 0, sizeof(double) * 2 * nbins, T->local[0]->stream));
    for (int l = 1; l < T->nlocal; ++l)
        if (d[l] != d[0]) CK(cudaMemsetAsync(d[l], 0, sizeof(double) * 2 * nbins, T->local[l]->stream));
    for (int l = 0; l < T->nlocal; ++l) {
        xfb_handle h = T->local[l];
        if (int e = launch_keff_hist(h, a[l], b[l], c[l], (long long)h->grids, nbins, cmin, cmax, d[l], d[l] + nbins)) return e;
    }
    return 0;
}

// ---- entry points used by xfb_api.cu for NCCL handles ----------------------------------------------------
int dist_keff_hist(xfb_handle h, int nbins, float cmin, float cmax, double *area, double *grad2, bool tracer_state)
{
    if (h->team->loopback) return fail(XFB_E_STATE, "loopback ranks are driven through xfb_loopback_*");
    double *d = (double *)h->spec_a;                 // free scratch of >= 2 * 2048 doubles once the inverses are done
    if (int e = team_keff_hist(h->team, nbins, cmin, cmax, &d, tracer_state)) return e;
    // one all-reduce of the 2 * nbins partial sums over the ranks (SURVEY.md 8e)
    NCK(g_nccl.AllReduce(d, d, (size_t)2 * nbins, ncclDouble, ncclSum, h->team->comm, h->stream));
    return keff_hist_finish(h, d, nbins, area, grad2);
}

int dist_diagnostics(xfb_handle h, float *tfil_rows, float *deform_rows)
{
    if (h->team->loopback) return fail(XFB_E_STATE, "loopback ranks are driven through xfb_loopback_*");
    const size_t bytes = sizeof(float) * h->grids;
    // host outputs are produced in spectral scratch (>= grids floats) that the last team_inverse has finished with
    float *dt = tfil_rows ? (float *)stage_out_target(tfil_rows, h->spec_b) : nullptr;
    float *dd = deform_rows ? (float *)stage_out_target(deform_rows, h->jint) : nullptr;
    if (int e = team_diagnostics(h->team, dt ? &dt : nullptr, dd ? &dd : nullptr)) return e;
    if (tfil_rows && stage_out(h, tfil_rows, dt, bytes, false)) return XFB_E_CUDA;
    if (deform_rows && stage_out(h, deform_rows, dd, bytes, false)) return XFB_E_CUDA;
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

int dist_set_vorticity(xfb_handle h, const float *vort_rows)
{
    if (h->team->loopback) return fail(XFB_E_STATE, "loopback ranks are driven through xfb_loopback_*");
    const void *din;
    if (stage_in(h, vort_rows, h->real_a, sizeof(float) * h->grids, &din)) return XFB_E_CUDA;
    const float *rows = (const float *)din;
    if (int e = team_set_vorticity(h->team, &rows)) return e;
    if (!is_device_ptr(vort_rows)) CK(cudaStreamSynchronize(h->stream));
    return 0;
}

// the passive tracer's initial field (device pointer, local rows): y pass, exchange, x pass into c0; collective
int dist_set_tracer(xfb_handle h, const float *tracer_rows_dev)
{
    if (h->team->loopback) return fail(XFB_E_STATE, "loopback ranks are driven through xfb_loopback_*");
    return team_set_vorticity(h->team, &tracer_rows_dev, true);
}

int dist_step(xfb_handle h, int nsteps, float dt)
{
    if (h->team->loopback) return fail(XFB_E_STATE, "loopback ranks are driven through xfb_loopback_*");
    return team_step(h->team, nsteps, dt);
}

int dist_get_field(xfb_handle h, int which, float *out_rows)
{
    if (h->team->loopback) return fail(XFB_E_STATE, "loopback ranks are driven through xfb_loopback_*");
    float *dout = (float *)stage_out_target(out_rows, h->real_a);
    if (int e = team_get_field(h->team, which, &dout)) return e;
    return stage_out(h, out_rows, dout, sizeof(float) * h->grids);
}

// quadratic invariants and shell spectra: every rank reduces its own column chunks, one all-reduce of the 3 + 2 * nshells
// sums (nothing is written that a peer reads: no exchange, no fence); collective
int dist_energy_spectrum(xfb_handle h, int which, int nshells, double *totals, double *e, double *z)
{
    if (h->team->loopback) return fail(XFB_E_STATE, "loopback ranks are driven through xfb_loopback_*");
    if (energy_spectrum_scratch(h)) return XFB_E_CUDA;
    const size_t n = 3 + 2 * (size_t)nshells;
    CK(cudaMemsetAsync(h->espec, 0, sizeof(double) * n, h->stream));
    if (int r = launch_energy_spectrum(h, which == XFB_TRACER ? h->c0 : h->z0, nshells, h->espec)) return r;
    NCK(g_nccl.AllReduce(h->espec, h->espec, n, ncclDouble, ncclSum, h->team->comm, h->stream));
    return energy_spectrum_finish(h, h->espec, nshells, totals, e, z);
}

// spectral budget: the terms of every rank (collective exchanges), the reduction of its own column chunks, one all-reduce
// of the 6 + 6 * nshells sums.  Every rank runs the source pass: no rank knows whether a peer has a source.
int dist_spectral_budget(xfb_handle h, int nshells, double *totals, double *budget)
{
    if (h->team->loopback) return fail(XFB_E_STATE, "loopback ranks are driven through xfb_loopback_*");
    if (spectral_budget_scratch(h)) return XFB_E_CUDA;
    if (int r = team_budget_terms(h->team, true)) return r;
    const size_t n = XFB_BUDGET_N * (1 + (size_t)nshells);
    CK(cudaMemsetAsync(h->bspec, 0, sizeof(double) * n, h->stream));
    if (int r = launch_spectral_budget(h, h->z0, h->spec_a, h->spec_b, nshells, h->bspec)) return r;
    NCK(g_nccl.AllReduce(h->bspec, h->bspec, n, ncclDouble, ncclSum, h->team->comm, h->stream));
    return spectral_budget_finish(h, h->bspec, nshells, totals, budget);
}

void dist_release(xfb_handle h)
{
    Team *T = h->team;
    if (!T) return;
    if (T->loopback) return;                      // owned by xfb_loopback_destroy
    cudaSetDevice(h->device);
    cudaStreamSynchronize(h->stream);
    cudaStreamSynchronize(h->comm_stream);
    for (int q = 0; q < T->nranks; ++q)
        if (h->p2p && q != h->rank && h->peer_recv[q]) cudaIpcCloseMemHandle(h->peer_recv[q]);
    if (T->comm) g_nccl.CommDestroy(T->comm);
    delete T;
    h->team = nullptr;
    destroy_impl(h);
}

}  // namespace xfb

using namespace xfb;

// ---- C ABI ---------------------------------------------------------------------------------------------------
extern "C" int xfb_nccl_unique_id(char *id128)
{
    if (!id128) return fail(XFB_E_ARG, "null id buffer");
    if (nccl_load()) return XFB_E_NCCL;
    ncclUniqueId id;
    NCK(g_nccl.GetUniqueId(&id));
    static_assert(sizeof(id) == 128, "ncclUniqueId is 128 bytes");
    memcpy(id128, &id, 128);
    return 0;
}

extern "C" int xfb_create_dist(xfb_handle *out, int nx, int ny, float lx, float ly, float nu, int device, int rank, int nranks,
                               int nchunks, const char *id128)
{
    if (!out) return fail(XFB_E_ARG, "null handle pointer");
    if (nranks == 1) return create_impl(out, nx, ny, lx, ly, nu, 1, device, 0, 1, 1);
    if (!id128) return fail(XFB_E_ARG, "xfb_create_dist: null unique id");
    if (nranks > 16) return fail(XFB_E_ARG, "xfb_create_dist: at most 16 ranks");
    if (nccl_load()) return XFB_E_NCCL;
    if (int e = create_impl(out, nx, ny, lx, ly, nu, 1, device, rank, nranks, nchunks)) return e;
    xfb_handle h = *out;
    if ((h->rows / nchunks) % 2 != 0 || h->rows % nchunks != 0) {
        destroy_impl(h);
        *out = nullptr;
        return fail(XFB_E_SIZE, "xfb_create_dist: %d local rows do not split into %d even chunks", h->rows, nchunks);
    }
    Team *T = new (std::nothrow) Team();
    if (!T) {
        destroy_impl(h);
        *out = nullptr;
        return fail(XFB_E_ARG, "out of host memory");
    }
    memset(T, 0, sizeof(*T));
    T->nranks = nranks; T->nlocal = 1; T->local[0] = h; T->loopback = false;
    ncclUniqueId id;
    memcpy(&id, id128, 128);
    ncclResult_t r = g_nccl.CommInitRank(&T->comm, nranks, id, rank);
    if (r != ncclSuccess) {
        delete T;
        destroy_impl(h);
        *out = nullptr;
        return fail(XFB_E_NCCL, "ncclCommInitRank: %s", g_nccl.GetErrorString(r));
    }
    h->team = T;
    h->ev_a2a = new std::vector<cudaEvent_t>();
    // peer-to-peer transport: export the receive block, gather everybody's handle with NCCL, map the peers' blocks.
    // XFB_SLAB_NCCL=1 keeps the grouped ncclSend/ncclRecv transport (A/B knob and fallback where IPC is not possible).
    const char *force_nccl = getenv("XFB_SLAB_NCCL");
    if (!(force_nccl && atoi(force_nccl) != 0)) {
        cudaIpcMemHandle_t mine, *all_d = nullptr;
        std::vector<cudaIpcMemHandle_t> all(nranks);
        bool ok = cudaIpcGetMemHandle(&mine, h->recv_block) == cudaSuccess &&
                  cudaMalloc((void **)&all_d, sizeof(mine) * nranks) == cudaSuccess;
        if (ok) {
            cudaMemcpyAsync(all_d + rank, &mine, sizeof(mine), cudaMemcpyHostToDevice, h->comm_stream);
            ok = g_nccl.AllGather(all_d + rank, all_d, sizeof(mine), ncclChar, T->comm, h->comm_stream) == ncclSuccess &&
                 cudaMemcpyAsync(all.data(), all_d, sizeof(mine) * nranks, cudaMemcpyDeviceToHost, h->comm_stream) == cudaSuccess &&
                 cudaStreamSynchronize(h->comm_stream) == cudaSuccess;
        }
        int mapped = ok ? 1 : 0;
        for (int q = 0; ok && q < nranks; ++q) {
            if (q == rank) { h->peer_recv[q] = h->recv_block; continue; }
            void *ptr = nullptr;
            if (cudaIpcOpenMemHandle(&ptr, all[q], cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { mapped = 0; cudaGetLastError(); break; }
            h->peer_recv[q] = (cpx *)ptr;
        }
        if (all_d) cudaFree(all_d);
        // everybody must agree on the transport: min over ranks of `mapped`
        float flag = (float)mapped, *flag_d = h->sync_buf;
        cudaMemcpyAsync(flag_d, &flag, sizeof(float), cudaMemcpyHostToDevice, h->comm_stream);
        g_nccl.AllReduce(flag_d, flag_d, 1, ncclFloat, ncclMin, T->comm, h->comm_stream);
        cudaMemcpyAsync(&flag, flag_d, sizeof(float), cudaMemcpyDeviceToHost, h->comm_stream);
        cudaStreamSynchronize(h->comm_stream);
        h->p2p = flag > 0.5f;
        if (!h->p2p)                       // some rank could not map its peers: nobody uses the mappings, give them back
            for (int q = 0; q < nranks; ++q) {
                if (q != rank && h->peer_recv[q]) cudaIpcCloseMemHandle(h->peer_recv[q]);
                h->peer_recv[q] = nullptr;
            }
        // who moves the bytes: copy engines, or a few CTAs of plain loads/stores (XFB_SLAB_PUSH=sm|ce).  The persistent
        // stepper kernels (NX, NY <= 8192) leave no SM free for a concurrent push kernel, so those grids default to ce.
        const char *push = getenv("XFB_SLAB_PUSH");
        h->push_sm = push ? (strcmp(push, "sm") == 0) : (nx > 8192 || ny > 8192);
        // CTAs per segment of the push kernel: a column -> row exchange of one chunk has nranks * 4 segments; enough CTAs to
        // keep NVLink busy without starving the transform kernels (8 GPUs at 16384^2: 1 -> 8.7, 2 -> 7.7, 4 -> 7.9 ms per
        // step; on 2 GPUs 2 CTAs per segment = 16 CTAs in all only reached 187 GB/s and the exchange bounded the step: 34.3 ms)
        // 2 GPUs: 8 -> 25.4, 16 -> 24.6, 32 -> 25.6 ms per step
        h->push_blocks = nranks >= 8 ? 2 : 32 / nranks;
        if (const char *pb = getenv("XFB_SLAB_PUSH_BLOCKS")) h->push_blocks = atoi(pb) < 1 ? 1 : atoi(pb);
        cudaMemsetAsync(h->sync_buf, 0, sizeof(float), h->comm_stream);
        cudaStreamSynchronize(h->comm_stream);
        if (h->p2p)
            if (int e = build_panel_table(h, h->peer_recv)) {
                dist_release(h);
                *out = nullptr;
                return e;
            }
    }
    return 0;
}

extern "C" int xfb_slab_transport(xfb_handle h)
{
    if (!h || h->nranks <= 1) return 0;
    return h->p2p ? (h->push_sm ? 3 : 2) : 1;   // 3: SM push kernel, 2: copy-engine pushes (both over CUDA IPC peer mappings), 1: ncclSend/ncclRecv
}

extern "C" int xfb_slab_fused(xfb_handle h)
{
    if (!h || h->nranks <= 1) return 0;
    return h->panel_base ? 1 : 0;
}

extern "C" int xfb_profile_read_a2a(xfb_handle h, double *a2a_ms, long long *exchanges)
{
    if (!h || !a2a_ms || !exchanges) return fail(XFB_E_ARG, "null argument");
    *a2a_ms = 0.0;
    *exchanges = 0;
    if (!h->ev_a2a) return 0;
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaStreamSynchronize(h->comm_stream));
    *exchanges = (long long)(h->ev_a2a_used / 2);
    for (size_t i = 0; i + 1 < h->ev_a2a_used; i += 2) {
        float ms = 0.f;
        CK(cudaEventElapsedTime(&ms, (*h->ev_a2a)[i], (*h->ev_a2a)[i + 1]));
        *a2a_ms += ms;
    }
    return 0;
}

// ---- loopback team: all ranks in this process on one device (slab indexing testable on a single GPU) ------
struct xfb_loopback_s {
    Team team;
    int nx, ny;
    float *full;             // device scratch, one full field
};

// rows[r] = rank r's rows of `full` (one whole field on the device, as L->full); all null when `full` is
static void rank_rows(const xfb_loopback_s *L, float *full, float **rows)
{
    for (int r = 0; r < L->team.nranks; ++r) rows[r] = full ? full + (size_t)r * L->team.local[0]->rows * L->ny : nullptr;
}

extern "C" int xfb_loopback_create(xfb_loopback_s **out, int nx, int ny, float lx, float ly, float nu, int device, int nranks,
                                   int nchunks)
{
    if (!out) return fail(XFB_E_ARG, "null pointer");
    *out = nullptr;
    if (nranks < 2 || nranks > 16) return fail(XFB_E_ARG, "xfb_loopback_create: 2..16 ranks");
    xfb_loopback_s *L = new (std::nothrow) xfb_loopback_s();
    if (!L) return fail(XFB_E_ARG, "out of host memory");
    memset(L, 0, sizeof(*L));
    L->nx = nx; L->ny = ny;
    L->team.nranks = nranks; L->team.nlocal = nranks; L->team.loopback = true;
    // a failure releases the ranks created so far
    auto bail = [&](int e) {
        for (int r = nranks - 1; r >= 0; --r) {
            xfb_handle h = L->team.local[r];
            if (!h) continue;
            h->team = nullptr;
            if (r > 0 && h->stream == L->team.local[0]->stream) h->stream = nullptr;     // shared with rank 0
            destroy_impl(h);
        }
        if (L->full) cudaFree(L->full);
        delete L;
        return e;
    };
    for (int r = 0; r < nranks; ++r) {
        xfb_handle h;
        if (int e = create_impl(&h, nx, ny, lx, ly, nu, 1, device, r, nranks, nchunks)) return bail(e);
        L->team.local[r] = h;
        if (h->rows % nchunks != 0 || (h->rows / nchunks) % 2 != 0)
            return bail(fail(XFB_E_SIZE, "xfb_loopback_create: %d local rows do not split into %d even chunks", h->rows, nchunks));
        // every rank works on rank 0's stream: program order is the only synchronisation needed
        if (r > 0) {
            cudaStreamDestroy(h->stream);
            h->stream = L->team.local[0]->stream;
        }
        h->team = &L->team;
    }
    {
        cpx *recv[16];
        for (int r = 0; r < nranks; ++r) recv[r] = L->team.local[r]->recv_block;
        for (int r = 0; r < nranks; ++r)
            if (int e = build_panel_table(L->team.local[r], recv)) return bail(e);
    }
    if (dev_alloc((void **)&L->full, sizeof(float) * (size_t)nx * ny)) return bail(XFB_E_CUDA);
    *out = L;
    return 0;
}

extern "C" int xfb_loopback_destroy(xfb_loopback_s *L)
{
    if (!L) return 0;
    cudaStreamSynchronize(L->team.local[0]->stream);
    for (int r = L->team.nranks - 1; r >= 0; --r) {
        xfb_handle h = L->team.local[r];
        h->team = nullptr;
        if (r > 0) CK(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));   // give it back a stream of its own to destroy
        destroy_impl(h);
    }
    cudaFree(L->full);
    delete L;
    return 0;
}

extern "C" int xfb_loopback_set_vorticity(xfb_loopback_s *L, const float *vort_full_host)
{
    if (!L || !vort_full_host) return fail(XFB_E_ARG, "null argument");
    xfb_handle h0 = L->team.local[0];
    CK(cudaSetDevice(h0->device));
    CK(cudaMemcpyAsync(L->full, vort_full_host, sizeof(float) * (size_t)L->nx * L->ny, cudaMemcpyHostToDevice, h0->stream));
    float *rows[16];
    rank_rows(L, L->full, rows);
    if (int e = team_set_vorticity(&L->team, rows)) return e;
    CK(cudaStreamSynchronize(h0->stream));
    return 0;
}

extern "C" int xfb_loopback_set_source(xfb_loopback_s *L, const float *src_full_host)
{
    if (!L) return fail(XFB_E_ARG, "null argument");
    for (int r = 0; r < L->team.nranks; ++r) {
        xfb_handle h = L->team.local[r];
        if (int e = xfb_set_source(h, 0, src_full_host ? src_full_host + (size_t)r * h->rows * L->ny : nullptr)) return e;
    }
    return 0;
}

extern "C" int xfb_loopback_set_tracer(xfb_loopback_s *L, const float *tracer_full_host, float kappa)
{
    if (!L || !tracer_full_host) return fail(XFB_E_ARG, "null argument");
    xfb_handle h0 = L->team.local[0];
    CK(cudaSetDevice(h0->device));
    for (int r = 0; r < L->team.nranks; ++r) {
        xfb_handle h = L->team.local[r];
        if (tracer_state_alloc(h)) return XFB_E_CUDA;
        h->has_tracer = true;
        h->kappa = kappa;
    }
    CK(cudaMemcpyAsync(L->full, tracer_full_host, sizeof(float) * (size_t)L->nx * L->ny, cudaMemcpyHostToDevice, h0->stream));
    float *rows[16];
    rank_rows(L, L->full, rows);
    if (int e = team_set_vorticity(&L->team, rows, true)) return e;
    CK(cudaStreamSynchronize(h0->stream));
    return 0;
}

// the same linear terms on every rank of the team (xfb_set_linear_terms is per rank and needs no communication)
extern "C" int xfb_loopback_set_linear_terms(xfb_loopback_s *L, float beta, float mu, float nu_h, int order)
{
    if (!L) return fail(XFB_E_ARG, "null argument");
    for (int r = 0; r < L->team.nranks; ++r)
        if (int e = xfb_set_linear_terms(L->team.local[r], beta, mu, nu_h, order)) return e;
    return 0;
}

extern "C" int xfb_loopback_step(xfb_loopback_s *L, int nsteps, float dt)
{
    if (!L) return fail(XFB_E_ARG, "null argument");
    if (!L->team.local[0]->have_state) return fail(XFB_E_STATE, "xfb_loopback_step before xfb_loopback_set_vorticity");
    CK(cudaSetDevice(L->team.local[0]->device));
    return team_step(&L->team, nsteps, dt);
}

extern "C" int xfb_loopback_get_field(xfb_loopback_s *L, int which, float *out_full_host)
{
    if (!L || !out_full_host) return fail(XFB_E_ARG, "null argument");
    xfb_handle h0 = L->team.local[0];
    if (!h0->have_state) return fail(XFB_E_STATE, "xfb_loopback_get_field before xfb_loopback_set_vorticity");
    CK(cudaSetDevice(h0->device));
    float *rows[16];
    rank_rows(L, L->full, rows);
    if (int e = team_get_field(&L->team, which, rows)) return e;
    CK(cudaMemcpyAsync(out_full_host, L->full, sizeof(float) * (size_t)L->nx * L->ny, cudaMemcpyDeviceToHost, h0->stream));
    CK(cudaStreamSynchronize(h0->stream));
    return 0;
}

extern "C" int xfb_loopback_get_diagnostics(xfb_loopback_s *L, float *tfil_full_host, float *deform_full_host)
{
    if (!L || (!tfil_full_host && !deform_full_host)) return fail(XFB_E_ARG, "null argument");
    xfb_handle h0 = L->team.local[0];
    if (!h0->have_state) return fail(XFB_E_STATE, "xfb_loopback_get_diagnostics before xfb_loopback_set_vorticity");
    CK(cudaSetDevice(h0->device));
    const size_t n = (size_t)L->nx * L->ny;
    float *second = nullptr;
    if (tfil_full_host && deform_full_host && dev_alloc((void **)&second, sizeof(float) * n)) return XFB_E_CUDA;
    float *t_rows[16], *d_rows[16];
    float *tbuf = tfil_full_host ? L->full : nullptr, *dbuf = deform_full_host ? (tfil_full_host ? second : L->full) : nullptr;
    rank_rows(L, tbuf, t_rows);
    rank_rows(L, dbuf, d_rows);
    int e = team_diagnostics(&L->team, tbuf ? t_rows : nullptr, dbuf ? d_rows : nullptr);
    if (!e && tbuf) e = cudaMemcpyAsync(tfil_full_host, tbuf, sizeof(float) * n, cudaMemcpyDeviceToHost, h0->stream) != cudaSuccess;
    if (!e && dbuf) e = cudaMemcpyAsync(deform_full_host, dbuf, sizeof(float) * n, cudaMemcpyDeviceToHost, h0->stream) != cudaSuccess;
    cudaStreamSynchronize(h0->stream);
    if (second) cudaFree(second);
    return e ? XFB_E_CUDA : 0;
}

extern "C" int xfb_loopback_get_keff_hist(xfb_loopback_s *L, int nbins, float cmin, float cmax, double *area, double *grad2)
{
    if (!L) return fail(XFB_E_ARG, "bad histogram arguments");
    if (int e = keff_hist_args(nbins, cmin, cmax, area, grad2)) return e;
    xfb_handle h0 = L->team.local[0];
    if (!h0->have_state) return fail(XFB_E_STATE, "xfb_loopback_get_keff_hist before xfb_loopback_set_vorticity");
    CK(cudaSetDevice(h0->device));
    // all ranks share the device and the stream: their kernels accumulate into ONE buffer (the all-reduce of the NCCL path)
    double *d[16];
    for (int r = 0; r < L->team.nranks; ++r) d[r] = (double *)L->full;
    if (int e = team_keff_hist(&L->team, nbins, cmin, cmax, d)) return e;
    return keff_hist_finish(h0, d[0], nbins, area, grad2);
}

extern "C" int xfb_loopback_get_energy_spectrum(xfb_loopback_s *L, int which, int nshells, double *totals, double *e, double *z)
{
    if (!L) return fail(XFB_E_ARG, "null argument");
    xfb_handle h0 = L->team.local[0];
    if (int r = energy_spectrum_args(h0, 0, which, nshells, totals, e, z, "xfb_loopback_")) return r;
    CK(cudaSetDevice(h0->device));
    // all ranks share the device and the stream: their launches add into rank 0's sums (the all-reduce of the NCCL path)
    if (energy_spectrum_scratch(h0)) return XFB_E_CUDA;
    CK(cudaMemsetAsync(h0->espec, 0, sizeof(double) * (3 + 2 * (size_t)nshells), h0->stream));
    for (int r = 0; r < L->team.nranks; ++r) {
        xfb_handle h = L->team.local[r];
        if (int e2 = launch_energy_spectrum(h, which == XFB_TRACER ? h->c0 : h->z0, nshells, h0->espec)) return e2;
    }
    return energy_spectrum_finish(h0, h0->espec, nshells, totals, e, z);
}

extern "C" int xfb_loopback_get_spectral_budget(xfb_loopback_s *L, int nshells, double *totals, double *budget)
{
    if (!L) return fail(XFB_E_ARG, "null argument");
    xfb_handle h0 = L->team.local[0];
    if (int r = spectral_budget_args(h0, 0, nshells, totals, budget, "xfb_loopback_")) return r;
    CK(cudaSetDevice(h0->device));
    bool with_src = false;
    for (int r = 0; r < L->team.nranks; ++r) with_src |= L->team.local[r]->has_src;
    if (spectral_budget_scratch(h0)) return XFB_E_CUDA;
    if (int r = team_budget_terms(&L->team, with_src)) return r;
    // all ranks share the device and the stream: their launches add into rank 0's sums (the all-reduce of the NCCL path)
    CK(cudaMemsetAsync(h0->bspec, 0, sizeof(double) * XFB_BUDGET_N * (1 + (size_t)nshells), h0->stream));
    for (int r = 0; r < L->team.nranks; ++r) {
        xfb_handle h = L->team.local[r];
        if (int e2 = launch_spectral_budget(h, h->z0, h->spec_a, with_src ? h->spec_b : nullptr, nshells, h0->bspec)) return e2;
    }
    return spectral_budget_finish(h0, h0->bspec, nshells, totals, budget);
}

extern "C" long long xfb_loopback_launch_count(xfb_loopback_s *L)
{
    long long n = 0;
    if (L)
        for (int r = 0; r < L->team.nranks; ++r) n += L->team.local[r]->launches;
    return n;
}

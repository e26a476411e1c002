// C ABI of the gadfly_b200 CUDA library (see include/gadfly_b200.h for the contract).
//
// Everything here is host-side plumbing: pointer classification and staging, batch
// descriptors, the heaviest-first work order, launch bookkeeping.  The arithmetic is in
// scan_fast.cu / scan_small.cu / scan_blk.cu / scan_ref.cu (O(N J^2) scans), sweep.cu (O(N J)
// sweeps) and psd.cu.
#include "../../include/gadfly_b200.h"
#include "common.cuh"

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <new>
#include <numeric>
#include <string>
#include <deque>
#include <vector>

namespace gf {
size_t scan_ref_scratch_bytes(int jmax, int grid);
cudaError_t launch_scan_ref(int mode, const ScanArgs &args, int jmax, int grid, double *scratch,
                            cudaStream_t stream);
cudaError_t launch_scan_fast(int mode, const ScanArgs &args, int jmax, int sm_count,
                             cudaStream_t stream, int *launches);
bool scan_small_supports(int mode, int jmax);
cudaError_t launch_scan_small(int mode, const ScanArgs &args, int jmax, int sm_count,
                              cudaStream_t stream, int *launches);
cudaError_t launch_sweep(int op, int64_t B, const int64_t *n_off, const int64_t *t_off,
                         const int64_t *j_off, const int64_t *w_off, const double *t,
                         const double *coef, const double *W, const double *Y, double *Z,
                         int jc_max, cudaStream_t stream);
cudaError_t launch_psd(int64_t B, const int64_t *j_off, const double *coef, const double *delta,
                       const double *omega, int64_t F, double *out, cudaStream_t stream);
cudaError_t measure_fp64_peak(int sm_count, cudaStream_t stream, double *flops);
cudaError_t launch_multi_prep(int64_t V, int64_t max_n, const int64_t *n_off_v, const int64_t *d_off,
                              const double *d, const double *normals, uint64_t seed, uint64_t seq0,
                              double *out, cudaStream_t stream);
cudaError_t launch_multi_quad(int64_t V, const int64_t *n_off_v, const int64_t *d_off, const double *d,
                              const double *z, double *quad, cudaStream_t stream);
struct FftPlan;
FftPlan *new_fft_plan();
void delete_fft_plan(FftPlan *fp);
cudaError_t launch_obs_power(FftPlan *fp, int64_t B, int64_t N, const double *flux, double d, int include_zero,
                             double2 *spec, double *power, cudaStream_t stream);
bool scan_blk_supports(int mode, int jmax);
cudaError_t launch_scan_blk(int mode, const ScanArgs &args, int sm_count, cudaStream_t stream);
int feed_max_terms();
cudaError_t launch_feed_hyper(const FeedArgs &A, double *sho_all, unsigned char *keep_all, int32_t *count,
                              cudaStream_t stream);
cudaError_t launch_feed_coef(const FeedArgs &A, const double *sho_all, const unsigned char *keep_all,
                             const int64_t *j_off, double *sho, double *coef, double *base, double *ddiag,
                             cudaStream_t stream);
cudaError_t launch_feed_sho(int64_t B, const int64_t *j_off, const double *sho, const double *delta,
                            double *coef, double *base, double *dterm, double *ddiag, int32_t *overdamped,
                            cudaStream_t stream);
cudaError_t launch_bandpass(int64_t B, const double *T, int64_t n_wl, const double *wl, const double *filt,
                            double *out, cudaStream_t stream);
cudaError_t launch_bin_power(int64_t B, int64_t F, int64_t nb, const int64_t *lo, const int64_t *cnt,
                             const double *x, const double *power, double constant, double *stat,
                             double *err, cudaStream_t stream);
cudaError_t launch_cond_mean(int64_t N, const double *t, int64_t M, const double *ts, int Jc,
                             const double *coef, const double *alpha, double *scratch, double *mu,
                             cudaStream_t stream);
}  // namespace gf

namespace {

constexpr int N_COUNTERS = 4096;

enum Slot {
    S_NOFF, S_TOFF, S_JOFF, S_WOFF, S_ORDER, S_COUNTER, S_T, S_Y, S_DIAG, S_COEF, S_DDIAG,
    S_OUT, S_OUTW, S_LOGDET, S_QUAD, S_STATUS, S_OMEGA, S_DELTA, S_W, S_SCRATCH,
    // k right-hand sides on one factor (gf_*_multi): the factor itself and the virtual-sequence descriptors
    S_MD, S_MW, S_MZ, S_MT, S_MDIAG, S_MCOEF, S_MDDIAG, S_VNOFF, S_VTOFF, S_VJOFF, S_VWOFF, S_VDOFF, S_VCOEF,
    S_MY, S_MOUT, S_MQUAD,
    // observed power spectrum
    S_FLUX, S_SPEC, S_POWER, S_BLO, S_BCNT, S_BAXIS, S_BSTAT, S_BERR, S_WIDE,
    // device feeder
    S_FM, S_FR, S_FT, S_FL, S_FALPHA, S_FGRAN, S_FMODES, S_FSHOALL, S_FKEEP, S_FCOUNT, S_FSHO, S_FBASE, S_FDDIAG, S_FWL, S_FFILT,
    N_SLOTS
};

// A staging buffer and the event of its last use (a kernel reading / writing it on the compute
// stream, or a copy on one of the copy streams).  Every slot is a ping-pong pair: a call takes
// the buffer whose last use has completed, so that the copies of one call never queue behind the
// kernel of the previous call (that is what lets H2D(y) run beside the sample kernel and D2H(x)
// beside the log-likelihood kernel); the second buffer is only allocated when that happens.
struct Buf {
    void *p = nullptr;
    size_t cap = 0;
    cudaEvent_t ev = nullptr;
    bool pending = false;
    uint64_t stamp = 0;
};
struct Pair {
    Buf b[2];
};

struct Deferred {
    void *user;            // pageable destination
    const char *pinned;    // where the copy-out stream puts it
    size_t bytes, ring_end;
    int64_t seq;
};
constexpr size_t BOUNCE_BYTES = 8u << 20;      // ring of pinned memory per handle
constexpr size_t BOUNCE_MAX = 1u << 20;        // larger pageable outputs are copied directly (host waits)

}  // namespace

struct gf_context {
    int device = 0;
    cudaStream_t stream = nullptr;       // compute
    cudaStream_t s_in = nullptr;         // host -> device staging copies
    cudaStream_t s_out = nullptr;        // device -> host copies of staged outputs
    cudaEvent_t ev_in = nullptr, ev_k = nullptr, ev_ext = nullptr;
    bool in_dirty = false;
    uint64_t stamp = 0;
    std::vector<Buf *> touched;          // staging buffers the kernel of the current call uses
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    int sm_count = 0;
    double fp64_flops = 0.0;
    int64_t launches = 0;
    int scan_path = GF_PATH_NONE;        // kernel of the most recent scan launch (gf_last_scan_path)
    bool timed = false;
    std::string err;
    gf::FftPlan *fft = nullptr;
    int *counters = nullptr;             // ring of zeroed work-queue heads (device)
    int counter_next = 0;
    cudaEvent_t ticket_ev[8] = {};       // completion tickets of GF_FLAG_ASYNC calls (gf_ticket / gf_wait)
    int64_t ticket_no[8] = {};
    int64_t ticket_seq[8] = {};          // last deferred output the ticket covers
    int64_t tickets = 0;
    // Small outputs into PAGEABLE host memory: a device-to-host cudaMemcpyAsync into pageable memory
    // returns only when the copy is done, i.e. it would hold the host until the kernel before it has
    // finished and GF_FLAG_ASYNC would not be asynchronous at all.  They go through a ring of pinned
    // memory instead and reach the caller's buffer in gf_synchronize / gf_wait / the next blocking call.
    char *bounce = nullptr;
    size_t bounce_head = 0, bounce_tail = 0;
    std::deque<Deferred> deferred;
    int64_t out_seq = 0;
    Pair buf[N_SLOTS];
};

namespace {

struct Guard {
    int prev = -1;
    explicit Guard(int dev) { cudaGetDevice(&prev); if (prev != dev) cudaSetDevice(dev); }
    // entry points that stage buffers: also drop what a failed earlier call may have left behind
    explicit Guard(gf_handle h) : Guard(h->device) { h->touched.clear(); }
    ~Guard() { if (prev >= 0) cudaSetDevice(prev); }
};

int fail(gf_handle h, int code, const char *what)
{
    if (h) {
        h->err = what;
        if (code > 0) { h->err += ": "; h->err += cudaGetErrorString((cudaError_t)code); }
    }
    return code;
}

#define GF_CUDA(h, expr)                                                      \
    do {                                                                      \
        cudaError_t e__ = (expr);                                             \
        if (e__ != cudaSuccess) return fail((h), (int)e__, #expr);            \
    } while (0)

enum { P_PAGEABLE = 0, P_PINNED = 1, P_DEVICE = 2 };
int pointer_kind(const void *p)
{
    cudaPointerAttributes a;
    cudaError_t e = cudaPointerGetAttributes(&a, p);
    if (e != cudaSuccess) { cudaGetLastError(); return P_PAGEABLE; }
    if (a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged) return P_DEVICE;
    return a.type == cudaMemoryTypeHost ? P_PINNED : P_PAGEABLE;
}
bool is_device_ptr(const void *p) { return pointer_kind(p) == P_DEVICE; }

// a slice of the pinned ring (nullptr: no room, or no ring)
char *bounce_alloc(gf_handle h, size_t bytes, size_t *ring_end)
{
    if (!h->bounce) return nullptr;
    bytes = (bytes + 63) & ~(size_t)63;
    if (h->deferred.empty()) h->bounce_head = h->bounce_tail = 0;
    size_t off;
    if (h->bounce_head >= h->bounce_tail) {
        if (h->bounce_head + bytes <= BOUNCE_BYTES) off = h->bounce_head;
        else if (bytes < h->bounce_tail) off = 0;
        else return nullptr;
    } else {
        if (h->bounce_head + bytes < h->bounce_tail) off = h->bounce_head;
        else return nullptr;
    }
    h->bounce_head = off + bytes;
    *ring_end = h->bounce_head;
    return h->bounce + off;
}

// the copy-out stream has completed every deferred output up to `upto`: hand them to the caller
void flush_deferred(gf_handle h, int64_t upto)
{
    while (!h->deferred.empty() && h->deferred.front().seq <= upto) {
        const Deferred &d = h->deferred.front();
        std::memcpy(d.user, d.pinned, d.bytes);
        h->bounce_tail = d.ring_end;
        h->deferred.pop_front();
    }
}

// A staging buffer of at least `bytes` for `slot` whose previous use is either complete or is
// ordered before everything `waiter` does from here on.
cudaError_t acquire(gf_handle h, int slot, size_t bytes, cudaStream_t waiter, Buf **out)
{
    Pair &pr = h->buf[slot];
    for (Buf &b : pr.b)
        if (b.pending && cudaEventQuery(b.ev) == cudaSuccess) b.pending = false;
    cudaGetLastError();   // cudaErrorNotReady of the queries above is not an error
    Buf *pick = nullptr;
    for (Buf &b : pr.b)
        if (!b.pending && b.cap >= bytes) { pick = &b; break; }
    if (!pick)
        for (Buf &b : pr.b)
            if (!b.pending) { pick = &b; break; }
    if (!pick) pick = (pr.b[0].stamp <= pr.b[1].stamp) ? &pr.b[0] : &pr.b[1];   // the older use
    if (pick->cap < bytes) {
        if (pick->pending) {
            cudaError_t e = cudaEventSynchronize(pick->ev);
            if (e != cudaSuccess) return e;
            pick->pending = false;
        }
        if (pick->p) { cudaFree(pick->p); pick->p = nullptr; pick->cap = 0; }
        const size_t cap = bytes + bytes / 8 + 256;
        cudaError_t e = cudaMalloc(&pick->p, cap);
        if (e != cudaSuccess) { pick->p = nullptr; return e; }
        pick->cap = cap;
    }
    if (!pick->ev) {
        cudaError_t e = cudaEventCreateWithFlags(&pick->ev, cudaEventDisableTiming);
        if (e != cudaSuccess) return e;
    }
    if (pick->pending) {
        cudaError_t e = cudaStreamWaitEvent(waiter, pick->ev, 0);
        if (e != cudaSuccess) return e;
    }
    *out = pick;
    return cudaSuccess;
}

// device scratch used by kernels only (never copied): ordered on the compute stream
cudaError_t reserve(gf_handle h, int slot, size_t bytes, void **p)
{
    Buf *b = nullptr;
    cudaError_t e = acquire(h, slot, bytes, h->stream, &b);
    if (e != cudaSuccess) return e;
    h->touched.push_back(b);
    *p = b->p;
    return cudaSuccess;
}

// Input that may live on the host: returns a device pointer valid for the kernel of this call
// (the copy runs on the copy-in stream; begin_kernel() makes the compute stream wait for it).
template <typename T>
cudaError_t stage_in(gf_handle h, int slot, const T *src, size_t count, const T **dev)
{
    if (!src || count == 0) { *dev = src; return cudaSuccess; }
    if (is_device_ptr(src)) { *dev = src; return cudaSuccess; }
    Buf *b = nullptr;
    cudaError_t e = acquire(h, slot, count * sizeof(T), h->s_in, &b);
    if (e != cudaSuccess) return e;
    e = cudaMemcpyAsync(b->p, src, count * sizeof(T), cudaMemcpyHostToDevice, h->s_in);
    h->in_dirty = true;
    h->touched.push_back(b);
    *dev = (const T *)b->p;
    return e;
}

// Output that may live on the host: device pointer now, copy back later.
template <typename T>
struct Out {
    T *user = nullptr;
    T *dev = nullptr;
    size_t count = 0;
    bool host = false;
    bool pageable = false;
    Buf *buf = nullptr;
};

template <typename T>
cudaError_t stage_out(gf_handle h, int slot, T *dst, size_t count, Out<T> *o)
{
    o->user = dst; o->count = count; o->host = false; o->pageable = false; o->dev = dst; o->buf = nullptr;
    if (!dst || count == 0) return cudaSuccess;
    const int kind = pointer_kind(dst);
    if (kind == P_DEVICE) return cudaSuccess;
    o->pageable = kind == P_PAGEABLE;
    cudaError_t e = acquire(h, slot, count * sizeof(T), h->stream, &o->buf);
    if (e != cudaSuccess) return e;
    o->dev = (T *)o->buf->p;
    o->host = true;
    return cudaSuccess;
}

// All inputs of this call are staged: the compute stream waits for the copy-in stream.
cudaError_t begin_kernel(gf_handle h)
{
    if (!h->in_dirty) return cudaSuccess;
    h->in_dirty = false;
    cudaError_t e = cudaEventRecord(h->ev_in, h->s_in);
    if (e != cudaSuccess) return e;
    return cudaStreamWaitEvent(h->stream, h->ev_in, 0);
}

// The kernel(s) of this call are launched: stamp the staging buffers they use, and let the
// copy-out stream wait for them.
cudaError_t end_kernel(gf_handle h)
{
    cudaError_t e = cudaEventRecord(h->ev_k, h->stream);
    if (e != cudaSuccess) return e;
    ++h->stamp;
    for (Buf *b : h->touched) {
        e = cudaEventRecord(b->ev, h->stream);
        if (e != cudaSuccess) return e;
        b->pending = true;
        b->stamp = h->stamp;
    }
    h->touched.clear();
    return cudaStreamWaitEvent(h->s_out, h->ev_k, 0);
}

template <typename T>
cudaError_t finish_out(gf_handle h, const Out<T> &o)
{
    if (!o.host || !o.user || o.count == 0) return cudaSuccess;
    const size_t bytes = o.count * sizeof(T);
    void *dst = o.user;
    size_t ring_end = 0;
    char *pinned = (o.pageable && bytes <= BOUNCE_MAX) ? bounce_alloc(h, bytes, &ring_end) : nullptr;
    if (pinned) {
        dst = pinned;
        h->deferred.push_back(Deferred{o.user, pinned, bytes, ring_end, ++h->out_seq});
    }
    cudaError_t e = cudaMemcpyAsync(dst, o.dev, bytes, cudaMemcpyDeviceToHost, h->s_out);
    if (e != cudaSuccess) return e;
    e = cudaEventRecord(o.buf->ev, h->s_out);
    o.buf->pending = true;
    o.buf->stamp = ++h->stamp;
    return e;
}

// outputs valid on return (unless GF_FLAG_ASYNC)
cudaError_t finish_call(gf_handle h, uint32_t flags)
{
    if (flags & GF_FLAG_ASYNC) return cudaSuccess;
    cudaError_t e = cudaStreamSynchronize(h->stream);
    if (e != cudaSuccess) return e;
    e = cudaStreamSynchronize(h->s_out);
    if (e == cudaSuccess) flush_deferred(h, h->out_seq);
    return e;
}

// Batch geometry shared by the scan entry points.
struct Geometry {
    int64_t total_n = 0;   // n_off[B]
    int64_t total_j = 0;   // j_off[B]
    int jmax = 0;          // widest state in the batch
    std::vector<int32_t> order;
};

int check_geometry(gf_handle h, int64_t B, const int64_t *n_off, const int64_t *t_off,
                   const int64_t *j_off, int64_t t_len, Geometry *g)
{
    if (!h) return GF_E_ARG;
    if (B < 0 || (B > 0 && (!n_off || !t_off || !j_off))) return fail(h, GF_E_ARG, "null batch descriptor");
    if (B > 0x7fffffff) return fail(h, GF_E_ARG, "batch too large");
    g->order.resize((size_t)B);
    std::vector<double> cost((size_t)B);
    for (int64_t b = 0; b < B; ++b) {
        int64_t N = n_off[b + 1] - n_off[b];
        int64_t Jc = j_off[b + 1] - j_off[b];
        if (N < 0 || Jc < 0) return fail(h, GF_E_ARG, "offsets must be non-decreasing");
        if (N > 0x7fffff00LL) return fail(h, GF_E_ARG, "a sequence is limited to 2^31 - 256 samples");
        if (2 * Jc > GF_MAX_J_WIDE) return fail(h, GF_E_TOO_WIDE, "state wider than GF_MAX_J_WIDE");
        if (t_off[b] < 0 || t_off[b] + N > t_len) return fail(h, GF_E_ARG, "t_off out of range");
        g->jmax = std::max(g->jmax, (int)(2 * Jc));
        cost[(size_t)b] = (double)N * (double)(4 * Jc * Jc + 8);
        g->order[(size_t)b] = (int32_t)b;
    }
    if (B > 0) {
        if (n_off[0] != 0 || j_off[0] < 0) return fail(h, GF_E_ARG, "offsets must start at 0");
        g->total_n = n_off[B];
        g->total_j = j_off[B];
    }
    // heaviest first: the persistent CTAs pull sequences from a queue
    std::stable_sort(g->order.begin(), g->order.end(),
                     [&](int32_t a, int32_t b) { return cost[(size_t)a] > cost[(size_t)b]; });
    return GF_OK;
}

struct Timer {
    gf_handle h;
    explicit Timer(gf_handle h_) : h(h_) { cudaEventRecord(h->ev0, h->stream); }
    ~Timer() { cudaEventRecord(h->ev1, h->stream); h->timed = true; }
};

int run_scan(gf_handle h, int mode, int64_t B, const int64_t *n_off, const int64_t *t_off,
             const int64_t *j_off, const int64_t *w_off, const double *t, int64_t t_len,
             const double *y, const double *diag, const double *coef, const double *ddiag,
             uint64_t seed, uint64_t seq0, double *out_x, double *out_W, int64_t w_len,
             double *logdet, double *quad, int32_t *status, uint32_t flags)
{
    Geometry g;
    int rc = check_geometry(h, B, n_off, t_off, j_off, t_len, &g);
    if (rc != GF_OK) return rc;
    if (B == 0) return GF_OK;
    if (!t || !coef || !ddiag || !status) return fail(h, GF_E_ARG, "null data pointer");
    Guard guard(h->device);

    gf::ScanArgs A;
    std::memset(&A, 0, sizeof(A));
    A.B = B;
    GF_CUDA(h, stage_in(h, S_NOFF, n_off, (size_t)B + 1, &A.n_off));
    GF_CUDA(h, stage_in(h, S_TOFF, t_off, (size_t)B, &A.t_off));
    GF_CUDA(h, stage_in(h, S_JOFF, j_off, (size_t)B + 1, &A.j_off));
    if (w_off) GF_CUDA(h, stage_in(h, S_WOFF, w_off, (size_t)B, &A.w_off));
    const int32_t *order_dev = nullptr;
    GF_CUDA(h, stage_in(h, S_ORDER, (const int32_t *)g.order.data(), (size_t)B, &order_dev));
    A.order = order_dev;
    {
        // Work-queue head of this launch: the next of a ring of pre-zeroed counters.  (Not a memset per
        // launch: a memset is a copy-engine operation, and behind a bulk H2D copy on that engine it
        // would hold the kernel back for the whole transfer -- the reason the H2D copy of the next
        // light curves did not overlap the running scan in round 1.)
        if (h->counter_next == N_COUNTERS) {
            GF_CUDA(h, cudaMemsetAsync(h->counters, 0, N_COUNTERS * sizeof(int), h->stream));
            h->counter_next = 0;
        }
        A.counter = h->counters + h->counter_next++;
    }
    // (the small, usually pageable arrays first: a pageable copy blocks the host until everything queued
    // before it on the copy-in stream has been copied -- behind the bulk arrays that would be their whole
    // transfer time)
    GF_CUDA(h, stage_in(h, S_COEF, coef, (size_t)g.total_j * 4, &A.coef));
    GF_CUDA(h, stage_in(h, S_DDIAG, ddiag, (size_t)B, &A.ddiag));
    GF_CUDA(h, stage_in(h, S_T, t, (size_t)t_len, &A.t));
    const bool shared_y = (flags & GF_FLAG_SHARED_Y) != 0;
    if (shared_y && mode != gf::MODE_LOGLIKE) return fail(h, GF_E_ARG, "GF_FLAG_SHARED_Y: log-likelihood only");
    A.y_like_t = shared_y ? 1 : 0;
    const size_t y_len = shared_y ? (size_t)t_len : (size_t)g.total_n;
    GF_CUDA(h, stage_in(h, S_Y, y, y_len, &A.y));
    GF_CUDA(h, stage_in(h, S_DIAG, diag, y_len, &A.diag));
    A.seed = seed;
    A.seq0 = seq0;

    Out<double> o_x, o_W, o_ld, o_q;
    Out<int32_t> o_st;
    GF_CUDA(h, stage_out(h, S_OUT, out_x, (size_t)g.total_n, &o_x));
    GF_CUDA(h, stage_out(h, S_OUTW, out_W, (size_t)w_len, &o_W));
    GF_CUDA(h, stage_out(h, S_LOGDET, logdet, (size_t)B, &o_ld));
    GF_CUDA(h, stage_out(h, S_QUAD, quad, (size_t)B, &o_q));
    GF_CUDA(h, stage_out(h, S_STATUS, status, (size_t)B, &o_st));
    A.out_x = o_x.dev; A.out_W = o_W.dev; A.quad = o_q.dev; A.status = o_st.dev;
    // the kernels always write logdet: give them scratch when the caller does not want it
    if (!o_ld.dev) {
        void *ld = nullptr;
        GF_CUDA(h, reserve(h, S_LOGDET, (size_t)B * sizeof(double), &ld));
        A.logdet = (double *)ld;
    } else {
        A.logdet = o_ld.dev;
    }

    GF_CUDA(h, begin_kernel(h));
    {
        Timer timer(h);
        if ((flags & GF_FLAG_REFERENCE_ORDER) || g.jmax > GF_MAX_J) {
            // reference order; a state wider than the register-resident kernels take (J > 176) lives
            // in L2-resident global scratch whatever the flags
            const int grid = (int)std::min<int64_t>(B, (int64_t)h->sm_count);
            const size_t bytes = gf::scan_ref_scratch_bytes(g.jmax, grid);
            void *state = nullptr;
            if (bytes) GF_CUDA(h, reserve(h, S_WIDE, bytes, &state));
            GF_CUDA(h, gf::launch_scan_ref(mode, A, g.jmax, grid, (double *)state, h->stream));
            h->launches += 1;
            h->scan_path = bytes ? GF_PATH_WIDE : GF_PATH_REF;
        } else if ((flags & GF_FLAG_BLOCKED) && gf::scan_blk_supports(mode, g.jmax)) {
            GF_CUDA(h, gf::launch_scan_blk(mode, A, h->sm_count, h->stream));
            h->launches += 1;
            h->scan_path = GF_PATH_BLOCKED;
        } else if (!(flags & GF_FLAG_WIDE_KERNEL) && gf::scan_small_supports(mode, g.jmax)) {
            // every sequence of the batch is narrow (J <= 32): one warp per sequence
            int n = 0;
            GF_CUDA(h, gf::launch_scan_small(mode, A, g.jmax, h->sm_count, h->stream, &n));
            h->launches += n;
            h->scan_path = GF_PATH_SMALL;
        } else {
            int n = 0;
            GF_CUDA(h, gf::launch_scan_fast(mode, A, g.jmax, h->sm_count, h->stream, &n));
            h->launches += n;
            h->scan_path = GF_PATH_FAST;
        }
    }

    GF_CUDA(h, end_kernel(h));
    // small outputs first: the caller's scalars do not wait behind the bulk copy
    GF_CUDA(h, finish_out(h, o_ld));
    GF_CUDA(h, finish_out(h, o_q));
    GF_CUDA(h, finish_out(h, o_st));
    GF_CUDA(h, finish_out(h, o_x));
    GF_CUDA(h, finish_out(h, o_W));
    GF_CUDA(h, finish_call(h, flags));
    return GF_OK;
}

}  // namespace

extern "C" {

int gf_create(int device, gf_handle *out)
{
    if (!out) return GF_E_ARG;
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess) return (int)e;
    if (device < 0 || device >= count) return GF_E_ARG;
    gf_context *h = new (std::nothrow) gf_context;
    if (!h) return GF_E_NOMEM;
    h->device = device;
    Guard guard(device);
    e = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&h->s_in, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&h->s_out, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->ev_in, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->ev_k, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->ev_ext, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreate(&h->ev0);
    if (e == cudaSuccess) e = cudaEventCreate(&h->ev1);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&h->sm_count, cudaDevAttrMultiProcessorCount, device);
    if (e == cudaSuccess) e = cudaMalloc((void **)&h->counters, N_COUNTERS * sizeof(int));
    if (e == cudaSuccess) e = cudaMemset(h->counters, 0, N_COUNTERS * sizeof(int));
    if (e == cudaSuccess) e = cudaHostAlloc((void **)&h->bounce, BOUNCE_BYTES, cudaHostAllocDefault);
    if (e != cudaSuccess) { gf_destroy(h); return (int)e; }
    *out = h;
    return GF_OK;
}

int gf_destroy(gf_handle h)
{
    if (!h) return GF_OK;
    Guard guard(h->device);
    for (cudaStream_t st : {h->stream, h->s_in, h->s_out}) if (st) cudaStreamSynchronize(st);
    for (auto &pr : h->buf)
        for (auto &b : pr.b) {
            if (b.p) cudaFree(b.p);
            if (b.ev) cudaEventDestroy(b.ev);
        }
    for (cudaEvent_t ev : {h->ev0, h->ev1, h->ev_in, h->ev_k, h->ev_ext}) if (ev) cudaEventDestroy(ev);
    for (cudaEvent_t ev : h->ticket_ev) if (ev) cudaEventDestroy(ev);
    for (cudaStream_t st : {h->stream, h->s_in, h->s_out}) if (st) cudaStreamDestroy(st);
    if (h->fft) gf::delete_fft_plan(h->fft);
    if (h->counters) cudaFree(h->counters);
    flush_deferred(h, h->out_seq);
    if (h->bounce) cudaFreeHost(h->bounce);
    delete h;
    return GF_OK;
}

int gf_synchronize(gf_handle h)
{
    if (!h) return GF_E_ARG;
    Guard guard(h->device);
    GF_CUDA(h, cudaStreamSynchronize(h->s_in));
    GF_CUDA(h, cudaStreamSynchronize(h->stream));
    GF_CUDA(h, cudaStreamSynchronize(h->s_out));
    flush_deferred(h, h->out_seq);
    return GF_OK;
}

int gf_wait_stream(gf_handle h, void *producer)
{
    if (!h) return GF_E_ARG;
    Guard guard(h->device);
    GF_CUDA(h, cudaEventRecord(h->ev_ext, (cudaStream_t)producer));
    GF_CUDA(h, cudaStreamWaitEvent(h->stream, h->ev_ext, 0));
    return GF_OK;
}

int64_t gf_ticket(gf_handle h)
{
    if (!h) return GF_E_ARG;
    Guard guard(h->device);
    const int64_t no = ++h->tickets;
    const int k = (int)(no & 7);
    if (!h->ticket_ev[k]) GF_CUDA(h, cudaEventCreateWithFlags(&h->ticket_ev[k], cudaEventDisableTiming));
    // everything issued so far: the kernels (compute stream), then the copies back (copy-out stream)
    GF_CUDA(h, cudaEventRecord(h->ev_ext, h->stream));
    GF_CUDA(h, cudaStreamWaitEvent(h->s_out, h->ev_ext, 0));
    GF_CUDA(h, cudaEventRecord(h->ticket_ev[k], h->s_out));
    h->ticket_no[k] = no;
    h->ticket_seq[k] = h->out_seq;
    return no;
}

int gf_wait(gf_handle h, int64_t ticket)
{
    if (!h) return GF_E_ARG;
    if (ticket <= 0 || ticket > h->tickets) return fail(h, GF_E_ARG, "unknown ticket");
    Guard guard(h->device);
    const int k = (int)(ticket & 7);
    // a ticket older than the ring has been overwritten by a later one: waiting for that is sufficient
    GF_CUDA(h, cudaEventSynchronize(h->ticket_ev[k]));
    flush_deferred(h, h->ticket_seq[k]);
    return GF_OK;
}

int gf_stream_wait(gf_handle h, void *consumer)
{
    if (!h) return GF_E_ARG;
    Guard guard(h->device);
    GF_CUDA(h, cudaEventRecord(h->ev_ext, h->stream));
    GF_CUDA(h, cudaStreamWaitEvent((cudaStream_t)consumer, h->ev_ext, 0));
    return GF_OK;
}

const char *gf_last_error(gf_handle h) { return h ? h->err.c_str() : "null handle"; }

void *gf_stream(gf_handle h) { return h ? (void *)h->stream : nullptr; }

int gf_device_info(gf_handle h, int *sm_count, double *fp64_flops, int measure)
{
    if (!h) return GF_E_ARG;
    Guard guard(h->device);
    if (sm_count) *sm_count = h->sm_count;
    if (measure && h->fp64_flops == 0.0) {
        GF_CUDA(h, gf::measure_fp64_peak(h->sm_count, h->stream, &h->fp64_flops));
        h->launches += 4;
    }
    if (fp64_flops) *fp64_flops = h->fp64_flops;
    return GF_OK;
}

int64_t gf_launch_count(gf_handle h) { return h ? h->launches : 0; }

int gf_last_scan_path(gf_handle h) { return h ? h->scan_path : GF_E_ARG; }

float gf_last_kernel_ms(gf_handle h)
{
    if (!h || !h->timed) return 0.0f;
    Guard guard(h->device);
    float ms = 0.0f;
    if (cudaEventSynchronize(h->ev1) != cudaSuccess) return 0.0f;
    if (cudaEventElapsedTime(&ms, h->ev0, h->ev1) != cudaSuccess) return 0.0f;
    return ms;
}

int gf_loglike_batched(gf_handle h, int64_t B, const int64_t *n_off, const int64_t *t_off,
                       const int64_t *j_off, const double *t, int64_t t_len, const double *y,
                       const double *diag, const double *coef, const double *ddiag,
                       double *logdet, double *quad, int32_t *status, uint32_t flags)
{
    if (!h) return GF_E_ARG;
    if (B > 0 && (!y || !logdet || !quad)) return fail(h, GF_E_ARG, "null data pointer");
    h->touched.clear();
    return run_scan(h, gf::MODE_LOGLIKE, B, n_off, t_off, j_off, nullptr, t, t_len, y, diag, coef,
                    ddiag, 0, 0, nullptr, nullptr, 0, logdet, quad, status, flags);
}

int gf_sample_batched(gf_handle h, int64_t B, const int64_t *n_off, const int64_t *t_off,
                      const int64_t *j_off, const double *t, int64_t t_len, const double *diag,
                      const double *coef, const double *ddiag, const double *normals,
                      uint64_t seed, uint64_t seq0, double *out, double *logdet, int32_t *status,
                      uint32_t flags)
{
    if (!h) return GF_E_ARG;
    if (B > 0 && !out) return fail(h, GF_E_ARG, "null output pointer");
    h->touched.clear();
    return run_scan(h, gf::MODE_SAMPLE, B, n_off, t_off, j_off, nullptr, t, t_len, normals, diag,
                    coef, ddiag, seed, seq0, out, nullptr, 0, logdet, nullptr, status, flags);
}

int gf_factor_batched(gf_handle h, int64_t B, const int64_t *n_off, const int64_t *t_off,
                      const int64_t *j_off, const int64_t *w_off, const double *t, int64_t t_len,
                      const double *diag, const double *coef, const double *ddiag, double *d,
                      double *W, double *logdet, int32_t *status, uint32_t flags)
{
    if (!h) return GF_E_ARG;
    if (B > 0 && !d) return fail(h, GF_E_ARG, "null output pointer");
    if (W && !w_off) return fail(h, GF_E_ARG, "W needs w_off");
    h->touched.clear();
    int64_t w_len = 0;
    if (W && B > 0 && n_off && j_off)
        for (int64_t b = 0; b < B; ++b)
            w_len = std::max(w_len, w_off[b] + (n_off[b + 1] - n_off[b]) * 2 * (j_off[b + 1] - j_off[b]));
    return run_scan(h, gf::MODE_FACTOR, B, n_off, t_off, j_off, W ? w_off : nullptr, t, t_len,
                    nullptr, diag, coef, ddiag, 0, 0, d, W, w_len, logdet, nullptr, status, flags);
}

int gf_sweep_batched(gf_handle h, int op, int64_t B, const int64_t *n_off, const int64_t *t_off,
                     const int64_t *j_off, const int64_t *w_off, const double *t, int64_t t_len,
                     const double *coef, const double *W, const double *Y, double *Z,
                     uint32_t flags)
{
    if (!h) return GF_E_ARG;
    if (op < 0 || op > 3) return fail(h, GF_E_ARG, "op must be 0..3");
    Geometry g;
    int rc = check_geometry(h, B, n_off, t_off, j_off, t_len, &g);
    if (rc != GF_OK) return rc;
    if (B == 0) return GF_OK;
    if (!t || !coef || !W || !Y || !Z || !w_off) return fail(h, GF_E_ARG, "null data pointer");
    Guard guard(h);
    int64_t w_len = 0;
    for (int64_t b = 0; b < B; ++b)
        w_len = std::max(w_len, w_off[b] + (n_off[b + 1] - n_off[b]) * 2 * (j_off[b + 1] - j_off[b]));
    const int64_t *d_noff, *d_toff, *d_joff, *d_woff;
    const double *d_t, *d_coef, *d_W, *d_Y;
    GF_CUDA(h, stage_in(h, S_NOFF, n_off, (size_t)B + 1, &d_noff));
    GF_CUDA(h, stage_in(h, S_TOFF, t_off, (size_t)B, &d_toff));
    GF_CUDA(h, stage_in(h, S_JOFF, j_off, (size_t)B + 1, &d_joff));
    GF_CUDA(h, stage_in(h, S_WOFF, w_off, (size_t)B, &d_woff));
    GF_CUDA(h, stage_in(h, S_T, t, (size_t)t_len, &d_t));
    GF_CUDA(h, stage_in(h, S_COEF, coef, (size_t)g.total_j * 4, &d_coef));
    GF_CUDA(h, stage_in(h, S_W, W, (size_t)w_len, &d_W));
    Out<double> o_z;
    // Z may alias Y: stage Y into the same slot the result is produced in
    if (!is_device_ptr(Z)) {
        GF_CUDA(h, stage_out(h, S_OUT, Z, (size_t)g.total_n, &o_z));
        if (!is_device_ptr(Y)) {
            // (on the compute stream: the buffer was acquired for it)
            GF_CUDA(h, cudaMemcpyAsync(o_z.dev, Y, (size_t)g.total_n * sizeof(double),
                                       cudaMemcpyHostToDevice, h->stream));
            d_Y = o_z.dev;
        } else {
            d_Y = Y;
        }
    } else {
        o_z.dev = Z;
        GF_CUDA(h, stage_in(h, S_Y, Y, (size_t)g.total_n, &d_Y));
    }
    GF_CUDA(h, begin_kernel(h));
    {
        Timer timer(h);
        GF_CUDA(h, gf::launch_sweep(op, B, d_noff, d_toff, d_joff, d_woff, d_t, d_coef, d_W, d_Y,
                                    o_z.dev, g.jmax / 2, h->stream));
        h->launches += 1;
    }
    GF_CUDA(h, end_kernel(h));
    GF_CUDA(h, finish_out(h, o_z));
    GF_CUDA(h, finish_call(h, flags));
    return GF_OK;
}

int gf_psd_batched(gf_handle h, int64_t B, const int64_t *j_off, const double *coef_base,
                   const double *delta, const double *omega, int64_t F, double *out,
                   uint32_t flags)
{
    if (!h) return GF_E_ARG;
    if (B < 0 || F < 0) return fail(h, GF_E_ARG, "negative size");
    if (B == 0 || F == 0) return GF_OK;
    if (!j_off || !coef_base || !omega || !out) return fail(h, GF_E_ARG, "null data pointer");
    for (int64_t b = 0; b < B; ++b)
        if (j_off[b + 1] < j_off[b]) return fail(h, GF_E_ARG, "offsets must be non-decreasing");
    Guard guard(h);
    const int64_t *d_joff;
    const double *d_coef, *d_delta, *d_omega;
    GF_CUDA(h, stage_in(h, S_JOFF, j_off, (size_t)B + 1, &d_joff));
    GF_CUDA(h, stage_in(h, S_COEF, coef_base, (size_t)j_off[B] * 4, &d_coef));
    GF_CUDA(h, stage_in(h, S_DELTA, delta, (size_t)B, &d_delta));
    GF_CUDA(h, stage_in(h, S_OMEGA, omega, (size_t)F, &d_omega));
    Out<double> o;
    GF_CUDA(h, stage_out(h, S_OUT, out, (size_t)B * (size_t)F, &o));
    GF_CUDA(h, begin_kernel(h));
    {
        Timer timer(h);
        GF_CUDA(h, gf::launch_psd(B, d_joff, d_coef, d_delta, d_omega, F, o.dev, h->stream));
        h->launches += (B + 65534) / 65535;
    }
    GF_CUDA(h, end_kernel(h));
    GF_CUDA(h, finish_out(h, o));
    GF_CUDA(h, finish_call(h, flags));
    return GF_OK;
}

int gf_conditional_mean(gf_handle h, int64_t N, const double *t, int64_t M, const double *ts,
                        int64_t Jc, const double *coef, const double *alpha, double *mu,
                        uint32_t flags)
{
    if (!h) return GF_E_ARG;
    if (N < 0 || M < 0 || Jc < 0) return fail(h, GF_E_ARG, "negative size");
    if (M == 0) return GF_OK;
    if (!ts || !mu || (N > 0 && (!t || !alpha)) || (Jc > 0 && !coef))
        return fail(h, GF_E_ARG, "null data pointer");
    if (Jc > 0x3fffffff) return fail(h, GF_E_ARG, "too many terms");
    Guard guard(h);
    const double *d_t, *d_ts, *d_coef, *d_alpha;
    GF_CUDA(h, stage_in(h, S_T, t, (size_t)N, &d_t));
    GF_CUDA(h, stage_in(h, S_OMEGA, ts, (size_t)M, &d_ts));
    GF_CUDA(h, stage_in(h, S_COEF, coef, (size_t)Jc * 4, &d_coef));
    GF_CUDA(h, stage_in(h, S_Y, alpha, (size_t)N, &d_alpha));
    void *scratch = nullptr;
    GF_CUDA(h, reserve(h, S_SCRATCH, (size_t)M * 2 * sizeof(double), &scratch));
    Out<double> o;
    GF_CUDA(h, stage_out(h, S_OUT, mu, (size_t)M, &o));
    GF_CUDA(h, begin_kernel(h));
    {
        Timer timer(h);
        GF_CUDA(h, gf::launch_cond_mean(N, d_t, M, d_ts, (int)Jc, d_coef, d_alpha,
                                        (double *)scratch, o.dev, h->stream));
        h->launches += 2;
    }
    GF_CUDA(h, end_kernel(h));
    GF_CUDA(h, finish_out(h, o));
    GF_CUDA(h, finish_call(h, flags));
    return GF_OK;
}

}  // extern "C"

// ---- k right-hand sides per sequence on one factor ------------------------------------------
namespace {

// mode 1: samples  out[b][r][:] = L_b (sqrt(d_b) o n_{b,r});   mode 0: quad[b][r] = z^T D^-1 z, z = L_b^-1 y_{b,r}
int run_multi(gf_handle h, int mode, int64_t B, const int64_t *n_off, const int64_t *t_off,
              const int64_t *j_off, const double *t, int64_t t_len, const double *diag,
              const double *coef, const double *ddiag, int64_t k, const double *in /* normals | y */,
              uint64_t seed, uint64_t seq0, double *out, double *logdet, double *quad, int32_t *status,
              uint32_t flags)
{
    if (!h) return GF_E_ARG;
    if (k < 1) return fail(h, GF_E_ARG, "k must be >= 1");
    Geometry g;
    int rc = check_geometry(h, B, n_off, t_off, j_off, t_len, &g);
    if (rc != GF_OK) return rc;
    if (B == 0) return GF_OK;
    if (!t || !coef || !ddiag || !status) return fail(h, GF_E_ARG, "null data pointer");
    if (B * k > 0x7fffffff) return fail(h, GF_E_ARG, "too many right-hand sides");
    Guard guard(h);

    // 1. the inputs the factor and the sweeps share, on the device once
    const double *d_t, *d_diag, *d_coef, *d_ddiag;
    GF_CUDA(h, stage_in(h, S_MT, t, (size_t)t_len, &d_t));
    GF_CUDA(h, stage_in(h, S_MDIAG, diag, (size_t)g.total_n, &d_diag));
    GF_CUDA(h, stage_in(h, S_MCOEF, coef, (size_t)g.total_j * 4, &d_coef));
    GF_CUDA(h, stage_in(h, S_MDDIAG, ddiag, (size_t)B, &d_ddiag));
    // 2. the factor: d[sum N], W[sum N J] in library scratch
    std::vector<int64_t> w_off((size_t)B);
    int64_t w_len = 0, max_n = 0;
    for (int64_t b = 0; b < B; ++b) {
        w_off[(size_t)b] = w_len;
        w_len += (n_off[b + 1] - n_off[b]) * 2 * (j_off[b + 1] - j_off[b]);
        max_n = std::max(max_n, n_off[b + 1] - n_off[b]);
    }
    void *d_d = nullptr, *d_W = nullptr;
    GF_CUDA(h, reserve(h, S_MD, (size_t)std::max<int64_t>(g.total_n, 1) * sizeof(double), &d_d));
    GF_CUDA(h, reserve(h, S_MW, (size_t)std::max<int64_t>(w_len, 1) * sizeof(double), &d_W));
    std::vector<Buf *> mine = h->touched;      // run_scan's end_kernel stamps and clears the list
    rc = run_scan(h, gf::MODE_FACTOR, B, n_off, t_off, j_off, w_off.data(), d_t, t_len, nullptr, d_diag,
                  d_coef, d_ddiag, 0, 0, (double *)d_d, (double *)d_W, w_len, logdet, nullptr, status,
                  flags | GF_FLAG_ASYNC);
    if (rc != GF_OK) return rc;
    h->touched = mine;
    // 3. virtual sequences v = b k + r: own samples, shared time stamps, factor and kernel
    const int64_t V = B * k;
    std::vector<int64_t> vn((size_t)V + 1), vt((size_t)V), vj((size_t)V + 1), vw((size_t)V), vd((size_t)V);
    std::vector<double> vcoef;
    vcoef.reserve((size_t)g.total_j * 4 * (size_t)k);
    vn[0] = 0; vj[0] = 0;
    for (int64_t b = 0; b < B; ++b) {
        const int64_t N = n_off[b + 1] - n_off[b], Jc = j_off[b + 1] - j_off[b];
        for (int64_t r = 0; r < k; ++r) {
            const size_t v = (size_t)(b * k + r);
            vn[v + 1] = vn[v] + N;
            vj[v + 1] = vj[v] + Jc;
            vt[v] = t_off[b];
            vw[v] = w_off[(size_t)b];
            vd[v] = n_off[b];
        }
    }
    const int64_t *d_vn, *d_vt, *d_vj, *d_vw, *d_vd;
    const double *d_vcoef = nullptr;
    GF_CUDA(h, stage_in(h, S_VNOFF, (const int64_t *)vn.data(), (size_t)V + 1, &d_vn));
    GF_CUDA(h, stage_in(h, S_VTOFF, (const int64_t *)vt.data(), (size_t)V, &d_vt));
    GF_CUDA(h, stage_in(h, S_VJOFF, (const int64_t *)vj.data(), (size_t)V + 1, &d_vj));
    GF_CUDA(h, stage_in(h, S_VWOFF, (const int64_t *)vw.data(), (size_t)V, &d_vw));
    GF_CUDA(h, stage_in(h, S_VDOFF, (const int64_t *)vd.data(), (size_t)V, &d_vd));
    {
        // the coefficient rows of sequence b, k times (the sweep kernel reads CSR rows per sequence)
        void *p = nullptr;
        GF_CUDA(h, reserve(h, S_VCOEF, (size_t)std::max<int64_t>(g.total_j * k, 1) * 4 * sizeof(double), &p));
        for (int64_t b = 0; b < B; ++b) {
            const int64_t Jc = j_off[b + 1] - j_off[b];
            for (int64_t r = 0; r < k; ++r)
                GF_CUDA(h, cudaMemcpyAsync((double *)p + 4 * vj[(size_t)(b * k + r)], d_coef + 4 * j_off[b],
                                           (size_t)Jc * 4 * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
        }
        d_vcoef = (const double *)p;
    }
    const size_t total_v = (size_t)g.total_n * (size_t)k;
    const double *d_in = nullptr;
    GF_CUDA(h, stage_in(h, S_MY, in, total_v, &d_in));
    if (mode == 1) {
        Out<double> o;
        GF_CUDA(h, stage_out(h, S_MOUT, out, total_v, &o));
        if (o.host) h->touched.push_back(o.buf);
        GF_CUDA(h, begin_kernel(h));
        {
            Timer timer(h);
            GF_CUDA(h, gf::launch_multi_prep(V, max_n, d_vn, d_vd, (const double *)d_d, d_in, seed, seq0, o.dev, h->stream));
            GF_CUDA(h, gf::launch_sweep(1, V, d_vn, d_vt, d_vj, d_vw, d_t, d_vcoef, (const double *)d_W, o.dev, o.dev, g.jmax / 2, h->stream));
            h->launches += 2;
        }
        GF_CUDA(h, end_kernel(h));
        GF_CUDA(h, finish_out(h, o));
    } else {
        void *d_z = nullptr;
        GF_CUDA(h, reserve(h, S_MZ, std::max<size_t>(total_v, 1) * sizeof(double), &d_z));
        Out<double> oq;
        GF_CUDA(h, stage_out(h, S_MQUAD, quad, (size_t)V, &oq));
        if (oq.host) h->touched.push_back(oq.buf);
        GF_CUDA(h, begin_kernel(h));
        {
            Timer timer(h);
            GF_CUDA(h, gf::launch_sweep(0, V, d_vn, d_vt, d_vj, d_vw, d_t, d_vcoef, (const double *)d_W, d_in, (double *)d_z, g.jmax / 2, h->stream));
            GF_CUDA(h, gf::launch_multi_quad(V, d_vn, d_vd, (const double *)d_d, (const double *)d_z, oq.dev, h->stream));
            h->launches += 2;
        }
        GF_CUDA(h, end_kernel(h));
        GF_CUDA(h, finish_out(h, oq));
    }
    GF_CUDA(h, finish_call(h, flags));
    return GF_OK;
}

}  // namespace

extern "C" {

int gf_sample_multi(gf_handle h, int64_t B, const int64_t *n_off, const int64_t *t_off,
                    const int64_t *j_off, const double *t, int64_t t_len, const double *diag,
                    const double *coef, const double *ddiag, int64_t k, const double *normals,
                    uint64_t seed, uint64_t seq0, double *out, double *logdet, int32_t *status,
                    uint32_t flags)
{
    if (!h) return GF_E_ARG;
    if (B > 0 && !out) return fail(h, GF_E_ARG, "null output pointer");
    return run_multi(h, 1, B, n_off, t_off, j_off, t, t_len, diag, coef, ddiag, k, normals, seed, seq0,
                     out, logdet, nullptr, status, flags);
}

int gf_loglike_multi(gf_handle h, int64_t B, const int64_t *n_off, const int64_t *t_off,
                     const int64_t *j_off, const double *t, int64_t t_len, const double *diag,
                     const double *coef, const double *ddiag, int64_t k, const double *y,
                     double *logdet, double *quad, int32_t *status, uint32_t flags)
{
    if (!h) return GF_E_ARG;
    if (B > 0 && (!y || !quad)) return fail(h, GF_E_ARG, "null data pointer");
    return run_multi(h, 0, B, n_off, t_off, j_off, t, t_len, diag, coef, ddiag, k, y, 0, 0, nullptr,
                     logdet, quad, status, flags);
}

}  // extern "C"

extern "C" {

int gf_power_spectrum_batched(gf_handle h, int64_t B, int64_t N, const double *flux, double d,
                              int include_zero, double *power, uint32_t flags)
{
    if (!h) return GF_E_ARG;
    if (B < 0 || N < 0) return fail(h, GF_E_ARG, "negative size");
    if (B == 0 || N == 0) return GF_OK;
    if (!flux || !power) return fail(h, GF_E_ARG, "null data pointer");
    if (N > 0x7fffffff || B > 0x7fffffff) return fail(h, GF_E_ARG, "too large for one cuFFT plan");
    Guard guard(h);
    if (!h->fft) h->fft = gf::new_fft_plan();
    const int64_t NC = N / 2 + 1, nout = NC - (include_zero ? 0 : 1);
    const double *d_flux;
    GF_CUDA(h, stage_in(h, S_FLUX, flux, (size_t)(B * N), &d_flux));
    void *spec = nullptr;
    GF_CUDA(h, reserve(h, S_SPEC, (size_t)(B * NC) * sizeof(double2), &spec));
    Out<double> o;
    GF_CUDA(h, stage_out(h, S_POWER, power, (size_t)(B * nout), &o));
    if (o.host) h->touched.push_back(o.buf);
    GF_CUDA(h, begin_kernel(h));
    {
        Timer timer(h);
        GF_CUDA(h, gf::launch_obs_power(h->fft, B, N, d_flux, d, include_zero, (double2 *)spec, o.dev, h->stream));
        h->launches += 1;      // our normalisation kernel (the transform is cuFFT's)
    }
    GF_CUDA(h, end_kernel(h));
    GF_CUDA(h, finish_out(h, o));
    GF_CUDA(h, finish_call(h, flags));
    return GF_OK;
}

int gf_bin_power_batched(gf_handle h, int64_t B, int64_t F, int64_t nb, const int64_t *lo,
                         const int64_t *cnt, const double *axis, const double *power, double constant,
                         double *stat, double *err, uint32_t flags)
{
    if (!h) return GF_E_ARG;
    if (B < 0 || F < 0 || nb < 0) return fail(h, GF_E_ARG, "negative size");
    if (B == 0 || nb == 0) return GF_OK;
    if (!lo || !cnt || !axis || !power || !stat || !err) return fail(h, GF_E_ARG, "null data pointer");
    for (int64_t k = 0; k < nb; ++k)
        if (lo[k] < 0 || cnt[k] < 0 || lo[k] + cnt[k] > F) return fail(h, GF_E_ARG, "bin range outside the axis");
    if (!(constant > 0.0)) return fail(h, GF_E_ARG, "constant must be positive");
    Guard guard(h);
    const int64_t *d_lo, *d_cnt;
    const double *d_axis, *d_power;
    GF_CUDA(h, stage_in(h, S_BLO, lo, (size_t)nb, &d_lo));
    GF_CUDA(h, stage_in(h, S_BCNT, cnt, (size_t)nb, &d_cnt));
    GF_CUDA(h, stage_in(h, S_BAXIS, axis, (size_t)F, &d_axis));
    GF_CUDA(h, stage_in(h, S_POWER, power, (size_t)(B * F), &d_power));
    Out<double> os, oe;
    GF_CUDA(h, stage_out(h, S_BSTAT, stat, (size_t)(B * nb), &os));
    GF_CUDA(h, stage_out(h, S_BERR, err, (size_t)(B * nb), &oe));
    if (os.host) h->touched.push_back(os.buf);
    if (oe.host) h->touched.push_back(oe.buf);
    GF_CUDA(h, begin_kernel(h));
    {
        Timer timer(h);
        GF_CUDA(h, gf::launch_bin_power(B, F, nb, d_lo, d_cnt, d_axis, d_power, constant, os.dev, oe.dev, h->stream));
        h->launches += 1;
    }
    GF_CUDA(h, end_kernel(h));
    GF_CUDA(h, finish_out(h, os));
    GF_CUDA(h, finish_out(h, oe));
    GF_CUDA(h, finish_call(h, flags));
    return GF_OK;
}

int gf_feed_stars(gf_handle h, int64_t B, const double *mass, const double *radius, const double *temperature,
                  const double *luminosity, const double *alpha, double wavelength_nm, const double *delta,
                  int64_t n_gran, const double *gran, int64_t n_modes, const double *modes, int64_t cap_terms,
                  int64_t *j_off, double *sho, double *coef, double *base, double *ddiag, uint32_t flags)
{
    if (!h) return GF_E_ARG;
    if (B < 0 || n_gran < 0 || n_modes < 0 || cap_terms < 0) return fail(h, GF_E_ARG, "negative size");
    if (n_gran + n_modes > gf::feed_max_terms()) return fail(h, GF_E_TOO_WIDE, "more solar terms than the feeder takes");
    if (!j_off) return fail(h, GF_E_ARG, "null j_off");
    j_off[0] = 0;
    if (B == 0) return GF_OK;
    if (!mass || !radius || !temperature || !luminosity || !delta || !coef || !ddiag ||
        (n_gran > 0 && !gran) || (n_modes > 0 && !modes))
        return fail(h, GF_E_ARG, "null data pointer");
    Guard guard(h);
    const int nt = (int)(n_gran + n_modes);
    gf::FeedArgs A;
    std::memset(&A, 0, sizeof(A));
    A.B = B;
    A.n_gran = (int)n_gran;
    A.n_modes = (int)n_modes;
    A.wl_nm = wavelength_nm;
    // solar normalisations of the scaling relations, in host arithmetic like the reference's
    // (gadfly/scale.py: amplitudes Huber+ 2011, granulation Kjeldsen & Bedding 2011)
    A.amp_huber_sun = std::pow(1.0, 0.886) / (std::pow(1.0, 1.89) * 5777.0 * std::pow(5777.0 / 5934.0, 0.8));
    A.gran_power_sun = 1.0 / (1.0 * std::pow(5777.0, 5.5));
    A.tau_sun = 1.0 / (1.0 * std::pow(5777.0, 3.5));
    GF_CUDA(h, stage_in(h, S_FM, mass, (size_t)B, &A.mass));
    GF_CUDA(h, stage_in(h, S_FR, radius, (size_t)B, &A.radius));
    GF_CUDA(h, stage_in(h, S_FT, temperature, (size_t)B, &A.temperature));
    GF_CUDA(h, stage_in(h, S_FL, luminosity, (size_t)B, &A.luminosity));
    GF_CUDA(h, stage_in(h, S_FALPHA, alpha, (size_t)B, &A.alpha));
    GF_CUDA(h, stage_in(h, S_DELTA, delta, (size_t)B, &A.delta));
    GF_CUDA(h, stage_in(h, S_FGRAN, gran, (size_t)n_gran * 3, &A.gran));
    GF_CUDA(h, stage_in(h, S_FMODES, modes, (size_t)n_modes * (size_t)(4 + n_gran), &A.modes));
    void *sho_all = nullptr, *keep_all = nullptr, *count = nullptr;
    GF_CUDA(h, reserve(h, S_FSHOALL, (size_t)B * nt * 3 * sizeof(double), &sho_all));
    GF_CUDA(h, reserve(h, S_FKEEP, (size_t)B * nt, &keep_all));
    GF_CUDA(h, reserve(h, S_FCOUNT, (size_t)B * sizeof(int32_t), &count));
    GF_CUDA(h, begin_kernel(h));
    GF_CUDA(h, gf::launch_feed_hyper(A, (double *)sho_all, (unsigned char *)keep_all, (int32_t *)count, h->stream));
    h->launches += 1;
    // the CSR offsets are a host array of the ABI: terms kept per star back to the host, prefix sum here
    std::vector<int32_t> cnt((size_t)B);
    GF_CUDA(h, cudaMemcpyAsync(cnt.data(), count, (size_t)B * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    GF_CUDA(h, cudaStreamSynchronize(h->stream));
    for (int64_t b = 0; b < B; ++b) {
        if (cnt[(size_t)b] < 0) return fail(h, GF_E_ARG, "a scaled term is overdamped (Q < 0.5): build that kernel per star");
        j_off[b + 1] = j_off[b] + cnt[(size_t)b];
    }
    const int64_t total = j_off[B];
    if (total > cap_terms) return fail(h, GF_E_ARG, "coefficient arrays too small (cap_terms)");
    const int64_t *d_joff;
    GF_CUDA(h, stage_in(h, S_JOFF, (const int64_t *)j_off, (size_t)B + 1, &d_joff));
    Out<double> o_sho, o_coef, o_base, o_dd;
    GF_CUDA(h, stage_out(h, S_FSHO, sho, (size_t)total * 3, &o_sho));
    GF_CUDA(h, stage_out(h, S_OUT, coef, (size_t)total * 4, &o_coef));
    GF_CUDA(h, stage_out(h, S_FBASE, base, (size_t)total * 4, &o_base));
    GF_CUDA(h, stage_out(h, S_FDDIAG, ddiag, (size_t)B, &o_dd));
    GF_CUDA(h, begin_kernel(h));
    if (total > 0 || B > 0) {
        GF_CUDA(h, gf::launch_feed_coef(A, (const double *)sho_all, (const unsigned char *)keep_all, d_joff,
                                        o_sho.dev, o_coef.dev, o_base.dev, o_dd.dev, h->stream));
        h->launches += 1;
    }
    GF_CUDA(h, end_kernel(h));
    GF_CUDA(h, finish_out(h, o_dd));
    GF_CUDA(h, finish_out(h, o_sho));
    GF_CUDA(h, finish_out(h, o_coef));
    GF_CUDA(h, finish_out(h, o_base));
    GF_CUDA(h, finish_call(h, flags));
    return GF_OK;
}

int gf_feed_sho(gf_handle h, int64_t B, const int64_t *j_off, const double *sho, const double *delta,
                double *coef, double *base, double *ddiag, uint32_t flags)
{
    if (!h) return GF_E_ARG;
    if (B < 0) return fail(h, GF_E_ARG, "negative size");
    if (B == 0) return GF_OK;
    if (!j_off || !sho || !delta || !coef || !ddiag) return fail(h, GF_E_ARG, "null data pointer");
    if (j_off[0] != 0) return fail(h, GF_E_ARG, "offsets must start at 0");
    for (int64_t b = 0; b < B; ++b)
        if (j_off[b + 1] < j_off[b]) return fail(h, GF_E_ARG, "offsets must be non-decreasing");
    const int64_t total = j_off[B];
    Guard guard(h);
    const int64_t *d_joff;
    const double *d_sho, *d_delta;
    GF_CUDA(h, stage_in(h, S_JOFF, j_off, (size_t)B + 1, &d_joff));
    GF_CUDA(h, stage_in(h, S_FSHOALL, sho, (size_t)total * 3, &d_sho));
    GF_CUDA(h, stage_in(h, S_DELTA, delta, (size_t)B, &d_delta));
    void *dterm = nullptr, *over = nullptr;
    GF_CUDA(h, reserve(h, S_FKEEP, (size_t)std::max<int64_t>(total, 1) * sizeof(double), &dterm));
    GF_CUDA(h, reserve(h, S_FCOUNT, sizeof(int32_t), &over));
    Out<double> o_coef, o_base, o_dd;
    GF_CUDA(h, stage_out(h, S_OUT, coef, (size_t)total * 4, &o_coef));
    GF_CUDA(h, stage_out(h, S_FBASE, base, (size_t)total * 4, &o_base));
    GF_CUDA(h, stage_out(h, S_FDDIAG, ddiag, (size_t)B, &o_dd));
    GF_CUDA(h, begin_kernel(h));
    GF_CUDA(h, cudaMemsetAsync(over, 0, sizeof(int32_t), h->stream));
    GF_CUDA(h, gf::launch_feed_sho(B, d_joff, d_sho, d_delta, o_coef.dev, o_base.dev, (double *)dterm, o_dd.dev,
                                   (int32_t *)over, h->stream));
    h->launches += 1;
    GF_CUDA(h, end_kernel(h));
    int32_t n_over = 0;
    GF_CUDA(h, cudaMemcpyAsync(&n_over, over, sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    GF_CUDA(h, cudaStreamSynchronize(h->stream));
    if (n_over) return fail(h, GF_E_ARG, "overdamped term (Q < 0.5): build that kernel per star");
    GF_CUDA(h, finish_out(h, o_dd));
    GF_CUDA(h, finish_out(h, o_coef));
    GF_CUDA(h, finish_out(h, o_base));
    GF_CUDA(h, finish_call(h, flags));
    return GF_OK;
}

int gf_bandpass_amplitude(gf_handle h, int64_t B, const double *temperature, int64_t n_wl, const double *wl_um,
                          const double *transmittance, double *out, uint32_t flags)
{
    if (!h) return GF_E_ARG;
    if (B < 0 || n_wl < 0) return fail(h, GF_E_ARG, "negative size");
    if (B == 0) return GF_OK;
    if (!temperature || !wl_um || !transmittance || !out || n_wl < 2) return fail(h, GF_E_ARG, "null data pointer");
    Guard guard(h);
    const double *d_T, *d_wl, *d_f;
    GF_CUDA(h, stage_in(h, S_FT, temperature, (size_t)B, &d_T));
    GF_CUDA(h, stage_in(h, S_FWL, wl_um, (size_t)n_wl, &d_wl));
    GF_CUDA(h, stage_in(h, S_FFILT, transmittance, (size_t)n_wl, &d_f));
    Out<double> o;
    GF_CUDA(h, stage_out(h, S_OUT, out, (size_t)B, &o));
    GF_CUDA(h, begin_kernel(h));
    GF_CUDA(h, gf::launch_bandpass(B, d_T, n_wl, d_wl, d_f, o.dev, h->stream));
    h->launches += 1;
    GF_CUDA(h, end_kernel(h));
    GF_CUDA(h, finish_out(h, o));
    GF_CUDA(h, finish_call(h, flags));
    return GF_OK;
}

}  // extern "C"

// C ABI of the gadfly_b200 CUDA library (see include/gadfly_b200.h for the contract).
//
// Everything here is host-side plumbing: pointer classification and staging, batch
// descriptors, the heaviest-first work order, launch bookkeeping.  Every entry point does its
// staging, launches and copies back through one `Call`.  The arithmetic is in
// scan_fast.cu / scan_small.cu / scan_blk.cu / scan_ref.cu (O(N J^2) scans), sweep.cu (O(N J)
// sweeps) and psd.cu.
#include "../../include/gadfly_b200.h"
#include "common.cuh"

#include <algorithm>
#include <cassert>
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
    std::vector<Buf *> touched;          // staging buffers the kernels of the current call use
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
struct Out {
    void *user = nullptr;
    void *dev = nullptr;
    size_t bytes = 0;
    bool host = false;
    bool pageable = false;
    Buf *buf = nullptr;
};

cudaError_t stage_out(gf_handle h, int slot, void *dst, size_t bytes, Out *o)
{
    *o = Out{dst, dst, bytes};
    if (!dst || bytes == 0) return cudaSuccess;
    const int kind = pointer_kind(dst);
    if (kind == P_DEVICE) return cudaSuccess;
    o->pageable = kind == P_PAGEABLE;
    cudaError_t e = acquire(h, slot, bytes, h->stream, &o->buf);
    if (e != cudaSuccess) return e;
    o->dev = o->buf->p;
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

// The kernel(s) of this call are launched: stamp the staging buffers the call has used so far, and
// let the copy-out stream wait for them.  The list is kept, so that a later kernel phase of the same
// call stamps again what it shares with an earlier one.
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
    return cudaStreamWaitEvent(h->s_out, h->ev_k, 0);
}

cudaError_t finish_out(gf_handle h, const Out &o)
{
    if (!o.host || !o.user || o.bytes == 0) return cudaSuccess;
    const size_t bytes = o.bytes;
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

// One entry point's work on the handle, in the order its steps are called: inputs, outputs and
// scratch staged in their slots (the order of the in() calls is the order of the H2D copies), one or
// more kernel phases, then finish(): the copies back in the order the outputs were registered, and
// the wait for them unless GF_FLAG_ASYNC.  The first CUDA error is kept; every later step does
// nothing, and finish() reports it.
//
// Staged outputs are not put on `touched`: finish() stamps each of them with its copy back, which the
// copy-out stream issues after the call's kernels.  Inputs and scratch are stamped at the end of every
// kernel phase.
class Call {
public:
    gf_handle const h;

    Call(gf_handle h_, uint32_t flags) : h(h_), flags_(flags), guard_(h_->device)
    {
        h->touched.clear();   // the buffers of earlier calls (stamped, unless such a call failed)
    }

    bool ok() const { return err_ == cudaSuccess; }
    void check(cudaError_t e, const char *what)
    {
        if (ok() && e != cudaSuccess) { err_ = e; what_ = what; }
    }

    // device pointer of an input (nullptr once the call has failed)
    template <typename T>
    const T *in(int slot, const T *src, size_t count)
    {
        const T *dev = nullptr;
        if (ok()) check(stage_in(h, slot, src, count, &dev), "stage_in");
        return ok() ? dev : nullptr;
    }

    // device pointer the kernel writes an output to; a host output is copied back by finish()
    template <typename T>
    T *out(int slot, T *dst, size_t count)
    {
        if (!ok()) return nullptr;
        Out o;
        check(stage_out(h, slot, dst, count * sizeof(T), &o), "stage_out");
        if (!ok()) return nullptr;
        if (o.host) {
            assert(n_outs_ < MAX_OUTS);
            outs_[n_outs_++] = o;
        }
        return (T *)o.dev;
    }

    // device scratch of the kernels (nullptr once the call has failed)
    void *scratch(int slot, size_t bytes)
    {
        void *p = nullptr;
        if (ok()) check(reserve(h, slot, bytes, &p), "reserve");
        return ok() ? p : nullptr;
    }

    // One kernel phase: `launch` issues the kernels on the compute stream once every input staged so
    // far has arrived (its errors go to check(), through GF_STEP) and returns how many it launched.
    template <typename F>
    void kernels(bool timed, F launch)
    {
        if (!ok()) return;
        check(begin_kernel(h), "begin_kernel");
        if (!ok()) return;
        if (timed) cudaEventRecord(h->ev0, h->stream);
        const int64_t launches = launch();
        if (timed) { cudaEventRecord(h->ev1, h->stream); h->timed = true; }
        if (!ok()) return;
        h->launches += launches;
        check(end_kernel(h), "end_kernel");
    }

    int finish()
    {
        for (int i = 0; i < n_outs_ && ok(); ++i) check(finish_out(h, outs_[i]), "finish_out");
        if (ok()) check(finish_call(h, flags_), "finish_call");
        return ok() ? GF_OK : fail(h, (int)err_, what_);
    }

private:
    static constexpr int MAX_OUTS = 5;
    uint32_t flags_;
    Guard guard_;
    cudaError_t err_ = cudaSuccess;
    const char *what_ = nullptr;
    Out outs_[MAX_OUTS];
    int n_outs_ = 0;
};

// a CUDA call an entry point makes itself: skipped once the call has failed, its error kept by the call
#define GF_STEP(c, expr) do { if ((c).ok()) (c).check((expr), #expr); } while (0)

// max over b of w_off[b] + N_b J_b: the length of a W laid out by w_off
int64_t w_extent(int64_t B, const int64_t *n_off, const int64_t *j_off, const int64_t *w_off)
{
    int64_t len = 0;
    for (int64_t b = 0; b < B; ++b)
        len = std::max(len, w_off[b] + (n_off[b + 1] - n_off[b]) * 2 * (j_off[b + 1] - j_off[b]));
    return len;
}

bool non_decreasing(int64_t B, const int64_t *off)
{
    for (int64_t b = 0; b < B; ++b)
        if (off[b + 1] < off[b]) return false;
    return true;
}

// Work-queue head of one scan launch: the next of a ring of pre-zeroed counters.  (Not a memset per
// launch: a memset is a copy-engine operation, and behind a bulk H2D copy on that engine it would hold
// the kernel back for the whole transfer -- the reason the H2D copy of the next light curves did not
// overlap the running scan in round 1.)
cudaError_t next_counter(gf_handle h, int **counter)
{
    if (h->counter_next == N_COUNTERS) {
        cudaError_t e = cudaMemsetAsync(h->counters, 0, N_COUNTERS * sizeof(int), h->stream);
        if (e != cudaSuccess) return e;
        h->counter_next = 0;
    }
    *counter = h->counters + h->counter_next++;
    return cudaSuccess;
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

// The argument checks of a scan, all before anything is staged; B == 0 passes them with nothing to do.
int check_scan(gf_handle h, int mode, int64_t B, const int64_t *n_off, const int64_t *t_off,
               const int64_t *j_off, const double *t, int64_t t_len, const double *coef, const double *ddiag,
               const int32_t *status, uint32_t flags, Geometry *g)
{
    int rc = check_geometry(h, B, n_off, t_off, j_off, t_len, g);
    if (rc != GF_OK || B == 0) return rc;
    if (!t || !coef || !ddiag || !status) return fail(h, GF_E_ARG, "null data pointer");
    if ((flags & GF_FLAG_SHARED_Y) && mode != gf::MODE_LOGLIKE)
        return fail(h, GF_E_ARG, "GF_FLAG_SHARED_Y: log-likelihood only");
    return GF_OK;
}

// The arguments of one scan launch, staged into `c`.
gf::ScanArgs stage_scan(Call &c, const Geometry &g, int64_t B, const int64_t *n_off, const int64_t *t_off,
                        const int64_t *j_off, const int64_t *w_off, const double *t, int64_t t_len,
                        const double *y, const double *diag, const double *coef, const double *ddiag,
                        uint64_t seed, uint64_t seq0, double *out_x, double *out_W, int64_t w_len,
                        double *logdet, double *quad, int32_t *status, uint32_t flags)
{
    gf::ScanArgs A;
    std::memset(&A, 0, sizeof(A));
    A.B = B;
    A.n_off = c.in(S_NOFF, n_off, (size_t)B + 1);
    A.t_off = c.in(S_TOFF, t_off, (size_t)B);
    A.j_off = c.in(S_JOFF, j_off, (size_t)B + 1);
    A.w_off = c.in(S_WOFF, w_off, (size_t)B);
    A.order = c.in(S_ORDER, (const int32_t *)g.order.data(), (size_t)B);
    GF_STEP(c, next_counter(c.h, &A.counter));
    // (the small, usually pageable arrays first: a pageable copy blocks the host until everything queued
    // before it on the copy-in stream has been copied -- behind the bulk arrays that would be their whole
    // transfer time)
    A.coef = c.in(S_COEF, coef, (size_t)g.total_j * 4);
    A.ddiag = c.in(S_DDIAG, ddiag, (size_t)B);
    A.t = c.in(S_T, t, (size_t)t_len);
    A.y_like_t = (flags & GF_FLAG_SHARED_Y) ? 1 : 0;
    const size_t y_len = A.y_like_t ? (size_t)t_len : (size_t)g.total_n;
    A.y = c.in(S_Y, y, y_len);
    A.diag = c.in(S_DIAG, diag, y_len);
    A.seed = seed;
    A.seq0 = seq0;
    // small outputs first: the caller's scalars do not wait behind the bulk copy
    A.logdet = c.out(S_LOGDET, logdet, (size_t)B);
    A.quad = c.out(S_QUAD, quad, (size_t)B);
    A.status = c.out(S_STATUS, status, (size_t)B);
    A.out_x = c.out(S_OUT, out_x, (size_t)g.total_n);
    A.out_W = c.out(S_OUTW, out_W, (size_t)w_len);
    // the kernels always write logdet: give them scratch when the caller does not want it
    if (!logdet) A.logdet = (double *)c.scratch(S_LOGDET, (size_t)B * sizeof(double));
    return A;
}

// Launch the scan kernel that serves the batch's widest state `jmax` under `flags`, record which one
// it was (gf_last_scan_path), and return how many launches it took.
int dispatch_scan(Call &c, int mode, const gf::ScanArgs &A, int jmax, uint32_t flags)
{
    gf_handle h = c.h;
    int path, n = 1;
    if ((flags & GF_FLAG_REFERENCE_ORDER) || jmax > GF_MAX_J) {
        // reference order; a state wider than the register-resident kernels take (J > 176) lives
        // in L2-resident global scratch whatever the flags
        const int grid = (int)std::min<int64_t>(A.B, (int64_t)h->sm_count);
        const size_t bytes = gf::scan_ref_scratch_bytes(jmax, grid);
        void *state = bytes ? c.scratch(S_WIDE, bytes) : nullptr;
        GF_STEP(c, gf::launch_scan_ref(mode, A, jmax, grid, (double *)state, h->stream));
        path = bytes ? GF_PATH_WIDE : GF_PATH_REF;
    } else if ((flags & GF_FLAG_BLOCKED) && gf::scan_blk_supports(mode, jmax)) {
        GF_STEP(c, gf::launch_scan_blk(mode, A, h->sm_count, h->stream));
        path = GF_PATH_BLOCKED;
    } else if (!(flags & GF_FLAG_WIDE_KERNEL) && gf::scan_small_supports(mode, jmax)) {
        // every sequence of the batch is narrow (J <= 32): one warp per sequence
        GF_STEP(c, gf::launch_scan_small(mode, A, jmax, h->sm_count, h->stream, &n));
        path = GF_PATH_SMALL;
    } else {
        GF_STEP(c, gf::launch_scan_fast(mode, A, jmax, h->sm_count, h->stream, &n));
        path = GF_PATH_FAST;
    }
    if (c.ok()) h->scan_path = path;
    return n;
}

int run_scan(gf_handle h, int mode, int64_t B, const int64_t *n_off, const int64_t *t_off,
             const int64_t *j_off, const int64_t *w_off, const double *t, int64_t t_len,
             const double *y, const double *diag, const double *coef, const double *ddiag,
             uint64_t seed, uint64_t seq0, double *out_x, double *out_W,
             double *logdet, double *quad, int32_t *status, uint32_t flags)
{
    Geometry g;
    int rc = check_scan(h, mode, B, n_off, t_off, j_off, t, t_len, coef, ddiag, status, flags, &g);
    if (rc != GF_OK || B == 0) return rc;
    const int64_t w_len = out_W ? w_extent(B, n_off, j_off, w_off) : 0;
    Call c(h, flags);
    const gf::ScanArgs A = stage_scan(c, g, B, n_off, t_off, j_off, w_off, t, t_len, y, diag, coef, ddiag,
                                      seed, seq0, out_x, out_W, w_len, logdet, quad, status, flags);
    c.kernels(true, [&] { return dispatch_scan(c, mode, A, g.jmax, flags); });
    return c.finish();
}

// ---- k right-hand sides per sequence on one factor ------------------------------------------
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
    int rc = check_scan(h, gf::MODE_FACTOR, B, n_off, t_off, j_off, t, t_len, coef, ddiag, status, flags, &g);
    if (rc != GF_OK || B == 0) return rc;
    if (B * k > 0x7fffffff) return fail(h, GF_E_ARG, "too many right-hand sides");
    Call c(h, flags);

    // 1. the inputs the factor and the sweeps share, on the device once
    const double *d_t = c.in(S_MT, t, (size_t)t_len);
    const double *d_diag = c.in(S_MDIAG, diag, (size_t)g.total_n);
    const double *d_coef = c.in(S_MCOEF, coef, (size_t)g.total_j * 4);
    const double *d_ddiag = c.in(S_MDDIAG, ddiag, (size_t)B);
    // 2. the factor: d[sum N], W[sum N J] in library scratch
    std::vector<int64_t> w_off((size_t)B);
    int64_t w_len = 0, max_n = 0;
    for (int64_t b = 0; b < B; ++b) {
        w_off[(size_t)b] = w_len;
        w_len += (n_off[b + 1] - n_off[b]) * 2 * (j_off[b + 1] - j_off[b]);
        max_n = std::max(max_n, n_off[b + 1] - n_off[b]);
    }
    double *d_d = (double *)c.scratch(S_MD, (size_t)std::max<int64_t>(g.total_n, 1) * sizeof(double));
    double *d_W = (double *)c.scratch(S_MW, (size_t)std::max<int64_t>(w_len, 1) * sizeof(double));
    const gf::ScanArgs A = stage_scan(c, g, B, n_off, t_off, j_off, w_off.data(), d_t, t_len, nullptr, d_diag,
                                      d_coef, d_ddiag, 0, 0, d_d, d_W, w_len, logdet, nullptr, status, flags);
    c.kernels(true, [&] { return dispatch_scan(c, gf::MODE_FACTOR, A, g.jmax, flags); });
    // 3. virtual sequences v = b k + r: own samples, shared time stamps, factor and kernel
    const int64_t V = B * k;
    std::vector<int64_t> vn((size_t)V + 1), vt((size_t)V), vj((size_t)V + 1), vw((size_t)V), vd((size_t)V);
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
    const int64_t *d_vn = c.in(S_VNOFF, (const int64_t *)vn.data(), (size_t)V + 1);
    const int64_t *d_vt = c.in(S_VTOFF, (const int64_t *)vt.data(), (size_t)V);
    const int64_t *d_vj = c.in(S_VJOFF, (const int64_t *)vj.data(), (size_t)V + 1);
    const int64_t *d_vw = c.in(S_VWOFF, (const int64_t *)vw.data(), (size_t)V);
    const int64_t *d_vd = c.in(S_VDOFF, (const int64_t *)vd.data(), (size_t)V);
    // the coefficient rows of sequence b, k times (the sweep kernel reads CSR rows per sequence)
    double *d_vcoef = (double *)c.scratch(S_VCOEF, (size_t)std::max<int64_t>(g.total_j * k, 1) * 4 * sizeof(double));
    for (int64_t b = 0; b < B; ++b) {
        const int64_t Jc = j_off[b + 1] - j_off[b];
        for (int64_t r = 0; r < k; ++r)
            GF_STEP(c, cudaMemcpyAsync(d_vcoef + 4 * vj[(size_t)(b * k + r)], d_coef + 4 * j_off[b],
                                       (size_t)Jc * 4 * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
    }
    const size_t total_v = (size_t)g.total_n * (size_t)k;
    const double *d_in = c.in(S_MY, in, total_v);
    if (mode == 1) {
        double *d_out = c.out(S_MOUT, out, total_v);
        c.kernels(true, [&] {
            GF_STEP(c, gf::launch_multi_prep(V, max_n, d_vn, d_vd, d_d, d_in, seed, seq0, d_out, h->stream));
            GF_STEP(c, gf::launch_sweep(1, V, d_vn, d_vt, d_vj, d_vw, d_t, d_vcoef, d_W, d_out, d_out, g.jmax / 2,
                                        h->stream));
            return 2;
        });
    } else {
        double *d_z = (double *)c.scratch(S_MZ, std::max<size_t>(total_v, 1) * sizeof(double));
        double *d_quad = c.out(S_MQUAD, quad, (size_t)V);
        c.kernels(true, [&] {
            GF_STEP(c, gf::launch_sweep(0, V, d_vn, d_vt, d_vj, d_vw, d_t, d_vcoef, d_W, d_in, d_z, g.jmax / 2,
                                        h->stream));
            GF_STEP(c, gf::launch_multi_quad(V, d_vn, d_vd, d_d, d_z, d_quad, h->stream));
            return 2;
        });
    }
    return c.finish();
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
    return run_scan(h, gf::MODE_LOGLIKE, B, n_off, t_off, j_off, nullptr, t, t_len, y, diag, coef,
                    ddiag, 0, 0, nullptr, nullptr, logdet, quad, status, flags);
}

int gf_sample_batched(gf_handle h, int64_t B, const int64_t *n_off, const int64_t *t_off,
                      const int64_t *j_off, const double *t, int64_t t_len, const double *diag,
                      const double *coef, const double *ddiag, const double *normals,
                      uint64_t seed, uint64_t seq0, double *out, double *logdet, int32_t *status,
                      uint32_t flags)
{
    if (!h) return GF_E_ARG;
    if (B > 0 && !out) return fail(h, GF_E_ARG, "null output pointer");
    return run_scan(h, gf::MODE_SAMPLE, B, n_off, t_off, j_off, nullptr, t, t_len, normals, diag,
                    coef, ddiag, seed, seq0, out, nullptr, logdet, nullptr, status, flags);
}

int gf_factor_batched(gf_handle h, int64_t B, const int64_t *n_off, const int64_t *t_off,
                      const int64_t *j_off, const int64_t *w_off, const double *t, int64_t t_len,
                      const double *diag, const double *coef, const double *ddiag, double *d,
                      double *W, double *logdet, int32_t *status, uint32_t flags)
{
    if (!h) return GF_E_ARG;
    if (B > 0 && !d) return fail(h, GF_E_ARG, "null output pointer");
    if (W && !w_off) return fail(h, GF_E_ARG, "W needs w_off");
    return run_scan(h, gf::MODE_FACTOR, B, n_off, t_off, j_off, W ? w_off : nullptr, t, t_len,
                    nullptr, diag, coef, ddiag, 0, 0, d, W, logdet, nullptr, status, flags);
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
    Call c(h, flags);
    const int64_t *d_noff = c.in(S_NOFF, n_off, (size_t)B + 1);
    const int64_t *d_toff = c.in(S_TOFF, t_off, (size_t)B);
    const int64_t *d_joff = c.in(S_JOFF, j_off, (size_t)B + 1);
    const int64_t *d_woff = c.in(S_WOFF, w_off, (size_t)B);
    const double *d_t = c.in(S_T, t, (size_t)t_len);
    const double *d_coef = c.in(S_COEF, coef, (size_t)g.total_j * 4);
    const double *d_W = c.in(S_W, W, (size_t)w_extent(B, n_off, j_off, w_off));
    // Z may alias Y: with Z on the host, a host Y goes into the buffer Z is produced in (on the compute
    // stream: the buffer was acquired for it)
    const bool z_on_device = is_device_ptr(Z);
    double *d_Z = c.out(S_OUT, Z, (size_t)g.total_n);
    const double *d_Y;
    if (z_on_device) {
        d_Y = c.in(S_Y, Y, (size_t)g.total_n);
    } else if (is_device_ptr(Y)) {
        d_Y = Y;
    } else {
        GF_STEP(c, cudaMemcpyAsync(d_Z, Y, (size_t)g.total_n * sizeof(double), cudaMemcpyHostToDevice,
                                   h->stream));
        d_Y = d_Z;
    }
    c.kernels(true, [&] {
        GF_STEP(c, gf::launch_sweep(op, B, d_noff, d_toff, d_joff, d_woff, d_t, d_coef, d_W, d_Y, d_Z,
                                    g.jmax / 2, h->stream));
        return 1;
    });
    return c.finish();
}

int gf_psd_batched(gf_handle h, int64_t B, const int64_t *j_off, const double *coef_base,
                   const double *delta, const double *omega, int64_t F, double *out,
                   uint32_t flags)
{
    if (!h) return GF_E_ARG;
    if (B < 0 || F < 0) return fail(h, GF_E_ARG, "negative size");
    if (B == 0 || F == 0) return GF_OK;
    if (!j_off || !coef_base || !omega || !out) return fail(h, GF_E_ARG, "null data pointer");
    if (!non_decreasing(B, j_off)) return fail(h, GF_E_ARG, "offsets must be non-decreasing");
    Call c(h, flags);
    const int64_t *d_joff = c.in(S_JOFF, j_off, (size_t)B + 1);
    const double *d_coef = c.in(S_COEF, coef_base, (size_t)j_off[B] * 4);
    const double *d_delta = c.in(S_DELTA, delta, (size_t)B);
    const double *d_omega = c.in(S_OMEGA, omega, (size_t)F);
    double *d_out = c.out(S_OUT, out, (size_t)B * (size_t)F);
    c.kernels(true, [&] {
        GF_STEP(c, gf::launch_psd(B, d_joff, d_coef, d_delta, d_omega, F, d_out, h->stream));
        return (B + 65534) / 65535;
    });
    return c.finish();
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
    Call c(h, flags);
    const double *d_t = c.in(S_T, t, (size_t)N);
    const double *d_ts = c.in(S_OMEGA, ts, (size_t)M);
    const double *d_coef = c.in(S_COEF, coef, (size_t)Jc * 4);
    const double *d_alpha = c.in(S_Y, alpha, (size_t)N);
    double *scratch = (double *)c.scratch(S_SCRATCH, (size_t)M * 2 * sizeof(double));
    double *d_mu = c.out(S_OUT, mu, (size_t)M);
    c.kernels(true, [&] {
        GF_STEP(c, gf::launch_cond_mean(N, d_t, M, d_ts, (int)Jc, d_coef, d_alpha, scratch, d_mu, h->stream));
        return 2;
    });
    return c.finish();
}

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


int gf_power_spectrum_batched(gf_handle h, int64_t B, int64_t N, const double *flux, double d,
                              int include_zero, double *power, uint32_t flags)
{
    if (!h) return GF_E_ARG;
    if (B < 0 || N < 0) return fail(h, GF_E_ARG, "negative size");
    if (B == 0 || N == 0) return GF_OK;
    if (!flux || !power) return fail(h, GF_E_ARG, "null data pointer");
    if (N > 0x7fffffff || B > 0x7fffffff) return fail(h, GF_E_ARG, "too large for one cuFFT plan");
    Call c(h, flags);
    if (!h->fft) h->fft = gf::new_fft_plan();
    const int64_t NC = N / 2 + 1, nout = NC - (include_zero ? 0 : 1);
    const double *d_flux = c.in(S_FLUX, flux, (size_t)(B * N));
    double2 *spec = (double2 *)c.scratch(S_SPEC, (size_t)(B * NC) * sizeof(double2));
    double *d_power = c.out(S_POWER, power, (size_t)(B * nout));
    // one launch: our normalisation kernel (the transform is cuFFT's)
    c.kernels(true, [&] {
        GF_STEP(c, gf::launch_obs_power(h->fft, B, N, d_flux, d, include_zero, spec, d_power, h->stream));
        return 1;
    });
    return c.finish();
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
    Call c(h, flags);
    const int64_t *d_lo = c.in(S_BLO, lo, (size_t)nb);
    const int64_t *d_cnt = c.in(S_BCNT, cnt, (size_t)nb);
    const double *d_axis = c.in(S_BAXIS, axis, (size_t)F);
    const double *d_power = c.in(S_POWER, power, (size_t)(B * F));
    double *d_stat = c.out(S_BSTAT, stat, (size_t)(B * nb));
    double *d_err = c.out(S_BERR, err, (size_t)(B * nb));
    c.kernels(true, [&] {
        GF_STEP(c, gf::launch_bin_power(B, F, nb, d_lo, d_cnt, d_axis, d_power, constant, d_stat, d_err, h->stream));
        return 1;
    });
    return c.finish();
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
    Call c(h, flags);
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
    A.mass = c.in(S_FM, mass, (size_t)B);
    A.radius = c.in(S_FR, radius, (size_t)B);
    A.temperature = c.in(S_FT, temperature, (size_t)B);
    A.luminosity = c.in(S_FL, luminosity, (size_t)B);
    A.alpha = c.in(S_FALPHA, alpha, (size_t)B);
    A.delta = c.in(S_DELTA, delta, (size_t)B);
    A.gran = c.in(S_FGRAN, gran, (size_t)n_gran * 3);
    A.modes = c.in(S_FMODES, modes, (size_t)n_modes * (size_t)(4 + n_gran));
    double *sho_all = (double *)c.scratch(S_FSHOALL, (size_t)B * nt * 3 * sizeof(double));
    unsigned char *keep_all = (unsigned char *)c.scratch(S_FKEEP, (size_t)B * nt);
    int32_t *count = (int32_t *)c.scratch(S_FCOUNT, (size_t)B * sizeof(int32_t));
    c.kernels(false, [&] {
        GF_STEP(c, gf::launch_feed_hyper(A, sho_all, keep_all, count, h->stream));
        return 1;
    });
    // the CSR offsets are a host array of the ABI: terms kept per star back to the host, prefix sum here
    std::vector<int32_t> cnt((size_t)B);
    GF_STEP(c, cudaMemcpyAsync(cnt.data(), count, (size_t)B * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    GF_STEP(c, cudaStreamSynchronize(h->stream));
    if (!c.ok()) return c.finish();
    for (int64_t b = 0; b < B; ++b) {
        if (cnt[(size_t)b] < 0) return fail(h, GF_E_ARG, "a scaled term is overdamped (Q < 0.5): build that kernel per star");
        j_off[b + 1] = j_off[b] + cnt[(size_t)b];
    }
    const int64_t total = j_off[B];
    if (total > cap_terms) return fail(h, GF_E_ARG, "coefficient arrays too small (cap_terms)");
    const int64_t *d_joff = c.in(S_JOFF, (const int64_t *)j_off, (size_t)B + 1);
    // small outputs first
    double *d_dd = c.out(S_FDDIAG, ddiag, (size_t)B);
    double *d_sho = c.out(S_FSHO, sho, (size_t)total * 3);
    double *d_coef = c.out(S_OUT, coef, (size_t)total * 4);
    double *d_base = c.out(S_FBASE, base, (size_t)total * 4);
    c.kernels(false, [&] {
        GF_STEP(c, gf::launch_feed_coef(A, sho_all, keep_all, d_joff, d_sho, d_coef, d_base, d_dd, h->stream));
        return 1;
    });
    return c.finish();
}

int gf_feed_sho(gf_handle h, int64_t B, const int64_t *j_off, const double *sho, const double *delta,
                double *coef, double *base, double *ddiag, uint32_t flags)
{
    if (!h) return GF_E_ARG;
    if (B < 0) return fail(h, GF_E_ARG, "negative size");
    if (B == 0) return GF_OK;
    if (!j_off || !sho || !delta || !coef || !ddiag) return fail(h, GF_E_ARG, "null data pointer");
    if (j_off[0] != 0) return fail(h, GF_E_ARG, "offsets must start at 0");
    if (!non_decreasing(B, j_off)) return fail(h, GF_E_ARG, "offsets must be non-decreasing");
    const int64_t total = j_off[B];
    Call c(h, flags);
    const int64_t *d_joff = c.in(S_JOFF, j_off, (size_t)B + 1);
    const double *d_sho = c.in(S_FSHOALL, sho, (size_t)total * 3);
    const double *d_delta = c.in(S_DELTA, delta, (size_t)B);
    double *dterm = (double *)c.scratch(S_FKEEP, (size_t)std::max<int64_t>(total, 1) * sizeof(double));
    int32_t *over = (int32_t *)c.scratch(S_FCOUNT, sizeof(int32_t));
    // small outputs first
    double *d_dd = c.out(S_FDDIAG, ddiag, (size_t)B);
    double *d_coef = c.out(S_OUT, coef, (size_t)total * 4);
    double *d_base = c.out(S_FBASE, base, (size_t)total * 4);
    c.kernels(false, [&] {
        GF_STEP(c, cudaMemsetAsync(over, 0, sizeof(int32_t), h->stream));
        GF_STEP(c, gf::launch_feed_sho(B, d_joff, d_sho, d_delta, d_coef, d_base, dterm, d_dd, over, h->stream));
        return 1;
    });
    int32_t n_over = 0;
    GF_STEP(c, cudaMemcpyAsync(&n_over, over, sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    GF_STEP(c, cudaStreamSynchronize(h->stream));
    if (c.ok() && n_over) return fail(h, GF_E_ARG, "overdamped term (Q < 0.5): build that kernel per star");
    return c.finish();
}

int gf_bandpass_amplitude(gf_handle h, int64_t B, const double *temperature, int64_t n_wl, const double *wl_um,
                          const double *transmittance, double *out, uint32_t flags)
{
    if (!h) return GF_E_ARG;
    if (B < 0 || n_wl < 0) return fail(h, GF_E_ARG, "negative size");
    if (B == 0) return GF_OK;
    if (!temperature || !wl_um || !transmittance || !out || n_wl < 2) return fail(h, GF_E_ARG, "null data pointer");
    Call c(h, flags);
    const double *d_T = c.in(S_FT, temperature, (size_t)B);
    const double *d_wl = c.in(S_FWL, wl_um, (size_t)n_wl);
    const double *d_f = c.in(S_FFILT, transmittance, (size_t)n_wl);
    double *d_out = c.out(S_OUT, out, (size_t)B);
    c.kernels(false, [&] {
        GF_STEP(c, gf::launch_bandpass(B, d_T, n_wl, d_wl, d_f, d_out, h->stream));
        return 1;
    });
    return c.finish();
}

}  // extern "C"

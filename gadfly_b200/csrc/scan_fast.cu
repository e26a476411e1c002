// Fast semiseparable scan (K1 log-likelihood, K2 sample, K3 factor) for sm_100a, FP64.
//
// One CTA per sequence (persistent CTAs pull sequences from a queue), 1 CTA per SM, three
// warpgroups with re-balanced register budgets (setmaxnreg), three roles:
//
//   matrix (WG0, WG1; 8 warps)  The J x J symmetric state lives in REGISTERS: each thread owns
//       one 8x8 tile of the upper triangle (253 tiles at J = 176).  Per time step and stored
//       element: one FMA for the rank-1 update and two FMAs for the two matrix-vector partial
//       products a symmetric tile contributes to -- 3 DFMA per element; the FP64 pipe is the
//       binding resource.  Tiles are grouped 2x2 per 4 lanes so that half of the partial sums
//       are combined by warp shuffles and the operand vectors are read as conflict-free /
//       broadcast LDS.128.  The matrix warps also reduce the quadratic form u~ S~ u~^T, so the
//       pivot needs no reduction on the vector side.
//   chain (WG2 warps 0-2)  one lane per complex term (cos + sin column): finishes the
//       matrix-vector product from the partial sums, forms the pivot d_n, the new row w~_n, the
//       forward-substitution state, the outputs, and publishes the operands of matrix phase n+2.
//   producer (WG2 warp 3)  generates the rows u~_n, v~_n on the fly from t (nothing of size N*J
//       is read): Cody-Waite sincos of the exactly rounded phase d*t_n, decay factors by a
//       product recurrence with a first-order correction for cadence jitter (exp only when the
//       cadence changes), Philox normals for sampling; hands rows over through a shared-memory
//       ring, half a ring at a time.
//
// Two algebraic rearrangements of the celerite recurrences (SURVEY.md A.6) make this fast;
// both are exact in exact arithmetic and differ from the reference order only in rounding:
//
//  (1) Lazy decay.  With q_n = exp(-c (t_n - t_ref)) and S = diag(q) S~ diag(q), the update
//      S <- P (S + d w w^T) P becomes a pure accumulation S~ += d w~ w~^T with w~ = w / q,
//      u~ = u q, v~ = v / q: the two multiplications per element per step disappear.  The
//      reference time is moved ("renormalisation": S~ <- r r^T o S~, r = exp(-c dt) <= 1)
//      every RENORM_STEPS steps or when c_max (t_n - t_ref) would exceed RENORM_LIMIT, so all
//      scaled quantities stay far inside the FP64 range; large gaps just drive r -> 0.
//  (2) One-step-stale matrix-vector product.  h_n = u~_n S~(n) is evaluated as
//      g_n + d_{n-1} alpha_n w~_{n-1} with g_n = u~_n S~(n-1) and alpha_n = u~_n . w~_{n-1}, so
//      matrix phase n needs only w~_{n-2}: the chain work of step n-1 overlaps matrix phase n
//      instead of serialising with it.  Likewise d_n = a_n - (u~_n S~(n-1) u~_n^T + d_{n-1}
//      alpha_n^2).  Synchronisation over double-buffered operands and partial sums: named
//      barriers (bar.arrive / bar.sync) matrix -> chain and chain <-> producer, mbarriers
//      chain -> matrix (see mbar_wait below for why).
#include "common.cuh"
#ifdef GF_TIMING
#include <cstdio>   // debug builds (tools/build_variant.sh x -DGF_TIMING): per-role cycle counts via printf
#endif

namespace gf {

namespace {

constexpr int FT_THREADS = 384;
constexpr int MAT_THREADS = 256;
constexpr int MAT_WARPS = 8;
constexpr int CH_THREADS = 96;
constexpr int TPW = 30;              // complex terms per chain warp (3 x 30 = 90 >= 88)
constexpr int JC_MAX = JP_MAX / 2;   // 88
constexpr int NSB_MAX = NB_MAX / 2;  // 16 x 16 super-blocks per side
// row pitch of the operand arrays A / C: 23 instead of 22 entries, so that the four 16-byte stores
// of neighbouring chain lanes (same block, elements 0, 2, 4, 6) fall into different banks
constexpr int NB_PAD = NB_MAX + 1;
constexpr int NSLOT = NSB_MAX + 1;   // partial-sum slots per column
// A slot of partial sums is JP_MAX doubles, stored as 16-byte chunks (one complex term: cos and
// sin column).  Chunk c of slot s lives at index c ^ ((s + (c >> 3)) & 1): neighbouring 2x2 groups
// of a warp then hit complementary banks and the 16-byte stores run conflict-free.
constexpr int CTL_RENORM = 1, CTL_STOP = 2;
__host__ __device__ constexpr int pchunk(int chunk, int slot) { return chunk ^ ((slot + (chunk >> 3)) & 1); }
#ifndef GF_QF_STAGES
#define GF_QF_STAGES 5               // butterfly stages of the quadratic form done in the matrix warps
                                     // (measured: 4 = same speed, 3 = 4 % slower -- the chain is co-critical)
#endif
constexpr int QF_PER_WARP = 32 >> GF_QF_STAGES;   // what is left per warp is summed by the chain
constexpr int RR = 16;               // row ring depth (two halves)
constexpr int HALF = 8;
#ifndef GF_REG_MAT
#define GF_REG_MAT 208
#endif
#ifndef GF_REG_HLP
#define GF_REG_HLP 88
#endif
constexpr int REG_MAT = GF_REG_MAT;
constexpr int REG_HLP = GF_REG_HLP;
constexpr int REG_LAUNCH = 168;      // registers per thread at launch (65536 / 384, multiple of 8)
// setmaxnreg.inc only draws on what the CTA's own warps released: the matrix warps would wait
// forever if the helpers did not give back enough
static_assert((REG_MAT - REG_LAUNCH) * MAT_THREADS <= (REG_LAUNCH - REG_HLP) * (FT_THREADS - MAT_THREADS),
              "register re-balancing does not add up");
constexpr double RENORM_LIMIT = 64.0;
constexpr int RENORM_STEPS = 64;

// named barriers (0 is __syncthreads); "operands of a matrix phase ready" [chain -> matrix] is
// the pair of mbarriers FastSmem::mb_ops
constexpr int BAR_PART = 3;    // 3, 4: partial sums of matrix phase ready       [matrix -> chain]
constexpr int BAR_CH = 5;      // chain-warp internal
constexpr int BAR_FULL = 6;    // 6, 7: ring half produced                       [producer -> chain]
constexpr int BAR_EMPTY = 8;   // 8, 9: ring half consumed                       [chain -> producer]
constexpr int N_OPS = CH_THREADS + MAT_THREADS;
constexpr int N_RING = CH_THREADS + 32;

// producer-warp scalars that are touched once per half or only on the exact path: kept in shared
// memory so that the registers of the (88-register) producer hold the per-term state instead
struct ProdScalars {
    const double *t, *y, *dg;
    unsigned long long seq, seed;
    long long N, m_ref;
    double sum_ad_a, ddiag, cmax, wmax, dt0, t_ref;
    int philox;
};

struct FastSmem {
    double2 A[2][TILE][NB_PAD];     // (u~_n[k], d w~[k]) for k = 8 b + e, indexed [e][b]
    double2 C[2][TILE][NB_PAD];     // (u~_n[k], w~[k])
    double R[2][JP_MAX];            // renormalisation factors r[k] of the phase
    double P[2][NSLOT][JP_MAX];     // partial sums of g_n, natural column order
    double QF[2][MAT_WARPS * QF_PER_WARP];   // partial sums of u~ S~ u~^T, QF_PER_WARP per matrix warp
    double2 red2[2][4];             // (alpha, gamma) per chain warp
    // row ring, written by the producer warp
    double2 RU[RR][JC_MAX];         // (u~ cos column, u~ sin column) per term
    double2 RV[RR][JC_MAX];         // (v~ cos column, v~ sin column)
    double Rr[RR][JC_MAX];          // frame change factor into this step's frame (1 if none)
    double Rq[RR][JC_MAX];          // q of this step (factor mode: W is stored unscaled)
    double Ra[RR];                  // a_n = (diag_n + ddiag) + sum a'
    double Ry[RR];                  // y_n, or the normal draw n_n
    int Rflag[RR];                  // this step renormalises
    double2 Kab[JC_MAX + 8];        // per-term (a', b')
    double2 Kcd[JC_MAX + 8];        // per-term (c, d)
    double2 Kp[JC_MAX + 8];         // per-term cached decay over the cadence dt0: (p0, 1 / p0)
    // uniform-cadence fast path of the producer: per term and step count i = 0..HALF,
    // (cos, sin)(d * (i dt)), exp(-c i dt), exp(+c i dt) for the cached cadence dt
    // per-term state of the last produced row: decay of the current frame (q, 1/q), (cos, sin)
    // and the rounded phase d t
    double2 PBq[JC_MAX + 8];
    double2 PBt[JC_MAX + 8];
    double PBx[JC_MAX + 8];
    double2 TabT[HALF + 1][JC_MAX + 8];   // (cos, sin)(d * (i dt))
    double2 TabQ[HALF + 1][JC_MAX + 8];   // exp(-c i dt), exp(+c i dt)
    // per step of the half being produced (written by lanes 0-7 of the producer warp)
    double Ht[HALF], Hde[HALF], Hrde[HALF];
    int Hcode[HALF];
    ProdScalars ps;
    unsigned long long mb_ops[2];   // mbarriers "operands of matrix phase parity p ready" [chain -> matrix]
    int ctl[2];                     // per matrix phase parity: CTL_RENORM / CTL_STOP
    int stop;                       // first matrix phase that must not run
    int next;
};

__device__ __forceinline__ void bar_sync(int id, int count)
{
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory");
}
__device__ __forceinline__ void bar_arrive(int id, int count)
{
    asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(count) : "memory");
}

// The hand-over chain -> matrix uses mbarriers instead of a named barrier: a named barrier would
// also synchronise the eight matrix warps with each other at every phase (the fastest waits for the
// slowest: measured 250 cycles per step), an mbarrier lets each matrix warp run at its own pace --
// (measured: 2226 -> 1930 cycles per step).
__device__ __forceinline__ void mbar_init(const uint32_t addr, const int count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(addr), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_inval(const uint32_t addr)
{
    asm volatile("mbarrier.inval.shared::cta.b64 [%0];" ::"r"(addr) : "memory");
}
__device__ __forceinline__ void mbar_arrive(const uint32_t addr)
{
    asm volatile("mbarrier.arrive.release.cta.shared::cta.b64 _, [%0];" ::"r"(addr) : "memory");
}
__device__ __forceinline__ bool mbar_test(const uint32_t addr, const uint32_t parity)
{
    uint32_t ok;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.test_wait.parity.acquire.cta.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n" : "=r"(ok) : "r"(addr), "r"(parity) : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(const uint32_t addr, const uint32_t parity)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "GF_MBAR_WAIT:\n"
        "mbarrier.try_wait.parity.acquire.cta.shared::cta.b64 p, [%0], %1;\n"
        "@p bra.uni GF_MBAR_DONE;\n"
        "bra.uni GF_MBAR_WAIT;\n"
        "GF_MBAR_DONE:\n"
        "}\n" ::"r"(addr), "r"(parity) : "memory");
}

__device__ __forceinline__ double shfl_xor_d(double x, int m)
{
    return __shfl_xor_sync(0xffffffffu, x, m);
}

// ------------------------------------------------------------------------------------------
// matrix warpgroups
// ------------------------------------------------------------------------------------------
struct TileMap {
    int bi, bj;        // block row / column of this thread's tile
    int kind;          // 0 off-diagonal 2x2 group lane, 1 diagonal tile, 2 off tile of a diagonal
                       // super-block, 3 idle
    int ri, cj;        // position inside the 2x2 group (kind 0)
    int slot_row, slot_col;
};

__device__ __forceinline__ TileMap make_tile_map(int mt, int nsb)
{
    TileMap m;
    m.bi = 0; m.bj = 0; m.kind = 3; m.ri = 0; m.cj = 0; m.slot_row = 0; m.slot_col = 0;
    const int n_off = 2 * nsb * (nsb - 1);
    if (mt < n_off) {
        int g = mt >> 2, l = mt & 3;
        int I = 0, rem = g;
        while (rem >= nsb - 1 - I) { rem -= nsb - 1 - I; ++I; }
        const int Jsb = I + 1 + rem;
        m.ri = l >> 1; m.cj = l & 1;
        m.bi = 2 * I + m.ri; m.bj = 2 * Jsb + m.cj;
        m.kind = 0;
        m.slot_row = Jsb;    // contribution to the columns of super-block I from (I, Jsb)
        m.slot_col = I;      // contribution to the columns of super-block Jsb from (I, Jsb)
    } else if (mt < n_off + 3 * nsb) {
        const int q = mt - n_off, I = q / 3, k = q - 3 * I;
        if (k == 0) { m.bi = m.bj = 2 * I; m.kind = 1; m.slot_col = I; }
        else if (k == 2) { m.bi = m.bj = 2 * I + 1; m.kind = 1; m.slot_col = I; }
        else { m.bi = 2 * I; m.bj = 2 * I + 1; m.kind = 2; m.slot_row = nsb; m.slot_col = nsb; }
    }
    return m;
}

// Per-thread constants of a matrix thread.  (All lanes of a warp read the operands in the same
// order: letting each lane of a 2x2 group walk its rows / columns in its own order would save the
// selects of the exchange but doubles the shared-memory wavefronts of the operand loads -- measured.)
struct MatConst {
    const double2 *a_lo, *a_hi, *c_lo, *c_hi;  // in A[0] / C[0]: operands of local rows / columns 0 and 4
    uint32_t pr0, pc0;                // shared-space addresses in P[0] of the first row / column chunk stored
    uint32_t ctl0;                    // shared-space address of ctl[0]
    int geom;                         // bi | bj << 8 | mr << 16 | mc << 20 | kind << 24 (rare paths)
    double qw;
};
__device__ __forceinline__ int geom_bi(int g) { return g & 255; }
__device__ __forceinline__ int geom_bj(int g) { return (g >> 8) & 255; }
__device__ __forceinline__ int geom_mr(int g) { return (g >> 16) & 15; }
__device__ __forceinline__ int geom_mc(int g) { return (g >> 20) & 15; }
__device__ __forceinline__ int geom_kind(int g) { return g >> 24; }

__device__ __forceinline__ MatConst make_mat_const(const FastSmem &sm, const TileMap &tm)
{
    MatConst m;
    // mr / mc: first of the four rows / columns whose sums this lane keeps after the exchange
    const int mr = (tm.kind == 0) ? 4 * tm.cj : 0;
    const int mc = (tm.kind == 0) ? 4 * tm.ri : 0;
    m.geom = tm.bi | (tm.bj << 8) | (mr << 16) | (mc << 20) | (tm.kind << 24);
    m.a_lo = &sm.A[0][0][tm.bi];
    m.a_hi = &sm.A[0][4][tm.bi];
    m.c_lo = &sm.C[0][0][tm.bj];
    m.c_hi = &sm.C[0][4][tm.bj];
    // first stored chunk: actual rows mr.. of block bi (kind 0: two chunks, else four); the k-th
    // chunk is at byte address pr0 ^ (16 k) thanks to the alignment of the groups of four chunks
    const double2 *P2 = reinterpret_cast<const double2 *>(&sm.P[0][0][0]);
    const int cr = 4 * tm.bi + mr / 2, cc = 4 * tm.bj + mc / 2;
    m.pr0 = (uint32_t)__cvta_generic_to_shared(P2 + tm.slot_row * (JP_MAX / 2) + pchunk(cr, tm.slot_row));
    m.pc0 = (uint32_t)__cvta_generic_to_shared(P2 + tm.slot_col * (JP_MAX / 2) + pchunk(cc, tm.slot_col));
    m.ctl0 = (uint32_t)__cvta_generic_to_shared(&sm.ctl[0]);
    // weight of this tile in the quadratic form: off-diagonal tiles stand for their mirror too
    m.qw = (tm.kind == 3) ? 0.0 : ((tm.bi == tm.bj) ? 1.0 : 2.0);
    return m;
}

// 16-byte shared-memory accesses at a per-thread base address plus a compile-time offset (kept as
// one register + immediate, so that no address arithmetic is hoisted into registers)
template <int OFF>
__device__ __forceinline__ double2 lds_v2(const uint32_t addr)
{
    double2 v;
    asm volatile("ld.shared.v2.f64 {%0, %1}, [%2+%3];" : "=d"(v.x), "=d"(v.y) : "r"(addr), "n"(OFF) : "memory");
    return v;
}
template <int OFF>
__device__ __forceinline__ void sts_v2(const uint32_t addr, const double x, const double y)
{
    asm volatile("st.shared.v2.f64 [%0+%1], {%2, %3};" ::"r"(addr), "n"(OFF), "d"(x), "d"(y) : "memory");
}
constexpr int P_PAR_BYTES = (int)sizeof(double) * NSLOT * JP_MAX;       // P[1] - P[0]
template <int PAR, int I>
__device__ __forceinline__ double2 mat_row_op(const MatConst &mc)
{
    return ((I < 4) ? mc.a_lo : mc.a_hi)[PAR * TILE * NB_PAD + (I & 3) * NB_PAD];
}
template <int PAR, int J>
__device__ __forceinline__ double2 mat_col_op(const MatConst &mc)
{
    return ((J < 4) ? mc.c_lo : mc.c_hi)[PAR * TILE * NB_PAD + (J & 3) * NB_PAD];
}

template <int I>
__device__ __forceinline__ void matrix_row_pair(const double2 a0, const double2 a1, double (&S)[TILE][TILE],
                                                const double (&uj)[TILE], const double (&wj)[TILE],
                                                double (&rowp)[TILE], double (&colp)[TILE])
{
    // update and column sums only: 16 independent updates, then 8 chains of depth 2
    (void)uj; (void)rowp;
    double T0[TILE], T1[TILE];
#pragma unroll
    for (int j = 0; j < TILE; ++j) T0[j] = fma(a0.y, wj[j], S[I][j]);
#pragma unroll
    for (int j = 0; j < TILE; ++j) T1[j] = fma(a1.y, wj[j], S[I + 1][j]);
#pragma unroll
    for (int j = 0; j < TILE; ++j) { S[I][j] = T0[j]; colp[j] = fma(a0.x, T0[j], colp[j]); }
#pragma unroll
    for (int j = 0; j < TILE; ++j) { S[I + 1][j] = T1[j]; colp[j] = fma(a1.x, T1[j], colp[j]); }
}

// Row sums of the updated tile, after the update: 16 independent chains of depth 4 (every row in
// two halves), so that one warp alone keeps the FP64 pipe busy (a dependent DFMA can issue 23
// cycles after its producer: at 2 cycles per DFMA that takes >= 12 independent instructions).
__device__ __forceinline__ void matrix_row_sums(const double (&S)[TILE][TILE], const double (&uj)[TILE],
                                                double (&rowp)[TILE])
{
    double ra[TILE], rb[TILE];
#pragma unroll
    for (int i = 0; i < TILE; ++i) ra[i] = S[i][0] * uj[0];
#pragma unroll
    for (int i = 0; i < TILE; ++i) rb[i] = S[i][1] * uj[1];
#pragma unroll
    for (int j = 2; j < TILE; j += 2) {
#pragma unroll
        for (int i = 0; i < TILE; ++i) ra[i] = fma(S[i][j], uj[j], ra[i]);
#pragma unroll
        for (int i = 0; i < TILE; ++i) rb[i] = fma(S[i][j + 1], uj[j + 1], rb[i]);
    }
#pragma unroll
    for (int i = 0; i < TILE; ++i) rowp[i] = ra[i] + rb[i];
}

// frame change: S~ <- r r^T o (S~ + d w~ w~^T); the rank-1 term is consumed here (rare)
template <int PAR>
__device__ __forceinline__ void matrix_renorm(FastSmem &sm, double (&S)[TILE][TILE], const int geom,
                                              double (&wj)[TILE])
{
    const int bi = geom_bi(geom), bj = geom_bj(geom);
#pragma unroll
    for (int i = 0; i < TILE; ++i) {
        const double dwi = sm.A[PAR][i][bi].y;
        const double rgi = sm.R[PAR][bi * TILE + i];
#pragma unroll
        for (int j = 0; j < TILE; ++j) {
            const double rgj = sm.R[PAR][bj * TILE + j];
            S[i][j] = (rgi * fma(dwi, wj[j], S[i][j])) * rgj;
        }
    }
#pragma unroll
    for (int e = 0; e < TILE; ++e) wj[e] = 0.0;
}

#ifdef GF_TIMING
#define g_wait tm_wait
#define g_notready tm_notready
#endif
#ifdef GF_TIMING
// clock read that cannot be scheduled before `v` is available
__device__ __forceinline__ long long clk_after(const double v)
{
    long long t;
    asm volatile("{\n.reg .f64 dd;\nmov.f64 dd, %1;\nmov.u64 %0, %%clock64;\n}\n" : "=l"(t) : "d"(v) : "memory");
    return t;
}
#endif
// One phase of a matrix thread: wait for the operands, (renormalisation,) the arithmetic, the
// exchange inside the 2x2 group, the warp reduction of the quadratic form, stores and hand-over.
template <int PAR>
__device__ __forceinline__ int matrix_phase(FastSmem &sm, double (&S)[TILE][TILE], const MatConst &mc,
                                            const int lane, const int warp, const uint32_t use,
                                            const bool last, bool &ready
#ifdef GF_TIMING
                                            , long long &tm_wait, int &tm_notready
#endif
                                            )
{
#ifdef GF_TIMING
    const long long tw0 = clock64();
#endif
    // `ready`: the test issued in the previous phase (its latency hidden there) already saw the
    // operands of this phase
    if (!ready) mbar_wait((uint32_t)__cvta_generic_to_shared(&sm.mb_ops[PAR]), use & 1u);
#ifdef GF_TIMING
    g_wait += clock64() - tw0;
    g_notready += ready ? 0 : 1;
#endif
    // control word: loaded through a per-thread address so that the test is an ordinary predicate
    // (the uniform-datapath form costs an R2UR round trip in front of the DFMA stream)
    int ctl;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(ctl) : "r"(mc.ctl0 + PAR * 4u) : "memory");
    double uj[TILE], wj[TILE];
    {
        double2 c;
        c = mat_col_op<PAR, 0>(mc); uj[0] = c.x; wj[0] = c.y;
        c = mat_col_op<PAR, 1>(mc); uj[1] = c.x; wj[1] = c.y;
        c = mat_col_op<PAR, 2>(mc); uj[2] = c.x; wj[2] = c.y;
        c = mat_col_op<PAR, 3>(mc); uj[3] = c.x; wj[3] = c.y;
        c = mat_col_op<PAR, 4>(mc); uj[4] = c.x; wj[4] = c.y;
        c = mat_col_op<PAR, 5>(mc); uj[5] = c.x; wj[5] = c.y;
        c = mat_col_op<PAR, 6>(mc); uj[6] = c.x; wj[6] = c.y;
        c = mat_col_op<PAR, 7>(mc); uj[7] = c.x; wj[7] = c.y;
    }
    if (ctl) {
        if (ctl & CTL_STOP) return ctl;
        matrix_renorm<PAR>(sm, S, mc.geom, wj);
    }

    double rowp[TILE], colp[TILE];
#pragma unroll
    for (int e = 0; e < TILE; ++e) colp[e] = 0.0;
    // two rows at a time so that the two row accumulators and the eight column accumulators are
    // independent chains
    matrix_row_pair<0>(mat_row_op<PAR, 0>(mc), mat_row_op<PAR, 1>(mc), S, uj, wj, rowp, colp);
    matrix_row_pair<2>(mat_row_op<PAR, 2>(mc), mat_row_op<PAR, 3>(mc), S, uj, wj, rowp, colp);
    matrix_row_pair<4>(mat_row_op<PAR, 4>(mc), mat_row_op<PAR, 5>(mc), S, uj, wj, rowp, colp);
    matrix_row_pair<6>(mat_row_op<PAR, 6>(mc), mat_row_op<PAR, 7>(mc), S, uj, wj, rowp, colp);
    matrix_row_sums(S, uj, rowp);

    // quadratic form u~ S~ u~^T: this tile's share, reduced over the warp
    double qf0 = colp[0] * uj[0], qf1 = colp[1] * uj[1];
#pragma unroll
    for (int j = 2; j < TILE; j += 2) { qf0 = fma(colp[j], uj[j], qf0); qf1 = fma(colp[j + 1], uj[j + 1], qf1); }
    double qf = (qf0 + qf1) * mc.qw;

    // are the operands of the next phase there already?  (normally yes: asked here, used at the top
    // of the next phase)
    ready = last ? false
                 : mbar_test((uint32_t)__cvta_generic_to_shared(&sm.mb_ops[PAR ^ 1]), (use + PAR) & 1u);
    // 2x2 group: combine the two tiles of a block row (lane ^ 1) and of a block column (lane ^ 2)
    // (each lane keeps four of the eight sums: rows 4 cj.., columns 4 ri..)
    const bool hr = geom_mr(mc.geom) != 0, hc = geom_mc(mc.geom) != 0;
    double rs[4], cs[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const double send_r = hr ? rowp[q] : rowp[4 + q];
        const double keep_r = hr ? rowp[4 + q] : rowp[q];
        rs[q] = keep_r + shfl_xor_d(send_r, 1);
        const double send_c = hc ? colp[q] : colp[4 + q];
        const double keep_c = hc ? colp[4 + q] : colp[q];
        cs[q] = keep_c + shfl_xor_d(send_c, 2);
    }
#pragma unroll
    for (int off = 16; off >= QF_PER_WARP; off >>= 1) qf += shfl_xor_d(qf, off);
    if (lane < QF_PER_WARP) sm.QF[PAR][warp * QF_PER_WARP + lane] = qf;

    const int kind = geom_kind(mc.geom);
    if (kind == 0) {
        sts_v2<PAR * P_PAR_BYTES>(mc.pr0, rs[0], rs[1]);
        sts_v2<PAR * P_PAR_BYTES>(mc.pr0 ^ 16u, rs[2], rs[3]);
        sts_v2<PAR * P_PAR_BYTES>(mc.pc0, cs[0], cs[1]);
        sts_v2<PAR * P_PAR_BYTES>(mc.pc0 ^ 16u, cs[2], cs[3]);
    } else if (kind == 1) {
        // diagonal tile: its (symmetric) contribution is stored once
#pragma unroll
        for (int q = 0; q < 4; ++q)
            sts_v2<PAR * P_PAR_BYTES>(mc.pc0 ^ (16u * q), colp[2 * q], colp[2 * q + 1]);
    } else if (kind == 2) {
        // off-diagonal tile of a diagonal super-block: both contributions, no partner lanes
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            sts_v2<PAR * P_PAR_BYTES>(mc.pr0 ^ (16u * q), rowp[2 * q], rowp[2 * q + 1]);
            sts_v2<PAR * P_PAR_BYTES>(mc.pc0 ^ (16u * q), colp[2 * q], colp[2 * q + 1]);
        }
    }
    bar_arrive(BAR_PART + PAR, N_OPS);
    return ctl;
}

__device__ __forceinline__ void matrix_loop(FastSmem &sm, const int mt, const int nsb, const int N)
{
    const MatConst mc = make_mat_const(sm, make_tile_map(mt, nsb));
    const int lane = mt & 31, warp = mt >> 5;
    double S[TILE][TILE];
#pragma unroll
    for (int i = 0; i < TILE; ++i)
#pragma unroll
        for (int j = 0; j < TILE; ++j) S[i][j] = 0.0;

    // the chain stops the matrix warps only at a phase it has not released yet
    bool ready = false;
#ifdef GF_TIMING
    long long tm_wait = 0; int tm_notready = 0;
    const long long tm_start = clock64();
#define GF_TM_ARGS , tm_wait, tm_notready
#else
#define GF_TM_ARGS
#endif
    for (int n = 0;;) {
        const uint32_t use = (uint32_t)n >> 1;   // this is the use-th phase of either parity
        int ctl = matrix_phase<0>(sm, S, mc, lane, warp, use, n + 1 >= N, ready GF_TM_ARGS);
        if (!(ctl & CTL_STOP)) {
            if (++n >= N) break;
            ctl = matrix_phase<1>(sm, S, mc, lane, warp, use, n + 1 >= N, ready GF_TM_ARGS);
        }
        if (ctl & CTL_STOP) break;
        if (++n >= N) break;
    }
#ifdef GF_TIMING
    if (blockIdx.x == 0 && lane == 0)
        printf("matrix warp %d: %.1f cyc/phase, ops wait %.1f cyc/phase, not ready at early test %.3f\n", warp,
               (double)(clock64() - tm_start) / N, (double)tm_wait / N, (double)tm_notready / N);
#endif
}

// ------------------------------------------------------------------------------------------
// producer warp: rows of U, V (scaled), a_n, y_n / normal draws -> ring
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ long long ring_halves(long long N) { return (N + 1) / HALF + 1; }

template <int MODE>
__device__ __forceinline__ void producer_loop(FastSmem &sm, const ScanArgs &A, const int lane,
                                              const int b, const long long N, const int Jc)
{
    const long long j0 = A.j_off[b];
    ProdScalars &ps = sm.ps;
    bool fast_allowed;
    {
        const long long n0 = A.n_off[b];
        const double *t = A.t + A.t_off[b];
        // sum of a' in term order (as the oracle adds it); largest decay rate and frequency
        double sum_a = 0.0, cmax = 0.0, dmax = 0.0;
        for (int j = 0; j < Jc; ++j) {
            sum_a += A.coef[4 * (j0 + j)];
            cmax = fmax(cmax, A.coef[4 * (j0 + j) + 2]);
            dmax = fmax(dmax, fabs(A.coef[4 * (j0 + j) + 3]));
        }
        // uniform-cadence fast path: rows by angle addition / decay products from the tables of
        // the cached cadence dtT.  Allowed while the rounded phases stay below 1e8 (their rounding
        // error, which the fast path reproduces to first order, is then < 1.5e-8 rad).
        fast_allowed = (N > 2 * HALF) && (dmax * fmax(fabs(t[0]), fabs(t[N - 1])) < 1.0e8);
        if (lane == 0) {
            ps.t = t;
            const long long y0 = A.y_like_t ? A.t_off[b] : n0;
            ps.y = A.y ? A.y + y0 : nullptr;
            ps.dg = A.diag ? A.diag + y0 : nullptr;
            ps.seq = A.seq0 + (uint64_t)b;
            ps.seed = A.seed;
            ps.N = N;
            ps.m_ref = 0;
            ps.sum_ad_a = sum_a;
            ps.ddiag = A.ddiag[b];
            ps.cmax = cmax;
            ps.wmax = fmax(cmax, dmax);
            ps.dt0 = 0.0;       // cadence the cached decay factors p0 belong to (exact path)
            ps.t_ref = 0.0;
            ps.philox = ((MODE == MODE_SAMPLE) && (A.y == nullptr)) ? 1 : 0;
        }
    }
    // this lane's terms: lane, lane + 32, lane + 64; their constants stay in shared memory
    constexpr int TPL = 3;
    bool act[TPL];
#pragma unroll
    for (int k = 0; k < TPL; ++k) {
        const int term = lane + 32 * k;
        act[k] = term < Jc;
        double4 cf = make_double4(0.0, 0.0, 0.0, 0.0);
        if (act[k]) cf = *reinterpret_cast<const double4 *>(A.coef + 4 * (j0 + term));
        sm.Kab[term] = make_double2(cf.x, cf.y);
        sm.Kcd[term] = make_double2(cf.z, cf.w);
        sm.Kp[term] = make_double2(1.0, 1.0);
        sm.PBq[term] = make_double2(1.0, 1.0);
        sm.PBt[term] = make_double2(1.0, 0.0);
        sm.PBx[term] = 0.0;
    }
    __syncwarp();
    double t_prev = 0.0;
    bool tab_ok = false;
    int cooldown = 0;
    double dtT = 0.0;
    int K = RENORM_STEPS;        // renormalisation period [steps] of the fast path
    int kb = 0;                  // steps since the last renormalisation at the last produced row

    // per-half input staging: lanes 0-7 t, 8-15 y (or normal), 16-23 diag
    auto load_half = [&](long long m0) -> double {
        const int role = lane >> 3;
        const long long m = m0 + (lane & 7);
        double v = 0.0;
        if (m < N) {
            if (role == 0) v = ps.t[m];
            else if (role == 1) {
                const double *y = ps.y;
                v = y ? y[m] : (ps.philox ? philox_normal(ps.seed, ps.seq, (uint64_t)m) : 0.0);
            } else if (role == 2) {
                const double *dg = ps.dg;
                v = dg ? dg[m] : 0.0;
            }
        }
        return v;
    };

    const long long nh = ring_halves(N);
    double pend = load_half(0);
    for (long long hi = 0; hi < nh; ++hi) {
        const int h = (int)(hi & 1);
        const double cur = pend;
        if (hi + 1 < nh) pend = load_half((hi + 1) * HALF);
        if (hi >= 2) bar_sync(BAR_EMPTY + h, N_RING);
        const bool aborted = sm.stop < N;    // the chain gave up: keep only the hand-shake going
        if (!aborted) {
            const long long m0 = hi * HALF;
            // ---- can this half take the fast path? ------------------------------------------
            bool fast = false;
            double e_mine = 0.0;             // lanes 0-7: deviation of t from the uniform grid
            if (fast_allowed && hi >= 1 && m0 + HALF <= N) {
                if (!tab_ok) {
                    if (cooldown > 0) {
                        --cooldown;
                    } else {
                        // (re)build the tables for the cadence seen at the start of this half
                        dtT = __shfl_sync(0xffffffffu, cur, 0) - t_prev;
                        const double cdt = ps.cmax * dtT;
                        const double kk = (cdt > 0.0) ? floor(RENORM_LIMIT / cdt) : 1.0e9;
                        K = (int)fmin(fmax(kk, 1.0), (double)RENORM_STEPS);
#pragma unroll 1
                        for (int i = 0; i <= HALF; ++i) {
                            const double tau = (double)i * dtT;
#pragma unroll
                            for (int k = 0; k < TPL; ++k) {
                                const int term = lane + 32 * k;
                                const double2 cdk = sm.Kcd[term];
                                double sn, cs;
                                sincos_cw(__dmul_rn(cdk.y, tau), &sn, &cs);
                                sm.TabT[i][term] = make_double2(cs, sn);
                                sm.TabQ[i][term] = make_double2(exp(-cdk.x * tau), exp(cdk.x * tau));
                            }
                        }
                        tab_ok = true;
                        __syncwarp();
                    }
                }
                if (tab_ok) {
                    e_mine = __dsub_rn(cur - t_prev, __dmul_rn((double)((lane & 7) + 1), dtT));
                    const bool ok = (lane >= HALF) || (fabs(e_mine) * ps.wmax < 1.0e-8);
                    fast = __all_sync(0xffffffffu, ok);
                    if (!fast) { tab_ok = false; cooldown = 4; }
                }
            }
            if (fast) {
                // ---- fast half: 8 rows x 3 terms per lane, all independent -----------------
                if (kb >= K) kb = K - 1;
                {
                    const int s = lane & 7;
                    const int ks = (kb + s + 1) % K;
                    const int rn = (ks == 0);
                    const int pst = rn ? K : ks;            // steps since the previous frame change
                    const bool inhalf = pst <= s;           // ... which happened at row s - pst of this half
                    const double eprev = __shfl_sync(0xffffffffu, e_mine, inhalf ? s - pst : 0);
                    const double ym = __shfl_sync(0xffffffffu, cur, 8 + s);
                    const double dm = __shfl_sync(0xffffffffu, cur, 16 + s);
                    if (lane < HALF) {
                        // decay of the current frame at this row: table index / relative to the base
                        // row or to the frame change inside this half; a row that changes the frame
                        // starts at q = 1 and hands the decay of the old frame over as r
                        const int ti = rn ? 0 : (inhalf ? pst : s + 1);
                        const int useb = (!rn && !inhalf) ? 1 : 0;
                        const int rti = inhalf ? pst : s + 1;
                        sm.Ht[s] = cur;
                        sm.Hde[s] = rn ? 0.0 : (inhalf ? e_mine - eprev : e_mine);
                        sm.Hrde[s] = inhalf ? e_mine - eprev : e_mine;
                        sm.Hcode[s] = ti | (useb << 4) | (rn << 5) | (rti << 8) | ((inhalf ? 0 : 1) << 12);
                        const int slot = h * HALF + s;
                        sm.Ra[slot] = (dm + ps.ddiag) + ps.sum_ad_a;
                        sm.Ry[slot] = ym;
                        sm.Rflag[slot] = rn;
                    }
                }
                __syncwarp();
                const bool resync = (hi & 7) == 7;
#pragma unroll 1
                for (int k = 0; k < TPL; ++k) {
                    const int term = lane + 32 * k;
                    const bool on = term < Jc;
                    const double2 ab = sm.Kab[term], cdk = sm.Kcd[term];
                    const double2 qb = sm.PBq[term], tb = sm.PBt[term];
                    const double xbk = sm.PBx[term];
                    double x_l = 0.0, cs_l = 1.0, sn_l = 0.0, q_l = 1.0, qi_l = 1.0;
#pragma unroll 4
                    for (int s = 0; s < HALF; ++s) {
                        const double ts = sm.Ht[s], de = sm.Hde[s];
                        const int code = sm.Hcode[s];
                        const int ti = code & 15;
                        const bool useb = (code & 16) != 0;
                        const bool rn = (code & 32) != 0;
                        const double tau = (double)(s + 1) * dtT;
                        const int slot = h * HALF + s;
                        const double2 T = sm.TabT[s + 1][term];
                        const double2 Tq = sm.TabQ[ti][term];
                        // phase: angle addition from the base row, first-order correction for the
                        // difference between the rounded phase and the table angle
                        // NOT contractible: x must be the ROUNDED product (the reference takes
                        // cos / sin of fl(d t)), and d * tau the rounded product the table was built
                        // from.  Left to nvcc these become FMAs on the exact products, the rows are
                        // then the cosines of un-rounded phases and the difference (up to 0.5 ulp of
                        // a phase of 1e3..1e4 rad per row) walks away from the reference through the
                        // base rows: 1e-8 after 2000 steps on a p-mode-only kernel (found by
                        // tools/stress.py, profiles/r1_v6_stress.txt).
                        const double x = __dmul_rn(cdk.y, ts);
                        const double eps = __dsub_rn(__dsub_rn(x, xbk), __dmul_rn(cdk.y, tau));
                        const double c1 = fma(tb.x, T.x, -(tb.y * T.y));
                        const double s1 = fma(tb.y, T.x, tb.x * T.y);
                        const double cs = fma(-eps, s1, c1);
                        const double sn = fma(eps, c1, s1);
                        // decay since the last frame change, first-order jitter correction
                        const double ce = cdk.x * de;
                        double qn = useb ? qb.x * Tq.x : Tq.x;
                        double qi = useb ? qb.y * Tq.y : Tq.y;
                        qn = fma(-ce, qn, qn);
                        qi = fma(ce, qi, qi);
                        double r = 1.0;
                        if (rn) {   // warp-uniform, rare
                            const int rti = (code >> 8) & 15;
                            const double rq = sm.TabQ[rti][term].x * (((code >> 12) & 1) ? qb.x : 1.0);
                            r = fma(-(cdk.x * sm.Hrde[s]), rq, rq);
                        }
                        if (term < JC_MAX) {
                            sm.RU[slot][term] = on ? make_double2((ab.x * cs + ab.y * sn) * qn,
                                                                  (ab.x * sn - ab.y * cs) * qn)
                                                   : make_double2(0.0, 0.0);
                            sm.RV[slot][term] = on ? make_double2(cs * qi, sn * qi) : make_double2(0.0, 0.0);
                            sm.Rr[slot][term] = on ? r : 1.0;
                            if (MODE == MODE_FACTOR) sm.Rq[slot][term] = qn;
                        }
                        x_l = x; cs_l = cs; sn_l = sn; q_l = qn; qi_l = qi;
                    }
                    if (resync) sincos_cw(x_l, &sn_l, &cs_l);
                    sm.PBq[term] = make_double2(q_l, qi_l);
                    sm.PBt[term] = make_double2(cs_l, sn_l);
                    sm.PBx[term] = x_l;
                }
                kb = (kb + HALF) % K;
                t_prev = __shfl_sync(0xffffffffu, cur, HALF - 1);
                ps.m_ref = m0 + HALF - 1 - kb;
                ps.t_ref = t_prev - (double)kb * dtT;
                __syncwarp();
            } else {
                // ---- exact half: one row at a time (first half, ragged or gappy cadences) ----
                const double cmax = ps.cmax;
                double dt0 = ps.dt0, t_ref = ps.t_ref;
                long long m_ref = ps.m_ref;
#pragma unroll 1
                for (int s = 0; s < HALF; ++s) {
                    const long long m = m0 + s;
                    const int slot = h * HALF + s;
                    const double tm = __shfl_sync(0xffffffffu, cur, s);
                    const double ym = __shfl_sync(0xffffffffu, cur, 8 + s);
                    const double dm = __shfl_sync(0xffffffffu, cur, 16 + s);
                    const bool valid = m < N;
                    const double dt = (m > 0) ? (tm - t_prev) : 0.0;
                    const bool rn = valid && m > 0 &&
                                    ((cmax * (tm - t_ref) > RENORM_LIMIT) || (m - m_ref >= RENORM_STEPS));
                    // decay over this step: cached factors, corrected to first order for a jittered
                    // cadence (|c eps| < 1e-8 for every term); exp only when the cadence changes
                    const double eps = dt - dt0;
                    const bool use_exp = valid && !(fabs(cmax * eps) < 1e-8);
#pragma unroll
                    for (int k = 0; k < TPL; ++k) {
                        double uc = 0.0, us = 0.0, vc = 0.0, vs = 0.0, r = 1.0, qk = 1.0;
                        const int term = lane + 32 * k;
                        if (valid && act[k]) {
                            const double2 ab = sm.Kab[term], cdk = sm.Kcd[term];
                            double p, pinv;
                            if (use_exp) {
                                p = exp(-cdk.x * dt);
                                pinv = exp(cdk.x * dt);
                                sm.Kp[term] = make_double2(p, pinv);
                            } else {
                                const double2 pc = sm.Kp[term];
                                const double ce = cdk.x * eps;
                                p = fma(-ce, pc.x, pc.x);
                                pinv = fma(ce, pc.y, pc.y);
                            }
                            const double2 qo = sm.PBq[term];
                            double qn = qo.x * p, qi = qo.y * pinv;
                            if (rn) { r = qn; qn = 1.0; qi = 1.0; }
                            qk = qn;
                            double sn, cs;
                            const double x = __dmul_rn(cdk.y, tm);   // the rounded phase, as the reference forms it
                            sincos_cw(x, &sn, &cs);
                            sm.PBq[term] = make_double2(qn, qi);
                            sm.PBt[term] = make_double2(cs, sn);
                            sm.PBx[term] = x;
                            uc = (ab.x * cs + ab.y * sn) * qn;
                            us = (ab.x * sn - ab.y * cs) * qn;
                            vc = cs * qi;
                            vs = sn * qi;
                        }
                        if (term < JC_MAX) {
                            sm.RU[slot][term] = make_double2(uc, us);
                            sm.RV[slot][term] = make_double2(vc, vs);
                            sm.Rr[slot][term] = r;
                            if (MODE == MODE_FACTOR) sm.Rq[slot][term] = qk;
                        }
                    }
                    if (use_exp) dt0 = dt;
                    if (rn) { t_ref = tm; m_ref = m; }
                    if (valid) { t_prev = tm; kb = (int)(m - m_ref); }
                    if (m == 0) t_ref = tm;
                    if (lane == 0) {
                        sm.Ra[slot] = (dm + ps.ddiag) + ps.sum_ad_a;
                        sm.Ry[slot] = ym;
                        sm.Rflag[slot] = rn ? 1 : 0;
                    }
                }
                __syncwarp();
                ps.dt0 = dt0; ps.t_ref = t_ref; ps.m_ref = m_ref;
                __syncwarp();
            }
        }
        bar_arrive(BAR_FULL + h, N_RING);
    }
}

// ------------------------------------------------------------------------------------------
// chain warps
// ------------------------------------------------------------------------------------------
// 1 / d for a positive normal d, branch-free: hardware seed (>= 20 bits) and one third-order step
// x (1 + e + e^2), e = 1 - d x (relative error e^3 < 2^-60; three dependent DFMA instead of the
// four of two Newton steps -- this sits on the chain's serial path)
__device__ __forceinline__ double fast_rcp(double d)
{
    double x;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(x) : "d"(d));
    const double e = fma(-d, x, 1.0);
    const double p = fma(e, e, e);
    return fma(x, p, x);
}

// Sum (a, b) over the three chain warps, in two parts so that independent work can be placed
// between them.  The first butterfly stage transposes: afterwards the low half-warp carries a and
// the high half-warp b, so four more stages finish both.
__device__ __forceinline__ double chain_reduce2_warp(int lane, double a, double b)
{
    const bool hi = (lane & 16) != 0;
    const double send = hi ? a : b, keep = hi ? b : a;
    double v = keep + shfl_xor_d(send, 16);
    v += shfl_xor_d(v, 8);
    v += shfl_xor_d(v, 4);
    v += shfl_xor_d(v, 2);
    v += shfl_xor_d(v, 1);
    return v;
}
template <int PAR>
__device__ __forceinline__ void chain_reduce2_cta(FastSmem &sm, int hw, int lane, double v, double &a, double &b)
{
    if ((lane & 15) == 0) reinterpret_cast<double *>(&sm.red2[PAR][hw])[lane >> 4] = v;
    bar_sync(BAR_CH, CH_THREADS);
    const double2 v0 = sm.red2[PAR][0], v1 = sm.red2[PAR][1], v2 = sm.red2[PAR][2];
    a = (v0.x + v1.x) + v2.x;
    b = (v0.y + v1.y) + v2.y;
}

// chain -> matrix: the operands of a matrix phase of parity par are in shared memory
__device__ __forceinline__ void ops_arrive(FastSmem &sm, const int par, const int lane)
{
    __syncwarp();
    if (lane == 0) mbar_arrive((uint32_t)__cvta_generic_to_shared(&sm.mb_ops[par]));
}

// State the chain carries from step to step.  The serial path of the recurrence is kept as short
// as possible: with t~_n = d_n w~_n = v~_n - h_n (no division) and tau_{n+1} = u~_{n+1} . t~_n,
//   alpha_{n+1} = tau_{n+1} / d_n,   h_{n+1} = g_{n+1} + alpha_{n+1} t~_n,
//   d_{n+1} = a_{n+1} - (u~ S~ u~^T + alpha_{n+1} tau_{n+1}),
// so the reciprocal of the pivot runs beside the reduction of tau instead of in front of it.  The
// forward substitution (F, gamma, z) lags one step behind and shares the reduction.
struct ChainState {
    double tc, ts;          // t~_{n-1} = d_{n-1} w~_{n-1}, in the frame of step n
    double wc, ws;          // w~_{n-1}, frame of step n
    double Fc, Fs;          // F~_{n-1}, frame of step n - 1
    double alpha, tau;      // u~_n . w~_{n-1},  u~_n . t~_{n-1}
    double rd;              // 1 / d_{n-1}
    double zp;              // y_{n-1} (log-likelihood) or sqrt(d_{n-1}) n_{n-1} (sampling)
    double logdet, prod, quad;
#ifdef GF_TIMING
    long long t_part = 0, t_crit = 0, t_seg[4] = {0, 0, 0, 0};
#endif
};

struct ChainConst {
    int ht, hw, lane, term, tix, tixA, tixB, k0, kb, ke, Jc, J, N, b;
    bool act;
    long long n0;
};

// Forward-substitution update for row m = n - 1 once gamma_m is known; returns the partial
// product of gamma_n.  u0 = u~_n, r0 = frame change factor of row n.
template <int MODE>
__device__ __forceinline__ double solver_update(const ScanArgs &A, ChainState &st, const ChainConst &c,
                                                const int m, const double gamma_m, const double2 u0,
                                                const double r0)
{
    if (MODE == MODE_FACTOR) return 0.0;
    double zp;
    if (MODE == MODE_LOGLIKE) {
        zp = st.zp - gamma_m;
        st.quad = fma(zp * zp, st.rd, st.quad);
    } else {
        zp = st.zp;
        if (c.ht == 0) A.out_x[c.n0 + m] = zp + gamma_m;
    }
    st.Fc = fma(st.wc, zp, st.Fc * r0);     // F~_n, frame of step n
    st.Fs = fma(st.ws, zp, st.Fs * r0);
    return c.act ? fma(u0.x, st.Fc, u0.y * st.Fs) : 0.0;
}

// One time step of the chain.  Returns false when the pivot is not positive.
template <int MODE, int PAR>
__device__ __forceinline__ bool chain_step(FastSmem &sm, const ScanArgs &A, ChainState &st,
                                           const ChainConst &c, const int n, double &gamma_prev)
{
    const int s0 = n & (RR - 1), s1 = (n + 1) & (RR - 1), s2 = (n + 2) & (RR - 1);
    const int tix = c.tix;
    // ---- before the matrix results are needed: ring reads, forward substitution of row n - 1 ---
    const double2 u0 = sm.RU[s0][tix];
    const double r0 = sm.Rr[s0][tix];
    const double2 vn = sm.RV[s0][tix];
    const double ra = sm.Ra[s0], yn = sm.Ry[s0];
    const double r1 = sm.Rr[s1][tix];
    const double2 u1 = sm.RU[s1][tix];
    const double2 u2 = sm.RU[s2][tix];
    const double r2 = sm.Rr[s2][tix];
    const int ctl2 = sm.Rflag[s2] ? CTL_RENORM : 0;   // read here: off the critical section below
    double gpart = 0.0;
    if (n > 0) gpart = solver_update<MODE>(A, st, c, n - 1, gamma_prev, u0, r0);

#ifdef GF_TIMING
    const long long tp0 = clock64();
#endif
    bar_sync(BAR_PART + PAR, N_OPS);
#ifdef GF_TIMING
    st.t_part += clock64() - tp0;
    const long long tc0 = clock64();
#endif
    // pivot d_n = a_n - (u~ S~(n-1) u~^T + alpha_n tau_n) and its reciprocal first: scalars of the
    // previous step and four loads, nothing of the g sum -- and no branch: a non-positive pivot
    // rides along as CTL_STOP in the hand-over and is reported after it, so that the whole section
    // up to the hand-over is one basic block and this chain overlaps the g sum and the butterfly
    double qf;
    {
        const double2 *Q2 = reinterpret_cast<const double2 *>(&sm.QF[PAR][0]);
        constexpr int NQ = MAT_WARPS * QF_PER_WARP / 2;
        double2 q[NQ];
#pragma unroll
        for (int i = 0; i < NQ; ++i) q[i] = Q2[i];
#pragma unroll
        for (int w = NQ / 2; w >= 1; w >>= 1)
#pragma unroll
            for (int i = 0; i < w; ++i) { q[i].x += q[i + w].x; q[i].y += q[i + w].y; }
        qf = q[0].x + q[0].y;
    }
    const double dn = ra - fma(st.alpha, st.tau, qf);
    const bool ok = dn > 0.0;
    const double rd = fast_rcp(dn);
    // g_n: unused slots hold zeros, so the sum always runs over all of them (two batches of six
    // slots to keep the register footprint of the loads small)
    static_assert(NSLOT == 12, "summation tree below is written for 12 slots");
    double gc, gs;
    {
        const double2 *Pp = reinterpret_cast<const double2 *>(&sm.P[PAR][0][0]);
        double2 v[6];
#pragma unroll
        for (int s = 0; s < 6; ++s) v[s] = Pp[s * (JP_MAX / 2) + ((s & 1) ? c.tixB : c.tixA)];
        const double gc0 = ((v[0].x + v[1].x) + (v[2].x + v[3].x)) + (v[4].x + v[5].x);
        const double gs0 = ((v[0].y + v[1].y) + (v[2].y + v[3].y)) + (v[4].y + v[5].y);
#pragma unroll
        for (int s = 0; s < 6; ++s) v[s] = Pp[(s + 6) * (JP_MAX / 2) + ((s & 1) ? c.tixB : c.tixA)];
        gc = gc0 + (((v[0].x + v[1].x) + (v[2].x + v[3].x)) + (v[4].x + v[5].x));
        gs = gs0 + (((v[0].y + v[1].y) + (v[2].y + v[3].y)) + (v[4].y + v[5].y));
    }
#ifdef GF_TIMING
    st.t_seg[0] += clk_after(gc + gs) - tc0;                 // PART -> g
#endif
    // t~_n = v~_n - (g_n + alpha_n t~_{n-1}), then into the frame of step n + 1
    const double tc = vn.x - fma(st.alpha, st.tc, gc), ts = vn.y - fma(st.alpha, st.ts, gs);
    const double tc1 = tc * r1, ts1 = ts * r1;
    // the serial path: tau_{n+1} = u~_{n+1} . t~_n (with gamma_n riding along)
    const double tpart = c.act ? fma(u1.x, tc1, u1.y * ts1) : 0.0;
    const double red = chain_reduce2_warp(c.lane, tpart, gpart);
#ifdef GF_TIMING
    st.t_seg[1] += clk_after(red) - tc0;                     // -> warp butterfly done
#endif

#ifdef GF_TIMING
    st.t_seg[2] += clk_after(rd) - tc0;                      // -> reciprocal of the pivot
#endif
    const double wc1 = tc1 * rd, ws1 = ts1 * rd;            // w~_n, frame of step n + 1
    // operands of matrix phase n + 2: row n + 2 and the rank-1 term of step n
    if (n + 2 < c.N) {
        if (c.act) {
            sm.A[PAR][c.ke][c.kb] = make_double2(u2.x, tc1);
            sm.A[PAR][c.ke + 1][c.kb] = make_double2(u2.y, ts1);
            sm.C[PAR][c.ke][c.kb] = make_double2(u2.x, wc1);
            sm.C[PAR][c.ke + 1][c.kb] = make_double2(u2.y, ws1);
            *reinterpret_cast<double2 *>(&sm.R[PAR][c.k0]) = make_double2(r2, r2);
        }
        if (c.ht == 0) sm.ctl[PAR] = ok ? ctl2 : CTL_STOP;
        ops_arrive(sm, PAR, c.lane);
    }
#ifdef GF_TIMING
    st.t_crit += clock64() - tc0;
#endif
    if (!ok) return false;
    // ---- off the matrix' critical path --------------------------------------------------------
    double tau, gamma;
    chain_reduce2_cta<PAR>(sm, c.hw, c.lane, red, tau, gamma);
#ifdef GF_TIMING
    st.t_seg[3] += clk_after(tau + gamma) - tc0;             // -> cross-warp sum
#endif
    if (MODE == MODE_FACTOR) {
        if (A.out_W && c.act) {
            const double qn = sm.Rq[s0][tix];
            double *Wn = A.out_W + A.w_off[c.b] + (long long)n * c.J;
            Wn[c.term] = (tc * rd) * qn;
            Wn[c.Jc + c.term] = (ts * rd) * qn;
        }
        if (c.ht == 0) A.out_x[c.n0 + n] = dn;
    }
    st.zp = (MODE == MODE_SAMPLE) ? yn * sqrt(dn) : yn;
    // log-determinant: the pivot's binary exponent goes straight into the log sum (one FMA) and only
    // its mantissa in [1, 2) into the product, which is flushed through a log every 8 steps -- a
    // product of raw pivots leaves the double range once the flux scale puts them beyond ~2^(1023/8).
    // No chain state is added: a separate exponent counter cost 2-3 % (DESIGN.md section 4).  (Pivots
    // are positive here; subnormal ones would need the exponent-field-0 case and are not handled.)
    {
        const int hi = __double2hiint(dn);
        st.logdet = fma(0.6931471805599453, (double)((hi >> 20) - 1023), st.logdet);
        st.prod *= __hiloint2double((hi & 0x800fffff) | 0x3ff00000, __double2loint(dn));
    }
    if ((n & 7) == 7) { if (c.ht == 0) st.logdet += log(st.prod); st.prod = 1.0; }
    st.tc = tc1; st.ts = ts1; st.wc = wc1; st.ws = ws1;
    st.tau = tau; st.alpha = tau * rd; st.rd = rd;
    gamma_prev = gamma;
    return true;
}

template <int MODE>
__device__ __forceinline__ void chain_loop(FastSmem &sm, const ScanArgs &A, const int ht,
                                           const int b, const int N, const int Jc)
{
    ChainConst c;
    c.ht = ht; c.hw = ht >> 5; c.lane = ht & 31;
    c.term = c.hw * TPW + c.lane;
    c.act = (c.lane < TPW) && (c.term < Jc);
    c.tix = c.act ? c.term : 0;              // inactive lanes shadow term 0 and store nothing
    c.tixA = pchunk(c.tix, 0); c.tixB = pchunk(c.tix, 1);   // chunk of this term in even / odd slots
    c.k0 = 2 * c.tix;                        // cos column; sin column is k0 + 1
    c.kb = c.k0 >> 3; c.ke = c.k0 & 7;       // both columns sit in block kb (ke is even)
    c.Jc = Jc; c.J = 2 * Jc; c.N = N; c.b = b;
    c.n0 = A.n_off[b];
    const int nh = (int)ring_halves(N);
    const int tix = c.tix;

    bar_sync(BAR_FULL + 0, N_RING);          // ring half 0: rows 0..7

    // operands of matrix phases 0 and 1: rows 0 / 1, no rank-1 term yet
    if (c.act) {
        const double2 u0 = sm.RU[0][tix], u1 = sm.RU[1][tix];
        sm.A[0][c.ke][c.kb] = make_double2(u0.x, 0.0);     sm.C[0][c.ke][c.kb] = make_double2(u0.x, 0.0);
        sm.A[0][c.ke + 1][c.kb] = make_double2(u0.y, 0.0); sm.C[0][c.ke + 1][c.kb] = make_double2(u0.y, 0.0);
        sm.A[1][c.ke][c.kb] = make_double2(u1.x, 0.0);     sm.C[1][c.ke][c.kb] = make_double2(u1.x, 0.0);
        sm.A[1][c.ke + 1][c.kb] = make_double2(u1.y, 0.0); sm.C[1][c.ke + 1][c.kb] = make_double2(u1.y, 0.0);
        sm.R[0][c.k0] = 1.0; sm.R[0][c.k0 + 1] = 1.0;
        const double r1 = sm.Rr[1][tix];
        sm.R[1][c.k0] = r1; sm.R[1][c.k0 + 1] = r1;
    }
    if (ht == 0) { sm.ctl[0] = 0; sm.ctl[1] = (N > 1 && sm.Rflag[1]) ? CTL_RENORM : 0; }
    ops_arrive(sm, 0, c.lane);
    if (N > 1) ops_arrive(sm, 1, c.lane);

    ChainState st;
    st.tc = st.ts = st.wc = st.ws = st.Fc = st.Fs = st.alpha = st.tau = 0.0;
    st.rd = 0.0; st.zp = 0.0;
    st.logdet = 0.0; st.prod = 1.0; st.quad = 0.0;
    double gamma_prev = 0.0;
    int32_t fail = 0;
    bool drain = false;

    for (int n = 0; n < N; ++n) {
        // ring hand-over: row n + 2 is first touched in this step
        if (((n + 2) & (HALF - 1)) == 0 && (n + 2) / HALF < nh)
            bar_sync(BAR_FULL + (((n + 2) / HALF) & 1), N_RING);
        if (!drain) {
            const bool ok = (n & 1) ? chain_step<MODE, 1>(sm, A, st, c, n, gamma_prev)
                                    : chain_step<MODE, 0>(sm, A, st, c, n, gamma_prev);
            if (!ok) {
                // not positive definite: stop the matrix warps at phase n + 2, absorb the
                // arrival of phase n + 1 (already released), then only keep the ring
                // hand-shake with the producer going until the natural end
                const int par = n & 1;
                fail = n + 1;
                if (ht == 0) sm.stop = n + 2;       // (the step itself handed CTL_STOP over)
                if (n + 1 < N) bar_sync(BAR_PART + (par ^ 1), N_OPS);
                drain = true;
            }
        }
        // ring hand-over: row n is dead now
        if ((n & (HALF - 1)) == HALF - 1 && n / HALF + 2 < nh)
            bar_arrive(BAR_EMPTY + ((n / HALF) & 1), N_RING);
    }
    // forward substitution of the last row
    if (!drain && MODE != MODE_FACTOR) {
        if (MODE == MODE_LOGLIKE) {
            const double z = st.zp - gamma_prev;
            st.quad = fma(z * z, st.rd, st.quad);
        } else if (ht == 0) {
            A.out_x[c.n0 + N - 1] = st.zp + gamma_prev;
        }
    }
#ifdef GF_TIMING
    if (blockIdx.x == 0 && c.lane == 0)
        printf("chain warp %d: PART wait %.1f, from PART: g %.0f, warp butterfly %.0f, 1/d %.0f, hand-over %.0f, "
               "cross-warp sum %.0f cycles/step\n", c.hw, (double)st.t_part / N, (double)st.t_seg[0] / N,
               (double)st.t_seg[1] / N, (double)st.t_seg[2] / N, (double)st.t_crit / N, (double)st.t_seg[3] / N);
#endif
    if (ht == 0) {
        // (the partial last group, or the pivots before a failure: log(1) = 0 when there are none)
        A.logdet[b] = st.logdet + log(st.prod);
        if (MODE == MODE_LOGLIKE && A.quad) A.quad[b] = st.quad;
        A.status[b] = fail;
    }
}

// Per-sequence prologue shared by all roles: claim the next sequence, clear the buffers.
// Returns false when the queue is empty.
struct SeqInfo {
    int b, Jc, nsb;
    int N;
    bool first = true;
};

__device__ __forceinline__ bool next_sequence(FastSmem &sm, const ScanArgs &A, const int tid, SeqInfo &q)
{
    __syncthreads();   // everybody is done with the previous sequence
    if (tid == 0) {
        sm.next = atomicAdd(A.counter, 1);
        // one arrival per chain warp; the phase parities restart with every sequence
        for (int p = 0; p < 2; ++p) {
            const uint32_t mb = (uint32_t)__cvta_generic_to_shared(&sm.mb_ops[p]);
            if (!q.first) mbar_inval(mb);
            mbar_init(mb, CH_THREADS / 32);
        }
    }
    q.first = false;
    // operand buffers (padding columns must read as zero) and partial sums
    {
        double *z = reinterpret_cast<double *>(&sm.A[0][0][0]);
        const int nz = (int)((sizeof(sm.A) + sizeof(sm.C) + sizeof(sm.R) + sizeof(sm.P)) / sizeof(double));
        for (int i = tid; i < nz; i += FT_THREADS) z[i] = 0.0;
    }
    __syncthreads();
    const int item = sm.next;
    if (item >= A.B) return false;
    q.b = A.order[item];
    q.N = (int)(A.n_off[q.b + 1] - A.n_off[q.b]);
    q.Jc = (int)(A.j_off[q.b + 1] - A.j_off[q.b]);
    const int nb = (2 * q.Jc + TILE - 1) / TILE;
    q.nsb = (nb + 1) / 2;
    if (tid == 0) sm.stop = q.N;
    __syncthreads();
    return true;
}

template <int MODE>
__global__ void __launch_bounds__(FT_THREADS, 1) scan_fast_kernel(ScanArgs A)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    FastSmem &sm = *reinterpret_cast<FastSmem *>(smem_raw);
    const int tid = threadIdx.x;
    // the roles never rejoin: each has its own persistent loop, so that the register budgets
    // set by setmaxnreg apply to the whole role
    if (tid < MAT_THREADS) {
        asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(REG_MAT));
        SeqInfo q;
        while (next_sequence(sm, A, tid, q)) {
            if (q.N > 0) matrix_loop(sm, tid, q.nsb, q.N);
        }
    } else {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(REG_HLP));
        const int ht = tid - MAT_THREADS;
        SeqInfo q;
        if (ht < CH_THREADS) {
            while (next_sequence(sm, A, tid, q)) {
                if (q.N > 0) {
                    chain_loop<MODE>(sm, A, ht, q.b, q.N, q.Jc);
                } else if (ht == 0) {
                    A.logdet[q.b] = 0.0;
                    if (A.quad) A.quad[q.b] = 0.0;
                    A.status[q.b] = 0;
                }
            }
        } else {
            while (next_sequence(sm, A, tid, q)) {
                if (q.N > 0) producer_loop<MODE>(sm, A, ht - CH_THREADS, q.b, q.N, q.Jc);
            }
        }
    }
}

template <int MODE>
cudaError_t launch_mode(const ScanArgs &args, int grid, cudaStream_t stream)
{
    // the opt-in to > 48 KB of dynamic shared memory is per device (a process may hold handles on
    // several devices)
    static bool configured[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64 || !configured[dev]) {
        cudaError_t e = cudaFuncSetAttribute(scan_fast_kernel<MODE>,
                                             cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             (int)sizeof(FastSmem));
        if (e != cudaSuccess) return e;
        if (dev >= 0 && dev < 64) configured[dev] = true;
    }
    scan_fast_kernel<MODE><<<grid, FT_THREADS, sizeof(FastSmem), stream>>>(args);
    return cudaGetLastError();
}

}  // namespace

#ifndef GF_SCAN_FAST_AS_HEADER   // scan_blk.cu includes this file for the producer warp and the tile map
cudaError_t launch_scan_fast(int mode, const ScanArgs &args, int jmax, int sm_count,
                             cudaStream_t stream, int *launches)
{
    (void)jmax;
    const int grid = (int)(args.B < sm_count ? args.B : sm_count);
    *launches = 1;
    switch (mode) {
    case MODE_LOGLIKE: return launch_mode<MODE_LOGLIKE>(args, grid, stream);
    case MODE_SAMPLE:  return launch_mode<MODE_SAMPLE>(args, grid, stream);
    default:           return launch_mode<MODE_FACTOR>(args, grid, stream);
    }
}

#endif  // GF_SCAN_FAST_AS_HEADER

}  // namespace gf

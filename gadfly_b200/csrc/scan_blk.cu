// Blocked semiseparable scan (K1 log-likelihood, K2 sample): KB = 4 time steps per hand-over.
//
// The k-step blocked recurrence of DESIGN.md section 5b in its bulk-synchronous form.  Same CTA as
// scan_fast.cu (this file includes it for the producer warp, the row ring, the lazy decay frames and
// the tile map): 8 matrix warps with the J x J state in registers, 3 "chain" warps, 1 producer warp.
// Per block of kk <= 4 consecutive rows of one decay frame:
//
//   M  (matrix warps)  rank-k update with the t~, w~ of the PREVIOUS block, frame change if the block
//                      starts one, then kk matrix-vector products g_i = u~_i S~ against the same state
//   C1 (all 352)       g-sums of the partial products, T0_i = v~_i - g_i
//   C2 (all 352)       ONE batch of dot products: q_i = g_i.u~_i, f_i = u~_i.F~, M_im = u~_i.T0_m (m < i)
//   C3 (chain warps)   the scalar k x k recursion, every lane redundantly:
//                        c_im = M_im - sum_{l<m} (c_ml / d_l) c_il
//                        d_i  = a_i - q_i - sum_{m<i} c_im^2 / d_m
//                        z_i  = y_i - f_i - sum_{m<i} (c_im / d_m) z_m      (sampling: x_i = nu_i + f_i + ...)
//   C4 (chain warps)   t~_i = T0_i - sum_{m<i} (c_im / d_m) t~_m,  w~_i = t~_i / d_i,  F~ += sum w~_i z_i,
//                      operands of the next block, outputs
//
// No reduction is on a serial path: it is block LDL^T on the k x k Schur complement, the arithmetic of
// the step-by-step recurrence up to summation order (tools/blocked_recurrence_check.py).
#define GF_SCAN_FAST_AS_HEADER
#include "scan_fast.cu"

#include <cstddef>

namespace gf {

namespace {

constexpr int KB = 4;                                     // rows per block
constexpr int BLK_THREADS = MAT_THREADS + CH_THREADS;     // everybody but the producer warp
// hand-overs between the matrix warps (bar.arrive / bar.sync with all 352 threads counted):
constexpr int BAR_S1 = 10;    // partial products of a block are in P            [matrix -> chain]
constexpr int BAR_S2 = 11;    // t~, w~ of the previous block are in T2 / W2       [chain -> matrix]
constexpr int BAR_S3 = 12;    // P consumed; rows / frame / descriptor of the next block ready  [chain -> matrix]
constexpr int BAR_S4 = 13;    // the update is applied, T2 / W2 may be rewritten   [matrix -> chain]

struct BlkSmem {
    double P23[2][NSLOT][JP_MAX];      // partial sums of rows 2, 3 of a block (rows 0, 1: FastSmem::P)
    double2 U2[KB][4][NB_PAD];         // rows u~_i of the block: element pairs (8 b + 2 q, + 1) at [q][b]
    double2 T2[KB][4][NB_PAD];         // t~ of the previous block
    double2 W2[KB][4][NB_PAD];         // w~ of the previous block
    double Rb[JP_MAX];                 // frame change factors applied to the state at the block start
    double2 T0[KB][JC_MAX];            // v~_i - g_i per term (g_i stale by the previous block's update)
    double2 TP[KB][JC_MAX];            // t~ of the previous block per term, in the current block's frame
    double2 F[JC_MAX];                 // forward-substitution state, frame of the current block
    double dot[32];
    int kk, flag, pad0, pad1;          // block descriptor, written by chain thread 0
};
static_assert(sizeof(FastSmem) % 16 == 0, "BlkSmem follows FastSmem in dynamic shared memory");
static_assert(sizeof(FastSmem) + sizeof(BlkSmem) <= 227 * 1024, "shared memory");

// byte offset of the partial sums of block row I relative to FastSmem::P[0]
constexpr int P_OFF_23 = (int)(sizeof(FastSmem) - offsetof(FastSmem, P)) + (int)offsetof(BlkSmem, P23);
template <int I>
__host__ __device__ constexpr int p_vec_off() { return I < 2 ? I * P_PAR_BYTES : P_OFF_23 + (I - 2) * P_PAR_BYTES; }

__device__ __forceinline__ int dot_id_q(int i) { return i; }
__device__ __forceinline__ int dot_id_f(int i) { return 4 + i; }
__device__ __forceinline__ int dot_id_m(int i, int m) { return 8 + i * (i - 1) / 2 + m; }

// ------------------------------------------------------------------------------------------
// matrix side
// ------------------------------------------------------------------------------------------
// 16-byte store without the "memory" clobber of scan_fast.cu's sts_v2: the compiler may move the operand
// loads of the next row above the stores of this one (different arrays; the hand-over barriers are
// volatile asm statements and keep their order with respect to these)
template <int OFF>
__device__ __forceinline__ void sts_v2_free(const uint32_t addr, const double x, const double y)
{
    asm volatile("st.shared.v2.f64 [%0+%1], {%2, %3};" ::"r"(addr), "n"(OFF), "d"(x), "d"(y));
}

template <int M>
__device__ __forceinline__ void blk_update(double (&S)[TILE][TILE], const double2 *tb, const double2 *wc)
{
    double t[TILE], w[TILE];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const double2 a = tb[(M * 4 + q) * NB_PAD], c = wc[(M * 4 + q) * NB_PAD];
        t[2 * q] = a.x; t[2 * q + 1] = a.y; w[2 * q] = c.x; w[2 * q + 1] = c.y;
    }
#pragma unroll
    for (int i = 0; i < TILE; ++i)
#pragma unroll
        for (int j = 0; j < TILE; ++j) S[i][j] = fma(t[i], w[j], S[i][j]);
}

template <int I>
__device__ __forceinline__ void blk_load_row(const double2 *ub, const double2 *uc, double (&ur)[TILE], double (&uj)[TILE])
{
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const double2 a = ub[(I * 4 + q) * NB_PAD], c = uc[(I * 4 + q) * NB_PAD];
        ur[2 * q] = a.x; ur[2 * q + 1] = a.y; uj[2 * q] = c.x; uj[2 * q + 1] = c.y;
    }
}

// One matrix-vector product of the block.  The operands of the NEXT row are fetched before this row's
// exchange and stores: ptxas never moves a shared-memory load above an earlier store it cannot
// disambiguate, so without this every row would start with an exposed load latency.
template <int I>
__device__ __forceinline__ void blk_matvec(const double (&S)[TILE][TILE], const MatConst &mc, const double2 *ub,
                                           const double2 *uc, double (&ur)[TILE], double (&uj)[TILE], const bool more)
{
    double rowp[TILE], colp[TILE];
#pragma unroll
    for (int j = 0; j < TILE; ++j) colp[j] = ur[0] * S[0][j];
#pragma unroll
    for (int i = 1; i < TILE; ++i)
#pragma unroll
        for (int j = 0; j < TILE; ++j) colp[j] = fma(ur[i], S[i][j], colp[j]);
#pragma unroll
    for (int i = 0; i < TILE; ++i) rowp[i] = S[i][0] * uj[0];
#pragma unroll
    for (int j = 1; j < TILE; ++j)
#pragma unroll
        for (int i = 0; i < TILE; ++i) rowp[i] = fma(S[i][j], uj[j], rowp[i]);
    if (I + 1 < KB && more) blk_load_row<(I + 1 < KB) ? I + 1 : I>(ub, uc, ur, uj);

    // 2x2 group exchange (unconditional: a warp mixes tile kinds) and stores: the layout of
    // scan_fast.cu's matrix_phase
    constexpr int OFF = p_vec_off<I>();
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
    const int kind = geom_kind(mc.geom);
    if (kind == 0) {
        sts_v2_free<OFF>(mc.pr0, rs[0], rs[1]);
        sts_v2_free<OFF>(mc.pr0 ^ 16u, rs[2], rs[3]);
        sts_v2_free<OFF>(mc.pc0, cs[0], cs[1]);
        sts_v2_free<OFF>(mc.pc0 ^ 16u, cs[2], cs[3]);
    } else if (kind == 1) {
        // diagonal tile: its (symmetric) contribution is stored once
#pragma unroll
        for (int q = 0; q < 4; ++q) sts_v2_free<OFF>(mc.pc0 ^ (16u * q), colp[2 * q], colp[2 * q + 1]);
    } else if (kind == 2) {
        // off-diagonal tile of a diagonal super-block: both contributions, no partner lanes
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            sts_v2_free<OFF>(mc.pr0 ^ (16u * q), rowp[2 * q], rowp[2 * q + 1]);
            sts_v2_free<OFF>(mc.pc0 ^ (16u * q), colp[2 * q], colp[2 * q + 1]);
        }
    }
}

// ------------------------------------------------------------------------------------------
// matrix loop: products of block B (stale by block B-1), then the rank-k update of block B-1
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void blk_matrix_loop(FastSmem &sm, BlkSmem &ex, const int mt, const int nsb)
{
    const MatConst mc = make_mat_const(sm, make_tile_map(mt, nsb));
    const int bi = geom_bi(mc.geom), bj = geom_bj(mc.geom);
    const double2 *ub = &ex.U2[0][0][bi], *uc = &ex.U2[0][0][bj];
    const double2 *tb = &ex.T2[0][0][bi], *wc = &ex.W2[0][0][bj];
    double S[TILE][TILE];
#pragma unroll
    for (int i = 0; i < TILE; ++i)
#pragma unroll
        for (int j = 0; j < TILE; ++j) S[i][j] = 0.0;
    int kprev = 0;
    for (;;) {
        bar_sync(BAR_S3, BLK_THREADS);          // rows, frame factors and descriptor of this block
        const int kk = ex.kk, flag = ex.flag;
        if (kk == 0) break;
        if (flag) {
#pragma unroll
            for (int i = 0; i < TILE; ++i) {
                const double ri = ex.Rb[bi * TILE + i];
#pragma unroll
                for (int j = 0; j < TILE; ++j) S[i][j] = (ri * S[i][j]) * ex.Rb[bj * TILE + j];
            }
        }
        {
            double ur[TILE], uj[TILE];
            blk_load_row<0>(ub, uc, ur, uj);
            blk_matvec<0>(S, mc, ub, uc, ur, uj, kk > 1);
            if (kk > 1) blk_matvec<1>(S, mc, ub, uc, ur, uj, kk > 2);
            if (kk > 2) blk_matvec<2>(S, mc, ub, uc, ur, uj, kk > 3);
            if (kk > 3) blk_matvec<3>(S, mc, ub, uc, ur, uj, false);
        }
        bar_arrive(BAR_S1, BLK_THREADS);        // partial products of this block are in P
        bar_sync(BAR_S2, BLK_THREADS);          // t~, w~ of the previous block, in this block's frame
        if (kprev > 0) blk_update<0>(S, tb, wc);
        if (kprev > 1) blk_update<1>(S, tb, wc);
        if (kprev > 2) blk_update<2>(S, tb, wc);
        if (kprev > 3) blk_update<3>(S, tb, wc);
        bar_arrive(BAR_S4, BLK_THREADS);        // T2 / W2 may be overwritten
        kprev = kk;
    }
}

// rows of the block that starts at n1: up to KB rows of one ring half, none but the first changes the frame
__device__ __forceinline__ int blk_rows(const FastSmem &sm, const int n1, const int N)
{
    int k = 1;
    while (k < KB && n1 + k < N && ((n1 + k) & (HALF - 1)) != 0 && !sm.Rflag[(n1 + k) & (RR - 1)]) ++k;
    return k;
}

// dot products of a block: 4 q_i, 4 f_i, 6 M0_im (m < i), 16 cross c'_im (previous block's t~_m)
constexpr int N_DOTS = 30;
__device__ __forceinline__ int dot_id_x(int i, int m) { return 14 + 4 * i + m; }

// ------------------------------------------------------------------------------------------
// chain loop (three warps): everything of block B while the matrix warps work on block B + 1
// ------------------------------------------------------------------------------------------
template <int MODE>
__device__ __forceinline__ void blk_chain_loop(FastSmem &sm, BlkSmem &ex, const ScanArgs &A, const int ht,
                                               const int b, const int N, const int Jc)
{
    const int term = ht;
    const bool act = term < Jc;
    const int tq = term & 3, tb = term >> 2;          // element pair / block of this term's two columns
    const int hw16 = ht >> 4, hl = ht & 15;           // half-warp and lane in it (dot products)
    const long long n0g = A.n_off[b];
    const int nh = (int)ring_halves(N);

    bar_sync(BAR_FULL + 0, N_RING);                   // ring half 0: rows 0..7
    int n0 = 0, kk = blk_rows(sm, 0, N), kp = 0;
    if (act) {
#pragma unroll
        for (int i = 0; i < KB; ++i)
            if (i < kk) ex.U2[i][tq][tb] = sm.RU[i][term];
    }
    if (ht == 0) { ex.kk = kk; ex.flag = 0; }
    bar_sync(BAR_CH, CH_THREADS);
    bar_arrive(BAR_S3, BLK_THREADS);                  // block 0 can start
    bar_arrive(BAR_S2, BLK_THREADS);                  // "the update before block 0": nothing
    double rdp[KB] = {0.0, 0.0, 0.0, 0.0};            // 1 / d of the previous block
    double logsum = 0.0, prod = 1.0, quad = 0.0;
    int esum32 = 0;                                   // pivot exponents since the last flush of prod
    long long esum = 0;                               // (N |exponent| passes 2^31 at large flux scales)
    int32_t fail = 0;
    bool dead = false;
#ifdef GF_BLK_TIMING
    long long tm[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    long long tc = clock64();
#define GF_TICK(k) { const long long now_ = clock64(); tm[k] += now_ - tc; tc = now_; }
#else
#define GF_TICK(k)
#endif

    for (;;) {
        bar_sync(BAR_S1, BLK_THREADS);                // partial products of block [n0, n0 + kk)
        GF_TICK(0)
        const int n1 = n0 + kk;
        if (dead) {
            // the block after a non-positive pivot: only the hand-shakes, and stop the matrix warps
            if (ht == 0) ex.kk = 0;
            bar_sync(BAR_CH, CH_THREADS);
            bar_arrive(BAR_S3, BLK_THREADS);
            bar_sync(BAR_S4, BLK_THREADS);
            break;
        }
        // ---- C1: g-sums, T0_i = v~_i - g_i ----------------------------------------------------
        for (int item = ht; item < KB * JC_MAX; item += CH_THREADS) {
            const int i = item / JC_MAX, tm = item - i * JC_MAX;
            if (i >= kk || tm >= Jc) continue;
            const double2 *Pp = (i < 2) ? reinterpret_cast<const double2 *>(&sm.P[i][0][0])
                                        : reinterpret_cast<const double2 *>(&ex.P23[i - 2][0][0]);
            const int tixA = pchunk(tm, 0), tixB = pchunk(tm, 1);
            double2 v[NSLOT];
#pragma unroll
            for (int s = 0; s < NSLOT; ++s) v[s] = Pp[s * (JP_MAX / 2) + ((s & 1) ? tixB : tixA)];
            const double gc = (((v[0].x + v[1].x) + (v[2].x + v[3].x)) + ((v[4].x + v[5].x) + (v[6].x + v[7].x))) +
                              ((v[8].x + v[9].x) + (v[10].x + v[11].x));
            const double gs = (((v[0].y + v[1].y) + (v[2].y + v[3].y)) + ((v[4].y + v[5].y) + (v[6].y + v[7].y))) +
                              ((v[8].y + v[9].y) + (v[10].y + v[11].y));
            const double2 vn = sm.RV[(n0 + i) & (RR - 1)][tm];
            ex.T0[i][tm] = make_double2(vn.x - gc, vn.y - gs);
        }
        GF_TICK(1)
        // ---- ring: the rows of this block are touched; the next block's rows must be there -------
        for (int n = n0; n < n1; ++n)
            if (((n + 2) & (HALF - 1)) == 0 && (n + 2) / HALF < nh)
                bar_sync(BAR_FULL + (((n + 2) / HALF) & 1), N_RING);
        // ---- next block: rows, frame change, descriptor (the matrix warps start it right away) ---
        const bool more = n1 < N;
        int kk1 = 0, flag1 = 0;
        if (more) { kk1 = blk_rows(sm, n1, N); flag1 = sm.Rflag[n1 & (RR - 1)]; }
        const double r1 = (act && more && flag1) ? sm.Rr[n1 & (RR - 1)][term] : 1.0;
        if (act) {
#pragma unroll
            for (int i = 0; i < KB; ++i)
                if (i < kk1) ex.U2[i][tq][tb] = sm.RU[(n1 + i) & (RR - 1)][term];
            ex.Rb[2 * term] = r1; ex.Rb[2 * term + 1] = r1;
        }
        if (ht == 0) { ex.kk = kk1; ex.flag = flag1; }
        bar_sync(BAR_CH, CH_THREADS);                 // T0 complete, P consumed, next rows written
        bar_arrive(BAR_S3, BLK_THREADS);
        GF_TICK(2)

        // ---- C2: one batch of dot products.  All dot products of a row share the operand u~_i; a WARP
        // walks the terms once (three per lane) with one accumulator per dot product and reduces all of
        // them in one transposing butterfly (16 shuffles for 16 values instead of 5 per value).
        //   warp 0: rows 0, 1 (13 values)   warp 1: row 2 (8)   warp 2: row 3 (9)
        {
            double v[16];
#pragma unroll
            for (int k = 0; k < 16; ++k) v[k] = 0.0;
            const int cw = ht >> 5, lane = ht & 31;
            // accumulates (q, f, M_row,0.., cross 0..3) of `row` into v[base ...]
            auto row_dots = [&](const int row, const int base, const int t) {
                const int slot = (n0 + row) & (RR - 1);
                const double2 u = sm.RU[slot][t], vv = sm.RV[slot][t], t0 = ex.T0[row][t], Ft = ex.F[t];
                v[base] = fma(u.x, vv.x - t0.x, fma(u.y, vv.y - t0.y, v[base]));
                v[base + 1] = fma(u.x, Ft.x, fma(u.y, Ft.y, v[base + 1]));
#pragma unroll
                for (int m = 0; m < 3; ++m)
                    if (m < row) { const double2 y = ex.T0[m][t]; v[base + 2 + m] = fma(u.x, y.x, fma(u.y, y.y, v[base + 2 + m])); }
#pragma unroll
                for (int m = 0; m < KB; ++m)
                    if (m < kp) { const double2 y = ex.TP[m][t]; v[base + 2 + row + m] = fma(u.x, y.x, fma(u.y, y.y, v[base + 2 + row + m])); }
            };
            for (int t = lane; t < Jc; t += 32) {
                if (cw == 0) { row_dots(0, 0, t); if (kk > 1) row_dots(1, 6, t); }
                else if (cw == 1) { if (kk > 2) row_dots(2, 0, t); }
                else { if (kk > 3) row_dots(3, 0, t); }
            }
            // transposing butterfly: after the stage with offset o a lane keeps the values whose index
            // has the same bit as its lane bit; lane (b4 b3 b2 b1 *) ends with value b4 + 2 b3 + 4 b2 + 8 b1
            double w8[8], w4[4], w2[2], w1;
            {
                const bool hi = (lane & 16) != 0;
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    const double keep = hi ? v[2 * k + 1] : v[2 * k], send = hi ? v[2 * k] : v[2 * k + 1];
                    w8[k] = keep + shfl_xor_d(send, 16);
                }
            }
            {
                const bool hi = (lane & 8) != 0;
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const double keep = hi ? w8[2 * k + 1] : w8[2 * k], send = hi ? w8[2 * k] : w8[2 * k + 1];
                    w4[k] = keep + shfl_xor_d(send, 8);
                }
            }
            {
                const bool hi = (lane & 4) != 0;
#pragma unroll
                for (int k = 0; k < 2; ++k) {
                    const double keep = hi ? w4[2 * k + 1] : w4[2 * k], send = hi ? w4[2 * k] : w4[2 * k + 1];
                    w2[k] = keep + shfl_xor_d(send, 4);
                }
            }
            {
                const bool hi = (lane & 2) != 0;
                const double keep = hi ? w2[1] : w2[0], send = hi ? w2[0] : w2[1];
                w1 = keep + shfl_xor_d(send, 2);
            }
            w1 += shfl_xor_d(w1, 1);
            if ((lane & 1) == 0) {
                const int idx = ((lane >> 4) & 1) + 2 * ((lane >> 3) & 1) + 4 * ((lane >> 2) & 1) + 8 * ((lane >> 1) & 1);
                // value index -> (row, which dot)
                int row, j;
                if (cw == 0) { row = (idx < 6) ? 0 : 1; j = (idx < 6) ? idx : idx - 6; }
                else { row = cw + 1; j = idx; }
                const int nv = 2 + row + KB;                 // q, f, M_row,0 .. M_row,row-1, cross 0..3
                if (row < kk && j < nv && (cw != 0 || idx < 13)) {
                    int id;
                    if (j == 0) id = dot_id_q(row);
                    else if (j == 1) id = dot_id_f(row);
                    else if (j < 2 + row) id = dot_id_m(row, j - 2);
                    else id = dot_id_x(row, j - 2 - row);
                    ex.dot[id] = w1;
                }
            }
        }
        bar_sync(BAR_CH, CH_THREADS);
        GF_TICK(3)

        // ---- C3: scalar recursion over the window (previous block + this one), every lane --------
        double cp[KB][KB], ep[KB][KB], e[KB][KB], cc[KB][KB], rd[KB], dd[KB], zz[KB], xx[KB];
        int bad = -1;
#pragma unroll
        for (int i = 0; i < KB; ++i) {
            rd[i] = 0.0; dd[i] = 1.0; zz[i] = 0.0; xx[i] = 0.0;
#pragma unroll
            for (int m = 0; m < KB; ++m) { e[i][m] = 0.0; cc[i][m] = 0.0; cp[i][m] = 0.0; ep[i][m] = 0.0; }
            if (i < kk) {
                const int slot = (n0 + i) & (RR - 1);
#pragma unroll
                for (int m = 0; m < KB; ++m)
                    if (m < kp) { cp[i][m] = ex.dot[dot_id_x(i, m)]; ep[i][m] = cp[i][m] * rdp[m]; }
#pragma unroll
                for (int m = 0; m < i; ++m) {
                    double c = ex.dot[dot_id_m(i, m)];
#pragma unroll
                    for (int l = 0; l < KB; ++l) c = fma(-ep[m][l], cp[i][l], c);
#pragma unroll
                    for (int l = 0; l < m; ++l) c = fma(-e[m][l], cc[i][l], c);
                    cc[i][m] = c;
                }
                double acc = ex.dot[dot_id_q(i)];
#pragma unroll
                for (int m = 0; m < KB; ++m) acc = fma(ep[i][m], cp[i][m], acc);
#pragma unroll
                for (int m = 0; m < i; ++m) {
                    e[i][m] = cc[i][m] * rd[m];
                    acc = fma(e[i][m], cc[i][m], acc);
                }
                dd[i] = sm.Ra[slot] - acc;
                if (!(dd[i] > 0.0) && bad < 0) bad = i;
                rd[i] = fast_rcp(dd[i]);
                double corr = ex.dot[dot_id_f(i)];
#pragma unroll
                for (int m = 0; m < i; ++m) corr = fma(e[i][m], zz[m], corr);
                if (MODE == MODE_LOGLIKE) {
                    zz[i] = sm.Ry[slot] - corr;
                } else {
                    zz[i] = sm.Ry[slot] * sqrt(dd[i]);
                    xx[i] = zz[i] + corr;
                }
            }
        }
        const int good = (bad < 0) ? kk : bad;        // rows of this block with a positive pivot
#ifdef GF_BLK_TIMING
        { double chk = rd[0] + rd[3] + zz[3]; asm volatile("" :: "d"(chk)); }
#endif
        GF_TICK(4)

        // ---- C4: vectors ---------------------------------------------------------------------------
        double2 tt[KB], ww[KB];
#pragma unroll
        for (int i = 0; i < KB; ++i) { tt[i] = make_double2(0.0, 0.0); ww[i] = make_double2(0.0, 0.0); }
        if (act) {
            double2 tp[KB];
#pragma unroll
            for (int m = 0; m < KB; ++m) tp[m] = (m < kp) ? ex.TP[m][term] : make_double2(0.0, 0.0);
            double2 F = ex.F[term];
#pragma unroll
            for (int i = 0; i < KB; ++i) {
                if (i < kk) {
                    double2 T = ex.T0[i][term];
#pragma unroll
                    for (int m = 0; m < KB; ++m) { T.x = fma(-ep[i][m], tp[m].x, T.x); T.y = fma(-ep[i][m], tp[m].y, T.y); }
#pragma unroll
                    for (int m = 0; m < i; ++m) { T.x = fma(-e[i][m], tt[m].x, T.x); T.y = fma(-e[i][m], tt[m].y, T.y); }
                    tt[i] = T;
                    ww[i] = make_double2(T.x * rd[i], T.y * rd[i]);
                    F.x = fma(ww[i].x, zz[i], F.x);
                    F.y = fma(ww[i].y, zz[i], F.y);
                }
            }
            ex.F[term] = make_double2(F.x * r1, F.y * r1);
        }
        if (ht == 0) {
#pragma unroll
            for (int i = 0; i < KB; ++i)
                if (i < good) {
                    logdet_push(dd[i], prod, esum32);
                    if (MODE == MODE_LOGLIKE) quad = fma(zz[i] * zz[i], rd[i], quad);
                    else A.out_x[n0g + n0 + i] = xx[i];
                }
            if ((n1 & 31) < KB || !more) { logsum += log(prod); prod = 1.0; esum += esum32; esum32 = 0; }
            if (bad >= 0) sm.stop = n0 + bad;         // the producer keeps only the hand-shake going
        }
        if (bad >= 0) { fail = n0 + bad + 1; dead = true; }

        GF_TICK(5)
        bar_sync(BAR_S4, BLK_THREADS);                // the update of the previous block is applied
        GF_TICK(6)
        if (act) {
#pragma unroll
            for (int i = 0; i < KB; ++i) {
                const double2 t1 = make_double2(tt[i].x * r1, tt[i].y * r1);
                ex.T2[i][tq][tb] = t1;
                ex.W2[i][tq][tb] = make_double2(ww[i].x * r1, ww[i].y * r1);
                ex.TP[i][term] = t1;
            }
        }
#pragma unroll
        for (int i = 0; i < KB; ++i) rdp[i] = rd[i];
        if (kk1 > 0) {
            bar_sync(BAR_CH, CH_THREADS);             // all of T2 / W2 written
            bar_arrive(BAR_S2, BLK_THREADS);
        }
        // ring: the rows of this block are dead
        for (int n = n0; n < n1; ++n)
            if ((n & (HALF - 1)) == HALF - 1 && n / HALF + 2 < nh)
                bar_arrive(BAR_EMPTY + ((n / HALF) & 1), N_RING);
        kp = kk; n0 = n1; kk = kk1;
        GF_TICK(7)
        if (kk == 0) break;
    }
#ifdef GF_BLK_TIMING
    if (blockIdx.x == 0 && (ht & 31) == 0)
        printf("chain warp %d, cycles per row: wait S1 %.0f | C1 %.0f | ring + next block + S3 %.0f | C2 %.0f | C3 %.0f | C4 %.0f | wait S4 %.0f | stores + S2 + ring %.0f\n",
               ht >> 5, (double)tm[0] / N, (double)tm[1] / N, (double)tm[2] / N, (double)tm[3] / N, (double)tm[4] / N,
               (double)tm[5] / N, (double)tm[6] / N, (double)tm[7] / N);
#endif
    // after a non-positive pivot: keep the ring hand-shake with the producer going until the natural end
    for (int n = n0; n < N; ++n) {
        if (((n + 2) & (HALF - 1)) == 0 && (n + 2) / HALF < nh)
            bar_sync(BAR_FULL + (((n + 2) / HALF) & 1), N_RING);
        if ((n & (HALF - 1)) == HALF - 1 && n / HALF + 2 < nh)
            bar_arrive(BAR_EMPTY + ((n / HALF) & 1), N_RING);
    }
    if (ht == 0) {
        if (prod != 1.0) logsum += log(prod);
        A.logdet[b] = logdet_total(logsum, 1.0, esum + esum32);
        if (MODE == MODE_LOGLIKE && A.quad) A.quad[b] = quad;
        A.status[b] = fail;
    }
}

template <int MODE>
__global__ void __launch_bounds__(FT_THREADS, 1) scan_blk_kernel(ScanArgs A)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    FastSmem &sm = *reinterpret_cast<FastSmem *>(smem_raw);
    BlkSmem &ex = *reinterpret_cast<BlkSmem *>(smem_raw + sizeof(FastSmem));
    const int tid = threadIdx.x;
    // per-sequence reset of the blocked buffers (padding columns must read as zero, Rb as one)
    auto reset = [&](const int xx) {
        double *z = reinterpret_cast<double *>(&ex);
        const int nz = (int)(offsetof(BlkSmem, dot) / sizeof(double));
        for (int i = xx; i < nz; i += BLK_THREADS) z[i] = 0.0;
        for (int i = xx; i < JP_MAX; i += BLK_THREADS) ex.Rb[i] = 1.0;
    };
    if (tid < MAT_THREADS) {
        asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(REG_MAT));
        SeqInfo q;
        while (next_sequence(sm, A, tid, q)) {
            if (q.N > 0) {
                reset(tid);
                bar_sync(BAR_S1, BLK_THREADS);
                blk_matrix_loop(sm, ex, tid, q.nsb);
            }
        }
    } else {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(REG_HLP));
        const int ht = tid - MAT_THREADS;
        SeqInfo q;
        if (ht < CH_THREADS) {
            while (next_sequence(sm, A, tid, q)) {
                if (q.N > 0) {
                    reset(tid);
                    bar_sync(BAR_S1, BLK_THREADS);
                    blk_chain_loop<MODE>(sm, ex, A, ht, q.b, q.N, q.Jc);
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
cudaError_t launch_blk_mode(const ScanArgs &args, int grid, cudaStream_t stream)
{
    static bool configured[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    const int bytes = (int)(sizeof(FastSmem) + sizeof(BlkSmem));
    if (dev < 0 || dev >= 64 || !configured[dev]) {
        cudaError_t e = cudaFuncSetAttribute(scan_blk_kernel<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
        if (e != cudaSuccess) return e;
        if (dev >= 0 && dev < 64) configured[dev] = true;
    }
    scan_blk_kernel<MODE><<<grid, FT_THREADS, bytes, stream>>>(args);
    return cudaGetLastError();
}

}  // namespace

bool scan_blk_supports(int mode, int jmax) { return mode != MODE_FACTOR && jmax <= JP_MAX; }

cudaError_t launch_scan_blk(int mode, const ScanArgs &args, int sm_count, cudaStream_t stream)
{
    const int grid = (int)(args.B < sm_count ? args.B : sm_count);
    return mode == MODE_LOGLIKE ? launch_blk_mode<MODE_LOGLIKE>(args, grid, stream)
                                : launch_blk_mode<MODE_SAMPLE>(args, grid, stream);
}

}  // namespace gf

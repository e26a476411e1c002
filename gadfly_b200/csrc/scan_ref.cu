// Reference-order semiseparable scan: the validation kernel (GF_FLAG_REFERENCE_ORDER) and the
// only kernel for states wider than the register-resident scans take (GF_MAX_J = 176 < J <=
// GF_MAX_J_WIDE = 352: the reference's ``kernel + more terms``, gadfly/core.py:405-427, accepts
// any number of extra SHO terms).
//
// One CTA per sequence, plain __syncthreads() phases, arithmetic in the order of the celerite2
// recurrences (SURVEY.md A.6):
//     S <- diag(p) (S + d_{n-1} w_{n-1}^T w_{n-1}) diag(p);  tmp = u_n S;
//     d_n = a_n - tmp.u_n;  w_n = (v_n - tmp) / d_n
// The U/V rows are generated on the fly from t and (a', b', c, d); nothing of size N*J is read.
// The upper triangle of the J x J state S is kept as 8x8 tiles in one of two stores:
//   RegState  J <= 176: one register tile per thread (253 tiles at most, 256 threads);
//   L2State   J <= 352: up to 990 tiles = 507 KB per sequence, which fits neither the register
//             file nor shared memory, in a global scratch buffer that stays L2-resident (126 MB
//             L2; 148 CTAs x 507 KB = 75 MB).  Every thread walks its tiles; correct rather than
//             fast: ~1 MB of L2 traffic per time step.
// Both stores run the same per-tile expressions in the same order, so a sequence gets the same
// bits from either.  This kernel is the simple cross-check for the warp-specialised fast scan
// (scan_fast.cu); it shares the entry points and the batching/work-queue conventions.
#include "common.cuh"

namespace gf {

namespace {

template <int JMAX, int THREADS>
struct RefSmem {
    double u[JMAX], v[JMAX], p[JMAX], w[JMAX], dw[JMAX];
    double part[JMAX / TILE][JMAX];
    double red[THREADS / 32][2];
    int next;
};

__device__ __forceinline__ double warp_sum(double x)
{
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) x += __shfl_xor_sync(0xffffffffu, x, off);
    return x;
}

// Sum (a, b) over the CTA; every thread returns the identical totals.
template <int THREADS>
__device__ __forceinline__ void block_sum2(double &a, double &b, double (*red)[2], int tid)
{
    a = warp_sum(a);
    b = warp_sum(b);
    if ((tid & 31) == 0) { red[tid >> 5][0] = a; red[tid >> 5][1] = b; }
    __syncthreads();
    double sa = 0.0, sb = 0.0;
#pragma unroll
    for (int w = 0; w < THREADS / 32; ++w) { sa += red[w][0]; sb += red[w][1]; }
    __syncthreads();
    a = sa; b = sb;
}

// Phase 2 on tile (bi, bj): S_ij <- p_i (S_ij + dw_i w_j) p_j, and its share of tmp = u S.  S(i, j)
// is the tile's element; the row operands (pi, dwi, ui) and column operands (pj, wj, uj) are
// either registers or shared memory.  Column block bj receives the column partials in slot bi;
// for an off-diagonal tile, row block bi receives the row partials in slot bj.
template <int JMAX, class Elem>
__device__ __forceinline__ void tile_update(Elem S, const double *pi, const double *dwi, const double *ui,
                                            const double *pj, const double *wj, const double *uj,
                                            double (*part)[JMAX], int bi, int bj)
{
    double rowp[TILE], colp[TILE];
#pragma unroll
    for (int e = 0; e < TILE; ++e) { rowp[e] = 0.0; colp[e] = 0.0; }
#pragma unroll
    for (int i = 0; i < TILE; ++i)
#pragma unroll
        for (int j = 0; j < TILE; ++j) {
            const double s = (pi[i] * (S(i, j) + dwi[i] * wj[j])) * pj[j];
            S(i, j) = s;
            colp[j] += ui[i] * s;     // tmp_j += u_i S_ij
            rowp[i] += s * uj[j];     // tmp_i += S_ij u_j  (mirror element S_ji)
        }
#pragma unroll
    for (int e = 0; e < TILE; ++e) part[bi][bj * TILE + e] = colp[e];
    if (bi != bj) {
#pragma unroll
        for (int e = 0; e < TILE; ++e) part[bj][bi * TILE + e] = rowp[e];
    }
}

// Thread tid owns tile tid.  ntile <= 253 < THREADS, so there is no loop over tiles and the tile
// stays in registers across time steps.
struct RegState {
    static constexpr int JMAX = JP_MAX, THREADS = 256;
    using Smem = RefSmem<JMAX, THREADS>;
    static constexpr size_t DYN_SMEM = 0;
    static __device__ __forceinline__ Smem &smem() { __shared__ Smem sm; return sm; }

    double S[TILE][TILE];
    int bi, bj;
    bool own;

    __device__ RegState(double *) {}

    __device__ void reset(int nb, int ntile, int tid)
    {
        own = tid < ntile;
        bi = bj = 0;
        if (own) tile_coords(tid, nb, bi, bj);
#pragma unroll
        for (int i = 0; i < TILE; ++i)
#pragma unroll
            for (int j = 0; j < TILE; ++j) S[i][j] = 0.0;
    }

    __device__ void update(Smem &sm, int, int, int)
    {
        if (!own) return;
        double pi[TILE], dwi[TILE], ui[TILE], pj[TILE], wj[TILE], uj[TILE];
#pragma unroll
        for (int e = 0; e < TILE; ++e) {
            pi[e] = sm.p[bi * TILE + e]; dwi[e] = sm.dw[bi * TILE + e]; ui[e] = sm.u[bi * TILE + e];
            pj[e] = sm.p[bj * TILE + e]; wj[e] = sm.w[bj * TILE + e];   uj[e] = sm.u[bj * TILE + e];
        }
        tile_update<JMAX>([&](int i, int j) -> double & { return S[i][j]; },
                          pi, dwi, ui, pj, wj, uj, sm.part, bi, bj);
    }
};

// Thread tid owns tiles tid, tid + THREADS, ...; element e of tile g at S[e * NT + g], so the 64
// loads / stores of a tile are coalesced across the threads of a warp.
struct L2State {
    static constexpr int JMAX = 352, THREADS = 384;        // GF_MAX_J_WIDE; >= JMAX column threads
    static constexpr int NT = (JMAX / TILE) * (JMAX / TILE + 1) / 2;   // 990 tiles
    using Smem = RefSmem<JMAX, THREADS>;
    static constexpr size_t DYN_SMEM = sizeof(Smem);       // 138 KB: dynamic, with the opt-in
    static __device__ __forceinline__ Smem &smem()
    {
        extern __shared__ __align__(16) unsigned char smem_raw[];
        return *reinterpret_cast<Smem *>(smem_raw);
    }

    double *S;
    static size_t bytes(int grid) { return (size_t)grid * NT * 64 * sizeof(double); }

    __device__ L2State(double *scratch) : S(scratch + (size_t)blockIdx.x * NT * 64) {}

    __device__ void reset(int, int ntile, int tid)
    {
        for (int g = tid; g < ntile; g += THREADS)
#pragma unroll 8
            for (int e = 0; e < 64; ++e) S[e * NT + g] = 0.0;
    }

    __device__ void update(Smem &sm, int nb, int ntile, int tid)
    {
        for (int g = tid; g < ntile; g += THREADS) {
            int bi, bj;
            tile_coords(g, nb, bi, bj);
            tile_update<JMAX>([&](int i, int j) -> double & { return S[(i * TILE + j) * NT + g]; },
                              &sm.p[bi * TILE], &sm.dw[bi * TILE], &sm.u[bi * TILE],
                              &sm.p[bj * TILE], &sm.w[bj * TILE], &sm.u[bj * TILE], sm.part, bi, bj);
        }
    }
};

template <int MODE, class State>
__global__ void __launch_bounds__(State::THREADS, 1) scan_ref_kernel(ScanArgs A, double *scratch)
{
    constexpr int JMAX = State::JMAX;
    typename State::Smem &sm = State::smem();
    const int tid = threadIdx.x;
    State st(scratch);

    for (;;) {
        if (tid == 0) sm.next = atomicAdd(A.counter, 1);
        __syncthreads();
        const int item = sm.next;
        __syncthreads();
        if (item >= A.B) break;
        const int b = A.order[item];

        const int64_t n0 = A.n_off[b];
        const int64_t N = A.n_off[b + 1] - n0;
        const int64_t j0 = A.j_off[b];
        const int Jc = (int)(A.j_off[b + 1] - j0);
        const int J = 2 * Jc;
        const int nb = (J + TILE - 1) / TILE;
        const int ntile = nb * (nb + 1) / 2;
        const double *t = A.t + A.t_off[b];
        const long long y0 = A.y_like_t ? A.t_off[b] : n0;
        const double *y = A.y ? A.y + y0 : nullptr;
        const double *dg = A.diag ? A.diag + y0 : nullptr;
        const double ddiag = A.ddiag[b];

        // column k = 2*term + s  (s = 0: cos column, s = 1: sin column)
        const bool colthread = tid < J;
        double ca = 0, cb = 0, cc = 0, cd = 0;
        if (colthread) {
            const double *cf = A.coef + 4 * (j0 + (tid >> 1));
            ca = cf[0]; cb = cf[1]; cc = cf[2]; cd = cf[3];
        }
        // sum of a' in term order (same on every thread)
        double sum_a = 0.0;
        for (int j = 0; j < Jc; ++j) sum_a += A.coef[4 * (j0 + j)];

        st.reset(nb, ntile, tid);

        double wk = 0.0, Fk = 0.0;       // this column's w_{n-1}, F
        double dprev = 0.0, zprev = 0.0;
        double logdet = 0.0, quad = 0.0;
        int32_t fail = 0;
        double tprev = 0.0;

        if (N <= 0) {
            if (tid == 0) { A.logdet[b] = 0.0; if (A.quad) A.quad[b] = 0.0; A.status[b] = 0; }
            continue;
        }

        for (int64_t n = 0; n < N; ++n) {
            const double tn = t[n];
            // ---- phase 1: row generation and O(J) state ---------------------------------
            if (tid < JMAX) {
                double u = 0.0, v = 0.0, p = 1.0;
                if (colthread) {
                    double sn, cs;
                    sincos(__dmul_rn(cd, tn), &sn, &cs);
                    if (tid & 1) { u = ca * sn - cb * cs; v = sn; }
                    else         { u = ca * cs + cb * sn; v = cs; }
                    if (n > 0) {
                        p = exp(cc * (tprev - tn));
                        Fk = p * (Fk + wk * zprev);
                    }
                }
                sm.u[tid] = u; sm.v[tid] = v; sm.p[tid] = p; sm.w[tid] = wk; sm.dw[tid] = dprev * wk;
            }
            __syncthreads();

            // ---- phase 2: S update + tmp = u S ------------------------------------------
            if (n > 0) st.update(sm, nb, ntile, tid);
            __syncthreads();

            // ---- phase 3: d_n, w_n, forward sweep ---------------------------------------
            double tmpk = 0.0, r1 = 0.0, r2 = 0.0, uk = 0.0, vk = 0.0;
            if (tid < JMAX) {
                uk = sm.u[tid]; vk = sm.v[tid];
                // columns beyond nb * TILE were never written by phase 2
                if (n > 0 && tid < nb * TILE) {
                    for (int s = 0; s < nb; ++s) tmpk += sm.part[s][tid];
                }
                r1 = tmpk * uk;
                r2 = uk * Fk;
            }
            block_sum2<State::THREADS>(r1, r2, sm.red, tid);
            const double an = ((dg ? dg[n] : 0.0) + ddiag) + sum_a;
            const double dn = an - r1;
            if (!(dn > 0.0)) { fail = (int32_t)(n + 1); break; }
            if (tid < JMAX) wk = (vk - tmpk) / dn;
            double zn;
            if (MODE == MODE_SAMPLE) {
                double nrm = y ? y[n] : philox_normal(A.seed, A.seq0 + (uint64_t)b, (uint64_t)n);
                double nu = nrm * sqrt(dn);
                zn = nu;
                if (tid == 0) A.out_x[n0 + n] = nu + r2;
            } else if (MODE == MODE_LOGLIKE) {
                zn = y[n] - r2;
            } else {
                zn = 0.0;
                if (tid == 0) A.out_x[n0 + n] = dn;
                if (A.out_W && colthread) {
                    // celerite2 blocked column order [cos-block | sin-block]
                    int col = (tid & 1) * Jc + (tid >> 1);
                    A.out_W[A.w_off[b] + n * (int64_t)J + col] = wk;
                }
            }
            if (tid == 0) {
                logdet += log(dn);
                if (MODE == MODE_LOGLIKE) quad += zn * zn / dn;
            }
            dprev = dn; zprev = zn; tprev = tn;
        }
        if (tid == 0) {
            A.logdet[b] = logdet;
            if (A.quad) A.quad[b] = quad;
            A.status[b] = fail;
        }
        __syncthreads();
    }
}

template <class State>
cudaError_t launch(int mode, const ScanArgs &args, int grid, double *scratch, cudaStream_t stream)
{
    const size_t smem = State::DYN_SMEM;
    switch (mode) {
    case MODE_LOGLIKE: scan_ref_kernel<MODE_LOGLIKE, State><<<grid, State::THREADS, smem, stream>>>(args, scratch); break;
    case MODE_SAMPLE:  scan_ref_kernel<MODE_SAMPLE, State><<<grid, State::THREADS, smem, stream>>>(args, scratch); break;
    default:           scan_ref_kernel<MODE_FACTOR, State><<<grid, State::THREADS, smem, stream>>>(args, scratch); break;
    }
    return cudaGetLastError();
}

}  // namespace

size_t scan_ref_scratch_bytes(int jmax, int grid)
{
    return jmax > RegState::JMAX ? L2State::bytes(grid) : 0;
}

// scratch: scan_ref_scratch_bytes(jmax, grid) bytes of device memory (none for J <= 176)
cudaError_t launch_scan_ref(int mode, const ScanArgs &args, int jmax, int grid, double *scratch,
                            cudaStream_t stream)
{
    if (jmax <= RegState::JMAX) return launch<RegState>(mode, args, grid, nullptr, stream);
    static bool configured[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64 || !configured[dev]) {
        // the L2 store's shared memory (138 KB for 352 columns) needs the opt-in above 48 KB
        const int smem = (int)L2State::DYN_SMEM;
        cudaError_t e = cudaFuncSetAttribute(scan_ref_kernel<MODE_LOGLIKE, L2State>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(scan_ref_kernel<MODE_SAMPLE, L2State>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(scan_ref_kernel<MODE_FACTOR, L2State>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e != cudaSuccess) return e;
        if (dev >= 0 && dev < 64) configured[dev] = true;
    }
    return launch<L2State>(mode, args, grid, scratch, stream);
}

}  // namespace gf

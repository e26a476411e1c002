// Shared device/host definitions of the gadfly_b200 CUDA library (sm_100a, FP64).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace gf {

constexpr int TILE = 8;                 // register tile edge of the J x J state
constexpr int NB_MAX = 22;              // blocks of TILE columns
constexpr int JP_MAX = NB_MAX * TILE;   // 176 = GF_MAX_J
constexpr int NTILE_MAX = NB_MAX * (NB_MAX + 1) / 2;  // 253 upper-triangular tiles

enum ScanMode { MODE_LOGLIKE = 0, MODE_SAMPLE = 1, MODE_FACTOR = 2 };

// One batched scan launch.  All pointers are device pointers.
struct ScanArgs {
    int64_t B;
    const int64_t *n_off;   // [B+1]
    const int64_t *t_off;   // [B]
    const int64_t *j_off;   // [B+1] complex-term offsets into coef
    const int64_t *w_off;   // [B]   (MODE_FACTOR with W)
    const int32_t *order;   // [B]   work order (heaviest first)
    int *counter;           // work-queue head
    const double *t;
    const double *y;        // data (loglike) or normals (sample; may be null -> Philox)
    const double *diag;     // nullable
    const double *coef;     // [sum Jc][4] a', b', c, d
    const double *ddiag;    // [B]
    double *out_x;          // sample out / d out (factor)
    double *out_W;          // factor W (nullable)
    double *logdet;         // [B]
    double *quad;           // [B]
    int32_t *status;        // [B]
    uint64_t seed;
    uint64_t seq0;
    int y_like_t;           // y / diag are addressed through t_off (shared light curve)
};

// ---------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al. 2011) and the normal draw fused into the sample kernel.
// Host mirror: gadfly_b200/philox.py.
// ---------------------------------------------------------------------------------------
__host__ __device__ inline void philox4x32_10(uint32_t c[4], uint32_t k0, uint32_t k1)
{
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint64_t p0 = (uint64_t)M0 * c[0];
        uint64_t p1 = (uint64_t)M1 * c[2];
        uint32_t hi0 = (uint32_t)(p0 >> 32), lo0 = (uint32_t)p0;
        uint32_t hi1 = (uint32_t)(p1 >> 32), lo1 = (uint32_t)p1;
        uint32_t n0 = hi1 ^ c[1] ^ k0, n2 = hi0 ^ c[3] ^ k1;
        c[0] = n0; c[1] = lo1; c[2] = n2; c[3] = lo0;
        k0 += W0; k1 += W1;
    }
}

// Standard normal for sample index n of global sequence `seq`: counter (n/2, seq), both
// Box-Muller outputs are used (even n -> cos branch, odd n -> sin branch).
__device__ inline double philox_normal(uint64_t seed, uint64_t seq, uint64_t n)
{
    uint64_t m = n >> 1;
    uint32_t c[4] = {(uint32_t)m, (uint32_t)(m >> 32), (uint32_t)seq, (uint32_t)(seq >> 32)};
    philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
    uint64_t a = ((uint64_t)c[1] << 32) | c[0];
    uint64_t b = ((uint64_t)c[3] << 32) | c[2];
    const double two53 = 1.1102230246251565e-16;  // 2^-53
    double u1 = ((double)(a >> 11) + 0.5) * two53;
    double u2 = ((double)(b >> 11) + 0.5) * two53;
    double r = sqrt(-2.0 * log(u1));
    double sn, cs;
    sincospi(2.0 * u2, &sn, &cs);
    return (n & 1) ? r * sn : r * cs;
}

// sin and cos of a double that is already the rounded phase d * t: three-constant Cody-Waite
// reduction with FMA (absolute error of the reduced argument ~2e-16 for |x| < 2^30) and the
// fdlibm kernel polynomials on [-pi/4, pi/4].  No slow path, no local memory.
__device__ __forceinline__ void sincos_cw(double x, double *sn, double *cs)
{
    if (!(fabs(x) < 1.0e9)) { sincos(x, sn, cs); return; }
    const double kd = rint(x * 0.6366197723675814);
    const int q = (int)kd;
    double r = fma(-kd, 1.5707963267948966, x);
    r = fma(-kd, 6.123233995736766e-17, r);
    r = fma(-kd, -1.4973849048591698e-33, r);
    const double z = r * r;
    double ps = fma(z, 1.58969099521155010221e-10, -2.50507602534068634195e-08);
    double pc = fma(z, -1.13596475577881948265e-11, 2.08757232129817482790e-09);
    ps = fma(ps, z, 2.75573137070700676789e-06);
    pc = fma(pc, z, -2.75573143513906633035e-07);
    ps = fma(ps, z, -1.98412698298579493134e-04);
    pc = fma(pc, z, 2.48015872894767294178e-05);
    ps = fma(ps, z, 8.33333333332248946124e-03);
    pc = fma(pc, z, -1.38888888888741095749e-03);
    ps = fma(ps, z, -1.66666666666666324348e-01);
    pc = fma(pc, z, 4.16666666666666019037e-02);
    const double s = fma(ps * z, r, r);
    const double c = fma(z * z, pc, fma(-0.5, z, 1.0));
    const double s1 = (q & 1) ? c : s;
    const double c1 = (q & 1) ? s : c;
    *sn = (q & 2) ? -s1 : s1;
    *cs = ((q + 1) & 2) ? -c1 : c1;
}

// log-determinant accumulation without a log per step: a positive normal pivot is split into its
// mantissa in [1, 2) (multiplied into `prod`) and its binary exponent (summed as an integer), so
// that the product cannot overflow or underflow whatever the flux scale; sum log d = sum log(prod)
// + ln 2 * esum.  The callers flush `prod` into a log and the int `esum` into a long long every
// 8 (scan_small) or 32 (scan_blk) pivots: a sequence's exponent sum can pass 2^31.  scan_fast
// splits its pivots the same way but adds ln 2 * exponent to its log sum directly (no counter in
// its register-bound chain); scan_ref.cu takes one log per pivot.  (Subnormal pivots
// keep their value here: their exponent field is 0 and they are multiplied in unscaled.)
__device__ __forceinline__ void logdet_push(double d, double &prod, int &esum)
{
    const int hi = __double2hiint(d);
    const int ef = (hi >> 20) & 0x7ff;
    const int e = ef ? ef - 1023 : 0;
    prod *= __hiloint2double(hi - (e << 20), __double2loint(d));
    esum += e;
}
__device__ __forceinline__ double logdet_total(double logsum, double prod, long long esum)
{
    return (logsum + log(prod)) + 0.6931471805599453 * (double)esum;
}

// (f2) device feeder: stars in, celerite coefficients out (feed.cu)
struct FeedArgs {
    int64_t B;
    const double *mass, *radius, *temperature, *luminosity, *alpha, *delta;   // [B] each (alpha may be null)
    double wl_nm, amp_huber_sun, gran_power_sun, tau_sun;
    int n_gran, n_modes;
    const double *gran;     // [n_gran][3]  solar (S0, w0, Q) of the granulation terms
    const double *modes;    // [n_modes][4 + n_gran]  solar nu, Q, Gamma, unscaled height, background PSDs
};

// Upper-triangular tile enumeration: tile id -> (bi, bj), bi <= bj, row-major over bi.
__host__ __device__ inline void tile_coords(int tile, int nb, int &bi, int &bj)
{
    int row = 0, rem = tile;
    while (rem >= nb - row) { rem -= nb - row; ++row; }
    bi = row; bj = row + rem;
}

}  // namespace gf

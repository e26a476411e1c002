/*
 * gadfly_b200 -- C ABI of the B200 (sm_100a) GP hot path.
 *
 * This is the drop-in boundary: the entry points below are what the reference's
 * binding to its native solver would bind for this path.  In the reference the
 * native solver is celerite2's pybind11 module ``celerite2.driver`` reached through
 * ``celerite2.GaussianProcess`` / ``celerite2.terms``; each entry point names the
 * reference call site (file:line under the reference repo) it stands in for.
 *
 * Conventions
 *  - All floating-point data is IEEE binary64.  Time is in 1/uHz (1e6 s), angular
 *    frequency in rad*uHz, flux in ppm (reference gadfly/gp.py:61-126).
 *  - A "sequence" is one light curve + one kernel (one star, one realisation, or one
 *    hyper-parameter grid point).  Batches are described CSR-style:
 *      n_off[B+1]  offsets of sequence b's samples in y / diag / out          (HOST int64)
 *      t_off[B]    offset of sequence b's time stamps in t (sequences may share t) (HOST int64)
 *      j_off[B+1]  offsets of sequence b's complex terms in coef               (HOST int64)
 *    coef is [sum Jc][4] = (a', b', c, d) per complex term, already exposure-integrated
 *    (TermConvolution coefficients); ddiag[B] is the constant added to the diagonal.
 *    A real term (a, c) is passed as the complex term (a, 0, c, 0).
 *    The state width of sequence b is J_b = 2 * (j_off[b+1] - j_off[b]).
 *  - Bulk pointers (t, y, diag, coef, ddiag, normals and all outputs) may each be a
 *    device pointer or a host pointer; the library classifies every pointer with
 *    cudaPointerGetAttributes and stages host buffers through its own device scratch
 *    (cudaMemcpyAsync on the handle's stream).  The three offset arrays are always host.
 *  - Return value: 0 = ok; < 0 = argument error (GF_E_*); > 0 = cudaError_t.
 *    gf_last_error() gives a message.  Per-sequence numeric failure (non-positive pivot)
 *    is reported in status[b] = 1 + index of the first d[n] <= 0, 0 if none -- the
 *    condition on which celerite2 raises LinAlgError (reference gadfly/gp.py:188-192).
 *  - No global state except the handle; calls on one handle are serialised by the caller.
 *    Entry points return after the work has completed (outputs valid), unless GF_FLAG_ASYNC
 *    is set, in which case all outputs are valid after gf_synchronize().
 *  - Streams.  A handle owns one compute stream (gf_stream) on which every kernel runs, and
 *    two copy streams for host buffers (staging in, results out), so that the copies of one
 *    call overlap the kernel of the previous GF_FLAG_ASYNC call (H2D of the next light curves
 *    beside the running scan, D2H of samples beside the next scan).
 *    DEVICE pointers are read and written on the compute stream only, and the library does not
 *    know who produced them: device inputs must be complete with respect to gf_stream(h) when
 *    the entry point is called, and consumers of device outputs must order themselves after
 *    it.  gf_wait_stream(h, producer) / gf_stream_wait(h, consumer) insert exactly these
 *    dependencies (event record + cudaStreamWaitEvent, nothing blocks the host); the Python
 *    binding calls them for every torch CUDA tensor it is handed.
 */
#ifndef GADFLY_B200_H
#define GADFLY_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct gf_context *gf_handle;

enum {
    GF_OK = 0,
    GF_E_ARG = -1,        /* null / inconsistent argument */
    GF_E_UNSORTED = -2,   /* reserved */
    GF_E_TOO_WIDE = -3,   /* J_b exceeds GF_MAX_J */
    GF_E_NOMEM = -4
};

/* widest state the register-resident scans support (22 blocks of 8) */
#define GF_MAX_J 176
/* widest state at all: batches containing a kernel with GF_MAX_J < J <= GF_MAX_J_WIDE (the solar kernel
 * plus up to 90 extra terms, reference gadfly/core.py:405-427) run on a slower kernel whose state lives
 * in L2-resident global scratch; the stored-factor sweeps (K4) take any width up to this one too */
#define GF_MAX_J_WIDE 352

/* flags */
#define GF_FLAG_ASYNC 1u          /* do not synchronise before returning: host outputs are valid (and
                                      their buffers must stay alive) until gf_synchronize / gf_wait /
                                      the next blocking call on the handle.  Pinned host outputs are
                                      written by the copy-out stream; PAGEABLE ones up to 1 MB each go
                                      through a pinned ring inside the handle and are delivered by those
                                      three calls (a device-to-host copy into pageable memory would hold
                                      the host until the kernel before it has finished); a larger
                                      pageable output is copied directly, i.e. the call blocks */
#define GF_FLAG_REFERENCE_ORDER 2u /* use the simple reference-order scan kernel (validation) */
#define GF_FLAG_WIDE_KERNEL 8u     /* do not take the one-warp-per-sequence path for narrow batches
                                      (all J <= 32); validation of that path against the wide kernel */
#define GF_FLAG_BLOCKED 16u        /* experimental: the 4-step blocked scan kernel (csrc/scan_blk.cu) for
                                      gf_loglike_batched / gf_sample_batched */
#define GF_FLAG_SHARED_Y 4u        /* y / diag (gf_loglike_batched) are laid out like t: sequence b
                                      reads y[t_off[b] + n], so that one light curve serves many
                                      hyper-parameter sets (stride-0 descriptor of SURVEY.md 8b) */

/* ---- lifetime --------------------------------------------------------------------- */
int gf_create(int device, gf_handle *out);
int gf_destroy(gf_handle h);
int gf_synchronize(gf_handle h);
const char *gf_last_error(gf_handle h);
/* the handle's compute stream as a cudaStream_t (so callers can record events on it) */
void *gf_stream(gf_handle h);
/* make the compute stream wait for everything enqueued so far on `producer` (a cudaStream_t;
 * NULL = the legacy default stream): call it before passing device buffers that `producer` wrote */
int gf_wait_stream(gf_handle h, void *producer);
/* Completion tickets for GF_FLAG_ASYNC calls with HOST outputs: gf_ticket() marks "everything issued on
 * this handle so far, including the copies back to host buffers" and returns a ticket (> 0);
 * gf_wait(h, ticket) blocks the host until that point -- and not until later calls -- has completed, so
 * that a caller can keep the next call's copies and kernels queued behind the running ones.
 * Up to 8 tickets may be outstanding. */
int64_t gf_ticket(gf_handle h);
int gf_wait(gf_handle h, int64_t ticket);
/* make `consumer` (a cudaStream_t) wait for everything enqueued so far on the compute stream:
 * call it before `consumer` reads device outputs of a GF_FLAG_ASYNC call */
int gf_stream_wait(gf_handle h, void *consumer);
/* SM count, measured FP64 FMA peak [flop/s] from a DFMA microbenchmark (0 if !measure) */
int gf_device_info(gf_handle h, int *sm_count, double *fp64_flops, int measure);
/* kernels launched by this handle since creation (the bench's gpu_launches claim) */
int64_t gf_launch_count(gf_handle h);
/* device time [ms] of the most recent scan / psd kernel launch, from CUDA events recorded
 * on the handle's stream around the launch (valid after the call returned / synchronised) */
float gf_last_kernel_ms(gf_handle h);
/* which scan kernel served the most recent scan launch of the handle (gf_loglike_batched,
 * gf_sample_batched, gf_factor_batched and the factor scan of gf_*_multi): one of GF_PATH_*,
 * GF_PATH_NONE before the first scan launch (a call with B = 0 launches nothing) */
enum {
    GF_PATH_NONE = -1,
    GF_PATH_FAST = 0,      /* csrc/scan_fast.cu: register-resident state, J <= GF_MAX_J */
    GF_PATH_SMALL = 1,     /* csrc/scan_small.cu: one warp per sequence, every J <= 32 */
    GF_PATH_REF = 2,       /* csrc/scan_ref.cu, state in registers: GF_FLAG_REFERENCE_ORDER */
    GF_PATH_WIDE = 3,      /* csrc/scan_ref.cu, state in L2-resident scratch: some J > GF_MAX_J */
    GF_PATH_BLOCKED = 4    /* csrc/scan_blk.cu: GF_FLAG_BLOCKED */
};
int gf_last_scan_path(gf_handle h);

/* ---- K1: fused factor + forward solve -> log-likelihood pieces ---------------------
 * Replaces, per sequence: celerite2 GaussianProcess.compute (driver.factor; reference
 * gadfly/gp.py:59,202-204) followed by log_likelihood (driver.solve_lower; reference
 * gadfly/gp.py:350):   logdet[b] = sum_n log d_n ,  quad[b] = sum_n z_n^2 / d_n  with
 * z = L^-1 y.  log L = -(quad + logdet + N log 2 pi) / 2 is formed by the caller.
 * Nothing of size N*J is materialised. */
int gf_loglike_batched(gf_handle h, int64_t B, const int64_t *n_off, const int64_t *t_off,
                       const int64_t *j_off, const double *t, int64_t t_len, const double *y,
                       const double *diag /* nullable */, const double *coef,
                       const double *ddiag, double *logdet, double *quad, int32_t *status,
                       uint32_t flags);

/* ---- K2: fused factor + lower-triangular dot -> samples ----------------------------
 * Replaces celerite2 GaussianProcess.compute + dot_tril / sample (driver.factor +
 * driver.matmul_lower; reference gadfly/gp.py:327,391):  out = L_c (sqrt(d) o n).
 * normals == NULL: n is drawn inside the kernel from Philox4x32-10 keyed by (seed), counter
 * (sample index / 2, global sequence id seq0 + b, stream), Box-Muller on two 53-bit uniforms
 * (reproducible on the host: see gadfly_b200/philox.py).  normals != NULL: n is read, laid out
 * like out.  logdet (nullable) also receives sum log d. */
int gf_sample_batched(gf_handle h, int64_t B, const int64_t *n_off, const int64_t *t_off,
                      const int64_t *j_off, const double *t, int64_t t_len,
                      const double *diag /* nullable */, const double *coef,
                      const double *ddiag, const double *normals /* nullable */, uint64_t seed,
                      uint64_t seq0, double *out, double *logdet /* nullable */,
                      int32_t *status, uint32_t flags);

/* ---- K1m / K2m: k right-hand sides per sequence on ONE factor ----------------------------
 * SURVEY.md 8b's `k` ("many y / many realisations per factor"): celerite2 factors once in
 * compute() and then serves sample(size=k) (reference gadfly/gp.py:372-395, the (N, k) branch of
 * np.random.randn) and repeated log_likelihood calls from the stored factor.  Here: one factor scan
 * per sequence (d and W in library scratch, sum_b N_b J_b doubles of device memory), then ALL B k
 * O(N J) sweeps in one launch, one CTA each, sharing the factor.
 *   gf_sample_multi   out[b][r][:] = L_b (sqrt(d_b) o n_{b,r}),  r < k;  out / normals are laid out
 *                     [b][r][n] (offset k n_off[b] + r N_b); normals == NULL draws n_{b,r} from
 *                     Philox with the global realisation index seq0 + b k + r (gadfly_b200/philox.py)
 *   gf_loglike_multi  quad[b][r] = z^T D^-1 z, z = L_b^-1 y_{b,r};  y laid out like out, quad is
 *                     [B][k]; logdet[B] (nullable), status[B] as for the fused entry points
 * For one realisation per factor the fused K1 / K2 are cheaper (nothing is stored). */
int gf_sample_multi(gf_handle h, int64_t B, const int64_t *n_off, const int64_t *t_off,
                    const int64_t *j_off, const double *t, int64_t t_len,
                    const double *diag /* nullable */, const double *coef, const double *ddiag,
                    int64_t k, const double *normals /* nullable */, uint64_t seed, uint64_t seq0,
                    double *out, double *logdet /* nullable */, int32_t *status, uint32_t flags);
int gf_loglike_multi(gf_handle h, int64_t B, const int64_t *n_off, const int64_t *t_off,
                     const int64_t *j_off, const double *t, int64_t t_len,
                     const double *diag /* nullable */, const double *coef, const double *ddiag,
                     int64_t k, const double *y, double *logdet /* nullable */, double *quad,
                     int32_t *status, uint32_t flags);

/* ---- K3: factor, materialising d[N] (and W[N,J] if W != NULL) ----------------------
 * Replaces driver.factor where the factor itself is wanted (reference gadfly/gp.py:202-204
 * followed by apply_inverse / predict, gadfly/gp.py:370,232).  d is laid out like y;
 * W is [sum_b N_b * J_b], row-major per sequence, offsets w_off[B] (HOST int64), columns in
 * celerite2's blocked order [cos-block | sin-block]. */
int gf_factor_batched(gf_handle h, int64_t B, const int64_t *n_off, const int64_t *t_off,
                      const int64_t *j_off, const int64_t *w_off, const double *t, int64_t t_len,
                      const double *diag /* nullable */, const double *coef,
                      const double *ddiag, double *d, double *W /* nullable */,
                      double *logdet, int32_t *status, uint32_t flags);

/* ---- K4: O(N J) sweeps on a stored factor -----------------------------------------
 * Replaces driver.solve_lower / matmul_lower / solve_upper / matmul_upper (reference
 * gadfly/gp.py:327,350,370).  op: 0 solve_lower (Z = L^-1 Y), 1 matmul_lower (Z = L Y),
 * 2 solve_upper (Z = L^-T Y), 3 matmul_upper (Z = L^T Y).  Y and Z are [N] per sequence,
 * laid out like y; Z may alias Y.  U rows are regenerated from (t, coef) on the fly. */
int gf_sweep_batched(gf_handle h, int op, int64_t B, const int64_t *n_off, const int64_t *t_off,
                     const int64_t *j_off, const int64_t *w_off, const double *t, int64_t t_len,
                     const double *coef, const double *W, const double *Y, double *Z,
                     uint32_t flags);

/* ---- K5: kernel power spectral density on a dense frequency grid -------------------
 * Replaces celerite2 Term.get_psd / TermConvolution.get_psd (reference gadfly/psd.py:151,
 * gadfly/tests/test_core.py:34; closed form gadfly/core.py:33-41):
 *   out[b][f] = sqrt(2/pi) sum_j ((a c + b d)(c^2+d^2) + (a c - b d) w^2)
 *                                / (w^4 + 2 (c^2 - d^2) w^2 + (c^2+d^2)^2)  * sinc^2(delta_b w / 2)
 * with the UN-convolved coefficients coef_base[sum Jc][4] and w = omega[f], shared by all b. */
int gf_psd_batched(gf_handle h, int64_t B, const int64_t *j_off, const double *coef_base,
                   const double *delta /* [B] */, const double *omega, int64_t F,
                   double *out /* [B][F] */, uint32_t flags);

/* ---- K7: observed power spectrum and its binning (the other side of the round trip) ------
 * Replaces PowerSpectrum._fft (reference gadfly/psd.py:566-587) and bin_power_spectrum with
 * spectral_binning / spectral_binning_err (gadfly/psd.py:186-297) for B evenly sampled light curves
 * at once, so that sample -> observed PSD -> binning -> comparison with gf_psd_batched stays on the
 * device.  The transform is cuFFT (D2Z, bound with dlopen at first use; a positive cudaError is
 * returned if libcufft is not installed); normalisation and binning are this library's kernels.
 *   gf_power_spectrum_batched  power[b][i] = |rfft(flux_b)|_i^2 * d / sqrt(2 pi) / N, flux [B][N] in
 *                              ppm, d = cadence in 1/uHz; i runs over N/2 + 1 frequencies
 *                              (rfftfreq(N, d)), without the first one unless include_zero
 *   gf_bin_power_batched       bins are index ranges [lo[k], lo[k] + cnt[k]) (HOST int64, from
 *                              searchsorted of the bin edges) of the shared monotone axis[F] (log10 f
 *                              or f); stat[b][k] = trapezoidal mean of power_b over the bin,
 *                              err[b][k] = std / sqrt(n) * mean(axis) / span / constant; one-point bins
 *                              return that point, empty bins NaN */
int gf_power_spectrum_batched(gf_handle h, int64_t B, int64_t N, const double *flux, double d,
                              int include_zero, double *power, uint32_t flags);
int gf_bin_power_batched(gf_handle h, int64_t B, int64_t F, int64_t nb, const int64_t *lo,
                         const int64_t *cnt, const double *axis, const double *power, double constant,
                         double *stat, double *err, uint32_t flags);

/* ---- K6: conditional mean at new times ------------------------------------------------
 * Replaces celerite2 driver.general_matmul_lower + general_matmul_upper as ConditionalDistribution
 * uses them for predict(y, t=new times) (reference gadfly/gp.py:243-306, docs/gadfly/synth.rst:193-201):
 *   mu[i] = sum_m k(|ts[i] - t[m]|) alpha[m],  k = the semiseparable kernel of coef[Jc][4]
 * (a', b', c, d after the exposure transform), alpha = K^-1 (y - mean) from the sweeps.
 * t[N] and ts[M] sorted ascending; O((N + M) Jc). */
int gf_conditional_mean(gf_handle h, int64_t N, const double *t, int64_t M, const double *ts,
                        int64_t Jc, const double *coef, const double *alpha, double *mu,
                        uint32_t flags);

/* ---- (f2) hyper-parameter feeder ------------------------------------------------------
 * Stellar parameters -> kernel coefficients for B stars at once: the batched form of
 * Hyperparameters.for_star (reference gadfly/core.py:107-333, scaling relations gadfly/scale.py) followed
 * by the kernel assembly of StellarOscillatorKernel.__init__ (gadfly/core.py:345-394: celerite2
 * SHOTerm.get_coefficients + TermConvolution.get_coefficients with its diagonal correction).
 *   mass, radius, temperature, luminosity [B]  in M_sun, R_sun, K, L_sun
 *   alpha [B] or NULL     bandpass amplitude ratio (gf_bandpass_amplitude; NULL = 1, flat bandpass)
 *   wavelength_nm         mean wavelength of the bandpass (550 for a flat one)
 *   delta [B]             exposure time in 1/uHz
 *   gran  [n_gran][3]     solar (S0, w0, Q) of the granulation terms        } the solar fit the reference
 *   modes [n_modes][4 + n_gran]  per solar p-mode: nu, Q, Gamma, unscaled   } ships as data/hyperparameters.json,
 *                         height, background PSD of each granulation term   } reduced on the host once
 * Outputs: j_off [B + 1] (HOST), and compacted in that CSR layout sho [.][3] = (S0, w0, Q) (may be NULL),
 * coef [.][4] = (a', b', c, d), base [.][4] = (a, b, c, d) (may be NULL), ddiag [B]; the arrays hold
 * cap_terms rows (B * (n_gran + n_modes) always suffices).  The reference drops scaled terms whose frequency
 * or power is not positive; a kept term with Q < 0.5 is an error (GF_E_ARG). */
int gf_feed_stars(gf_handle h, int64_t B, const double *mass, const double *radius, const double *temperature,
                  const double *luminosity, const double *alpha, double wavelength_nm, const double *delta,
                  int64_t n_gran, const double *gran, int64_t n_modes, const double *modes, int64_t cap_terms,
                  int64_t *j_off, double *sho, double *coef, double *base, double *ddiag, uint32_t flags);
/* The kernel-assembly half alone, for hyper-parameters that are already (S0, w0, Q) in CSR layout (a
 * hyper-parameter lattice, the perturbed kernels of a finite-difference gradient): sho [j_off[B]][3] ->
 * coef, base (may be NULL) [j_off[B]][4], ddiag [B]; celerite2 SHOTerm.get_coefficients +
 * TermConvolution.get_coefficients as called from reference gadfly/core.py:345-394.  Q < 0.5: GF_E_ARG. */
int gf_feed_sho(gf_handle h, int64_t B, const int64_t *j_off, const double *sho, const double *delta,
                double *coef, double *base, double *ddiag, uint32_t flags);
/* Morris et al. (2020) Eqn 11 amplitude ratio of a tabulated bandpass for B effective temperatures
 * (reference gadfly/scale.py:635-729): trapezoid quadratures of the Planck function and its temperature
 * derivative over wl_um [n_wl] (micron) weighted by transmittance [n_wl] */
int gf_bandpass_amplitude(gf_handle h, int64_t B, const double *temperature, int64_t n_wl, const double *wl_um,
                          const double *transmittance, double *out, uint32_t flags);

#ifdef __cplusplus
}
#endif
#endif /* GADFLY_B200_H */

/*
 * gpb200.h - C ABI of libgpb200.so: the B200 (sm_100a) Gaussian-process inference hot path
 * behind the GPtest Python API.
 *
 * The reference (osurdml/GPtest) has no FFI: its boundary is the Python module API of GPr.py,
 * GPc.py and GPpref.py.  Each entry point below is what a ctypes binding of one reference
 * method needs; the reference method it replaces is cited as file:line into the reference.
 * gptest_b200/{GPr,GPc,GPpref}.py are those bindings (see INTEGRATION.md).
 *
 * Conventions
 *   - every function returns 0 on success, < 0 on argument / CUDA errors (text through
 *     gpb_last_error), and reports numerical failure LAPACK-style through *info
 *     (info > 0: leading minor of that order is not positive definite) so that the Python side
 *     can raise numpy.linalg.LinAlgError exactly where the reference does (GPr.py:62,
 *     GPpref.py:126-135);
 *   - all matrices are fp64, row-major (numpy C order), sizes are in elements;
 *   - "host" pointers are ordinary process memory, copied inside the call; pointers named
 *     *_dev are CUDA device pointers on the handle's device;
 *   - one handle = one device + one stream; calls on a handle are serialised by the caller;
 *   - host-pointer calls return after their results are in host memory;
 *   - there is no CPU fallback anywhere: without a CUDA device gpb_create fails.
 */
#ifndef GPB200_H
#define GPB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct gpb_handle gpb_handle;

/* ---- lifecycle ------------------------------------------------------------------------ */
int gpb_version(void);
/* The handle owns a private stream; gpb_set_stream adopts a caller stream instead (a
 * cudaStream_t such as torch.cuda.current_stream().cuda_stream; 0 = the legacy default stream).
 * All kernels of the handle are ordered on that stream; gpb_get_stream returns it so that the
 * caller can record CUDA events on it. */
int gpb_create(int device, gpb_handle** out);
int gpb_set_stream(gpb_handle* h, void* stream);
void* gpb_get_stream(gpb_handle* h);
int gpb_destroy(gpb_handle* h);
const char* gpb_last_error(gpb_handle* h);            /* h may be NULL: last create error */
/* tunables: "lookahead" (0/1), "nb_tiles" (outer block = nb_tiles*128 columns: 1,2,4),
 * "cov_kind" (covariance of the regression entry points: 0 squared exponential = GPr.py:90-110, the default;
 * 1 Matern 3/2, 2 Matern 5/2 - same hyper-parameter layout and ARD scaling; extension, SURVEY 8f rank 4),
 * "batch_chunk" (problems resident at once in the batched path), "la_max_batch" (largest batch that
 * uses the look-ahead schedule; default: all), and the schedule knobs (defaults are the measured best; the A/B
 * scripts under tools/ use them): "nb_switch8", "nb_switch4", "nb_switch2" (block width 8/4/2 tiles while at least
 * that many tile columns remain), "split_tiles", "small_tile_threshold", "dag_streams", "dag_min_tiles",
 * "dag_min_width", "dag_big_tiles" (chunked multi-stream trailing update), "chain_on_panel_stream", "pdl",
 * "pdl_max_tiles", "pdl_tail" (programmatic dependent launch), "potrf_variant" (3: diagonal tile blocked inside the CTA,
 * the default; 2: the register-resident sweep of round 1), "potrf_refine", "thin_tile_max" (32-row CTA-tiles on the panel
 * chain), "tri_skip" (zero / unused halves skipped in the panel TRSM and the symmetric updates), "fuse_rhs" (the forward
 * substitution L z = y - m rides on the factorisation: diagonal-tile kernel + panel TRSM epilogue; 0 = appended row /
 * separate pass as in round 1), "trsm_balance" (8-warp CTAs for a panel TRSM with a triangular B), "trsm_persist" (resident waves of its grid), "trsm_tile_threshold"
 * (128-tile count from which the panel TRSM uses 128 x 128 CTA-tiles; default never), "batch_small_k" (batched updates
 * with k up to this use 64 x 64 CTA-tiles), "batch_plain_width", "fine_warps", "persistent_waves", "stagger" (see
 * gpb_context.cuh).  "pdl", "potrf_variant", "potrf_refine", "fine_warps", "trsm_balance", "trsm_persist", "persistent_waves" and
 * "stagger" are process-wide, the rest per handle.  Returns <0 if unknown. */
int gpb_set_option(gpb_handle* h, const char* name, int64_t value);
/* stage times (ms) of the last GPr/potrf call measured with CUDA events on the handle's
 * stream: [0]=covariance assembly [1]=factorisation (+fused forward solves)
 * [2]=reductions/finish [3]=gradient stage [4]=whole device section.  n <= 8.
 * After gpb_pref_evidence_grad: [0]=factorisation of K^-1 + W at the mode (0 if already factored) [1]=dense stages
 * (the two sweeps, G^-1, A) [2]=per-pair / per-item kernels, vectors and the trace pass [4]=whole call.
 * After gpb_gpc_evidence_grad: [0]=factorisation of I + W^1/2 K W^1/2 at the mode (0 if already factored) [1]=dense
 * stages (the sweep of K W^1/2, B^-1) [2]=per-item kernel, R, vectors and the trace pass [4]=whole call. */
int gpb_get_timings(gpb_handle* h, float* ms, int n);
/* number of kernels launched by this handle since creation (bench.py's gpu_launches) */
int64_t gpb_launch_count(gpb_handle* h);

/* ---- training data: GaussianProcess.__init__ (GPr.py:17-42) stores trainInput/Target --- */
int gpb_set_train(gpb_handle* h, const double* X, int64_t n, int32_t d, const double* y);
int gpb_set_train_dev(gpb_handle* h, const double* X_dev, int64_t n, int32_t d, const double* y_dev);

/* ---- covariance assembly ---------------------------------------------------------------
 * SquaredExponential.compute_Kxx_matrix (GPr.py:99-103): sn2*I + sf2*exp(-0.5*sqdist(x/l,x/l)),
 * full symmetric n x n.  khyp = [l_1..l_D, sf2, sn2]: the NATURAL parameters exactly as
 * SquaredExponential.__init__ derives them on the host (GPr.py:93-97: hyp = exp(logHyp),
 * M = hyp[:n-2], sf2 = hyp[n-2]**2, sn2 = hyp[n-1]**2) - the binding keeps those three lines so
 * that the attributes .hyp/.M/.sf2/.sn2 stay bit-identical to the reference's.
 * flags bit0: clip r^2 at 0 and force a zero diagonal distance (GPy RBF semantics, GPpref.py:122);
 * out_is_dev != 0: K_out is a device pointer (n*n doubles). */
int gpb_se_ard_kxx(gpb_handle* h, const double* khyp, double* K_out, int32_t out_is_dev, int32_t flags);
/* SquaredExponential.compute_Kxz_matrix (GPr.py:105-110): n x m, no noise. Z is host (m x d). */
int gpb_se_ard_kxz(gpb_handle* h, const double* khyp, const double* Z, int64_t m,
                   double* Kxz_out, int32_t out_is_dev);

/* squared_distance(A, B) (GPr.py:4-13) between the training inputs (A, n x d) and B (m x d, host):
 * |a|^2 + |b|^2 - 2ab, n x m to host memory. */
int gpb_sqdist(gpb_handle* h, const double* B, int64_t m, double* out);

/* ---- regression -------------------------------------------------------------------------
 * GaussianProcess.compute_likelihood (GPr.py:57-69): nlml = 0.5 (y-m)' K^-1 (y-m) +
 * sum(log diag L) + n/2 log(2 pi).  grad (d+2 doubles, may be NULL): d nlml / d loghyp
 * w.r.t. the LOG hyper-parameters [log l_1..l_D, log sf, log sn] (the value+gradient GPy's
 * optimiser consumes in GP_parameter_fit.py:32-33). */
int gpb_gpr_nlml(gpb_handle* h, const double* khyp, double mean, double* nlml,
                 double* grad, int32_t* info);
/* GaussianProcess.compute_prediction (GPr.py:45-54): fz = Kzx K^-1 y, cov = sf2 - diag(Kzx K^-1 Kxz)
 * for m test points Z (host, m x d); outputs host arrays of m doubles. */
int gpb_gpr_predict(gpb_handle* h, const double* khyp, double mean, const double* Z, int64_t m,
                    double* fz, double* cov, int32_t* info);
/* Joint posterior of the latent f at mz test points Z (host, mz x d), beyond the reference's diagonal (GPr.py:50):
 * fz (mz, host) exactly what gpb_gpr_predict returns for the same arguments, and
 * cov (mz x mz, row-major, full symmetric) = K(Z,Z) - Kzx K^-1 Kxz, plus sn2 * I when flags bit0 is set
 * (the predictive of noisy observations).  cov_is_dev != 0: cov is a device pointer.
 * info > 0: K is not positive definite (as gpb_gpr_predict).
 * Stage times (gpb_get_timings): [0]=assembly of K, Kzx, Kzz [1]=factorisation with the test rows riding along
 * [2]=the product Kzz - V V^T (V = Kzx L^-T) [4]=whole call. */
int gpb_gpr_predict_full(gpb_handle* h, const double* khyp, double mean, const double* Z, int64_t mz,
                         double* fz, double* cov, int32_t cov_is_dev, int32_t flags, int32_t* info);
/* nsamp joint draws f_s = fz + L e_s with L L^T = cov + jitter * I (cov as above, same flags), samples nsamp x mz host.
 * e_s[i] are standard normals generated on the device from (seed, s, i) alone: Philox4x32-10 with counter
 * (i/2 lo, i/2 hi, s lo, s hi) and key (seed lo, seed hi), then Box-Muller on the pair (DESIGN.md section 4.8).
 * jitter (may be NULL): 0 if cov factors, otherwise the first of 1e-12 sf2, 1e-11 sf2, ... sf2 that does; an error
 * (return < 0) if none does.  info > 0: K is not positive definite, no samples are written.
 * Stage times as gpb_gpr_predict_full, and [3]=the factorisation attempts of cov, the normals, D = E L^T, the finish
 * and the copy-out. */
int gpb_gpr_sample(gpb_handle* h, const double* khyp, double mean, const double* Z, int64_t mz, int64_t nsamp,
                   uint64_t seed, int32_t flags, double* samples, double* jitter, int32_t* info);
/* B independent evaluations of compute_likelihood on the same (X, y) with different
 * hyper-parameters (the grid / multi-start fits GP_parameter_fit.py:32-33 runs one by one).
 * khyp: B x (d+2) host, NATURAL parameters [l_1..l_d, sf2, sn2] per row (as for gpb_gpr_nlml); nlml: B host;
 * grad: B x (d+2) host or NULL, w.r.t. the LOG hyper-parameters; info: B host. */
int gpb_gpr_nlml_batched(gpb_handle* h, const double* khyp, int64_t B, double mean,
                         double* nlml, double* grad, int32_t* info);

/* ---- growing training sets (GP_parameter_fit.py:61-63,52) ----------------------------------
 * The reference replays an experiment by calling set_XY on ever longer prefixes (five more points each time)
 * and predicting on a 100x100 grid - a full refit per step.  With fixed hyper-parameters the factor of the
 * longer prefix extends the factor of the shorter one, so the handle keeps it on the device:
 *   gpb_gpr_grow_begin   fixes khyp = [l_1..l_d, sf2, sn2], the mean and the capacity (points); n = 0
 *   gpb_gpr_grow_append  adds m points (X_new m x d, y_new m; host) and returns the NLML of the enlarged set
 *                        (what gpb_gpr_nlml returns for it); work O((n+m)^2 m) instead of (n+m)^3/3;
 *                        info > 0: non-positive pivot at that (1-based) row, the stored factor is then invalid
 *   gpb_gpr_grow_predict compute_prediction (GPr.py:45-54) from the stored factor, any mz
 *   gpb_gpr_grow_size    points appended so far (-1 without gpb_gpr_grow_begin)
 * The state has its own buffers: other calls on the handle do not disturb it. */
int gpb_gpr_grow_begin(gpb_handle* h, const double* khyp, int32_t d, double mean, int64_t capacity);
int gpb_gpr_grow_append(gpb_handle* h, const double* X_new, const double* y_new, int64_t m, double* nlml,
                        int32_t* info);
int gpb_gpr_grow_predict(gpb_handle* h, const double* Z, int64_t mz, double* fz, double* cov);
int64_t gpb_gpr_grow_size(gpb_handle* h);

/* ---- dense factorisation on caller-owned device memory (np.linalg.cholesky, GPr.py:62) ---
 * In-place lower Cholesky of the n x n row-major matrix A_dev (leading dimension lda >= n,
 * n % 128 == 0, lda % 2 == 0); only the lower triangle is read and written. */
int gpb_potrf_lower_dev(gpb_handle* h, double* A_dev, int64_t n, int64_t lda, int32_t* info);
/* Same on a host matrix of any n (copied, padded, factored, lower triangle copied back,
 * strict upper triangle zeroed like numpy). */
int gpb_potrf_lower(gpb_handle* h, double* A, int64_t n, int32_t* info);
/* C (M x N, ldc) = beta*C + alpha * A (M x K, lda) * B (N x K, ldb)^T on device memory through
 * the TMA-fed DMMA tile kernel; M, N, K multiples of 128, alpha/beta in {(1,0), (-1,1)}.
 * Test / bench hook for the kernel the factorisation spends its time in. */
int gpb_dgemm_nt_dev(gpb_handle* h, double* C_dev, int64_t ldc, const double* A_dev, int64_t lda,
                     const double* B_dev, int64_t ldb, int64_t M, int64_t N, int64_t K,
                     double alpha, double beta);

/* ---- binary classification (GPc.py intent; R&W Alg. 3.1 / 3.2) ---------------------------
 * labels y in {-1,+1} (host, n), khyp = [l_1..l_D, sf2], link 0 = probit (GPc.py:21),
 * 1 = logit (GPc.py:17-19).  f_inout: start (if use_f0) and result mode (n).
 * trace (2*max_iter doubles or NULL): (f_error, objective) per iteration.
 * A handle keeps one Laplace state: the one the last gpb_gpc_laplace or gpb_pref_laplace left in the work space.
 * gpb_gpc_predict / gpb_gpc_evidence_grad need it to come from gpb_gpc_laplace; a fit of either kind replaces it,
 * and any other call that uses the work space invalidates it (error, not garbage). */
int gpb_gpc_laplace(gpb_handle* h, const double* y, const double* khyp, int32_t link,
                    double delta_f, int32_t max_iter, int32_t use_f0, double* f_inout,
                    double* lml, int32_t* iters, double* trace, double* jitter, int32_t* info);
int gpb_gpc_predict(gpb_handle* h, const double* Z, int64_t m, double* mu, double* var, double* prob);
/* gpb_gpc_evidence_grad (opt-in, beyond the reference): the lml the last gpb_gpc_laplace returned (R&W eq. 3.32, bit for
 *   bit) and its exact gradient, grad[d + 1] = d lml / d [log l_1 .. log l_d, log sf] (the loghyp layout of the GPc
 *   binding; sf2 = khyp[d]), with the jitter the fit chose held fixed.  R&W Alg. 5.1 at the returned mode f = K a, with
 *   the implicit term's sign as in GPML's infLaplace (DESIGN.md section 4.3).  Exact only at a stationary point, so a
 *   fit whose loop stopped on max_iter with max|f_new - f| > delta_f is refused; so is a call without a current
 *   gpb_gpc_laplace state.  A refused call leaves the state usable.  Costs about 1.67 n^3 flop on the DMMA kernels.  The
 *   factor of B = I + W^1/2 K W^1/2 is overwritten, so the next gpb_gpc_predict (or gradient) factors it again (same
 *   results). */
int gpb_gpc_evidence_grad(gpb_handle* h, double* lml, double* grad);

/* ---- pairwise preferences ----------------------------------------------------------------
 * PreferenceGaussianProcess.calc_laplace (GPpref.py:112-157).  uvi: P x 2 int64 item indices
 * (column 0 = u, column 1 = v), y: P labels in {-1,+1}, khyp = [l_1..l_D, variance] as the
 * binding sets them on the kernel (GPpref.py:113-114).  grad_mode 0 = the reference's last-write-wins gradient (GPpref.py:77-78),
 * 1 = accumulate (true Newton).  sigma is the probit noise actually used (1.0 reproduces the
 * reference, GPpref.py:115).  The loop runs on the device until max|f_new - f| <= delta_f or
 * max_iter; trace gets (f_error, lml) per iteration like the reference's print (GPpref.py:154). */
int gpb_pref_laplace(gpb_handle* h, const int64_t* uvi, const double* y, int64_t P,
                     const double* khyp, double sigma, double delta_f, int32_t max_iter,
                     int32_t grad_mode, int32_t use_f0, double* f_inout, double* lml,
                     int32_t* iters, double* trace, double* jitter, int32_t* info);
/* Opt-in extensions beyond the reference (SURVEY 8f rank 3).  They use the handle's one Laplace state (mode, K^-1,
 * comparison graph), which must come from gpb_pref_laplace: a later gpb_gpc_laplace replaces it, and any other call
 * that uses the work space invalidates it (error, not garbage).  W is re-evaluated at the returned mode and K^-1 + W
 * factored once, on first use.
 * gpb_pref_evidence: the Laplace approximation of the log evidence, R&W eq. 3.32:
 *   sum_k log Phi(z_k) - f' K^-1 f / 2 - log|I + K W| / 2
 *   (the reference's log_marginal, GPpref.py:90-94, has no W term and counts log|K| a quarter, GPpref.py:131).
 * gpb_pref_predict: latent posterior at mz test items Z (host, mz x d): mean = k*' K^-1 f and
 *   var = k** - k*' (K + W^-1)^-1 k* = k** - k*' K^-1 k* + (K^-1 k*)' (K^-1 + W)^-1 (K^-1 k*)   (W singular: never inverted).
 *   With Zb != NULL the same for the difference f(Zb_i) - f(Z_i), and prob_i = Phi(mean_i / sqrt(2 sigma^2 + var_i)):
 *   the probability that Zb_i is preferred to Z_i (the likelihood of GPpref.py:56-66 under the posterior). */
int gpb_pref_evidence(gpb_handle* h, double* evidence);
/* gpb_pref_evidence_grad: the same evidence and its exact gradient, grad[d + 2] = d evidence / d [log l_1 .. log l_d,
 *   log sf, log sigma] (the loghyp layout of GPpref.py:99,113-115; sf2 = khyp[d]), with the jitter the fit chose held
 *   fixed.  Exact at a stationary point of sum log Phi - f'K^-1 f / 2, so the state must come from grad_mode = 1 (error
 *   otherwise); an error too when K^-1 + W is not positive definite at the mode.  Costs about 2.7 n^3 flop on the DMMA
 *   kernels (DESIGN.md section 4.3).  The state stays usable; the factor of K^-1 + W is overwritten, so the next
 *   gpb_pref_evidence / gpb_pref_predict factors it again (same results). */
int gpb_pref_evidence_grad(gpb_handle* h, double* evidence, double* grad);
int gpb_pref_predict(gpb_handle* h, const double* Z, const double* Zb, int64_t mz, double* mean, double* var,
                     double* prob);
/* PrefProbit.log_marginal (GPpref.py:90-94) for caller-supplied f (n), iK (n x n, host) and logdetK:
 * sum log Phi(z) - f' iK f / 2 - logdetK / 2 - n/2 log(2 pi), reduced on the device. */
int gpb_pref_log_marginal(gpb_handle* h, const int64_t* uvi, const double* y, int64_t P, int64_t n, const double* f,
                          const double* iK, double logdetK, double sigma, double* out);
/* PrefProbit.derivatives (GPpref.py:68-88) on its own: dense W (n x n) and gradient (n). */
int gpb_pref_derivatives(gpb_handle* h, const int64_t* uvi, const double* y, int64_t P, int64_t n,
                         const double* f, double sigma, int32_t grad_mode, double* W_out, double* g_out);

/* ---- micro-benchmarks used by bench.py / tools to fix the roofline denominators ---------- */
/* kind 0: DMMA.8x8x4 issue rate, 1: DFMA rate; returns TFLOP/s */
int gpb_microbench(gpb_handle* h, int32_t kind, double* tflops);

#ifdef __cplusplus
}
#endif
#endif /* GPB200_H */

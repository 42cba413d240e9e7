/* mfgp_b200 -- C ABI of the B200-native multi-fidelity GP hot path.
 *
 * The reference (MartinKlapacz/multifidelity-datafusion-GPs) has no FFI: its hot path is the
 * Python object protocol of GPy.models.GPRegression, reached from
 *   src/MFDataFusion.py:93-100   (construction = inference, then AbstractMFGP.ARD)
 *   src/abstractMFGP.py:131-137  (optimize / optimize_restarts -> one LML+gradient per step)
 *   src/MFDataFusion.py:153-156  (augment, then hf_model.predict)
 *   src/abstractMFGP.py:100-104  (low-fidelity GP and its mean predictor f_low)
 *   src/abstractMFGP.py:124-129  (acquisition: argmax of the predictive variance)
 * Each entry point below names the reference call it replaces.  The host side that binds them
 * (ctypes) is multifidelity_datafusion_gps_b200/_ffi.py; INTEGRATION.md shows the binding a
 * reference maintainer would add.
 *
 * Conventions
 *  - All arithmetic is FP64, indices are int64.  Matrices are row-major.
 *  - Pointers named d_* are DEVICE pointers owned by the caller (torch tensors' data_ptr());
 *    pointers named h_* are HOST pointers.  The library owns only the opaque handle, which holds
 *    a fixed-size scratch allocated in mfgp_create -- no allocation happens in any other call.
 *  - Every call enqueues on the handle's stream (mfgp_set_stream).  Calls with h_* outputs
 *    synchronise that stream before returning; all other calls are asynchronous.
 *  - Return value: 0 ok; >0 LAPACK-style info (1-based index of the first non-positive pivot of
 *    the Cholesky factorisation) so the host can replay GPy's jitter schedule; <0 bad argument or
 *    CUDA failure (message via mfgp_last_error).  There is no CPU fallback.
 *  - "Npad" = mfgp_padded_n(N): N rounded up to a multiple of 128.  Factor buffers are
 *    Npad x Npad with leading dimension Npad; the pad block is the identity.
 *  - theta (HOST, P doubles):  kind=MFGP_KIND_COMPOSITE, P=7:
 *        [var1, len1 | var2, len2 | var3, len3 | noise]   K = k1(z,z')k2(x,x') + k3(x,x')
 *    kind=MFGP_KIND_RBF, P=3: [var, len | noise].   x = first d columns, z = columns d..D-1.
 */
#ifndef MFGP_B200_H
#define MFGP_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MFGP_KIND_RBF 0        /* GPy.kern.RBF(D)          src/abstractMFGP.py:59-60 */
#define MFGP_KIND_COMPOSITE 1  /* RBF(z)*RBF(x) + RBF(x)   src/abstractMFGP.py:62-80 */

#define MFGP_UPLO_LOWER 0
#define MFGP_UPLO_FULL 1

#define MFGP_MAX_D 32          /* augmented input width d + E */
#define MFGP_MAX_E 16

typedef struct mfgp_ctx* mfgp_handle_t;

/* One fitted GP level: what GPy keeps in GPRegression after inference (X, kernel parameters,
 * posterior woodbury_vector = alpha, woodbury_chol = L; we keep W = L^-1 instead of L). */
typedef struct {
  int32_t kind;          /* MFGP_KIND_* */
  int32_t N;             /* training points */
  int32_t D;             /* columns of X */
  int32_t d;             /* leading columns that are the plain inputs x */
  int32_t P;             /* len(theta) */
  int32_t reserved;
  const double* d_X;     /* (N, D) row-major */
  const double* h_theta; /* HOST (P,) */
  const double* d_W;     /* (Npad, Npad) lower-triangular L^-1, ld = Npad; may be NULL for mean-only use */
  const double* d_alpha; /* (Npad,)  K_y^-1 y, zero padded */
} mfgp_level_t;

int mfgp_version(void);
int mfgp_padded_n(int N);

int mfgp_create(int device, mfgp_handle_t* out);
int mfgp_destroy(mfgp_handle_t h);
int mfgp_set_stream(mfgp_handle_t h, void* cuda_stream);
const char* mfgp_last_error(mfgp_handle_t h);
/* number of kernels this handle has launched since creation (bench.py's gpu_launches) */
long long mfgp_launch_count(mfgp_handle_t h);

/* Per-kernel-class timing for bench.py's roofline: when enabled, launches are bracketed by CUDA
 * event pairs on the handle's stream (first 512 launches per class).  mfgp_profile_read synchronises
 * and returns, per class, the average launch duration in ms (h_ms[10]) and the launch count
 * (h_count[10]); classes: 0 assemble, 1 potrf leaf, 2 gemm (potrf/trtri), 3 solve, 4 lauum,
 * 5 grad_reduce, 6 cross-covariance, 7 trmm+sumsq, 8 misc, 9 argmax (acquisition: the arg-max, the batch
 * acquisition's fused update and arg-max stage, and the ALC reduction). */
int mfgp_profile_enable(mfgp_handle_t h, int on);
int mfgp_profile_read(mfgp_handle_t h, double* h_ms, long long* h_count);

/* K1 -- covariance assembly.  Replaces kern.K(X) + diag.add(Ky, noise + 1e-8)
 * (GPy exact_gaussian_inference.py, reached from src/MFDataFusion.py:93-98).
 * Writes K_y = K + (noise + 1e-8 + jitter) I into d_K (N x N, leading dimension ldk);
 * uplo=LOWER writes the lower triangle including the diagonal only. */
int mfgp_assemble(mfgp_handle_t h, int kind, const double* d_X, int N, int D, int d,
                  const double* h_theta, int P, double jitter, double* d_K, long long ldk, int uplo);

/* K2+K3 -- factorise and solve.  Replaces pdinv(Ky) / dpotrs (GPy exact_gaussian_inference.py)
 * as run by GPRegression construction (src/MFDataFusion.py:93-98, src/abstractMFGP.py:100-102).
 * d_A, d_W: (Npad, Npad) caller buffers; on return d_A holds L (lower; upper triangle undefined),
 * d_W holds L^-1, d_alpha (Npad) holds K_y^-1 y.  h_out[0..2] = {LML, logdet, y^T alpha}. */
int mfgp_factorize(mfgp_handle_t h, int kind, const double* d_X, const double* d_y, int N, int D,
                   int d, const double* h_theta, int P, double jitter, double* d_A, double* d_W,
                   double* d_alpha, double* h_out);

/* K1..K5 -- one log-marginal-likelihood + gradient evaluation at fixed theta: the objective
 * paramz evaluates once per L-BFGS-B step (src/abstractMFGP.py:134,137).
 * On return d_A holds K_y^-1 (lower triangle), d_W holds L^-1, d_alpha holds alpha.
 * h_lml[0] = LML; h_grad[0..P-1] = dLML/dtheta (untransformed, ordered as theta). */
int mfgp_lml_grad(mfgp_handle_t h, int kind, const double* d_X, const double* d_y, int N, int D,
                  int d, const double* h_theta, int P, double jitter, double* d_A, double* d_W,
                  double* d_alpha, double* h_lml, double* h_grad);

/* Same evaluation with per-stage CUDA-event timings (ms) for bench.py / the roofline report:
 * h_ms[0..5] = {assemble, potrf, trtri, solve(alpha), K^-1 = W^T W, grad_reduce}. */
int mfgp_lml_grad_timed(mfgp_handle_t h, int kind, const double* d_X, const double* d_y, int N,
                        int D, int d, const double* h_theta, int P, double jitter, double* d_A,
                        double* d_W, double* d_alpha, double* h_lml, double* h_grad, double* h_ms);

/* Batched objective at the reference's own problem sizes (N <= 128: 5-30 high-fidelity points refitted by
 * 1 + 6 L-BFGS-B runs per adaptation step, src/abstractMFGP.py:131-137, src/gpc/mfgp_gpc.py:17-20).
 * B hyper-parameter vectors (h_thetas: HOST (B, P)) are evaluated by ONE launch, one CTA each, on the same
 * training data; only scalars come back -- no factor is written.  This is what lets the independent restarts
 * of optimize_restarts (src/abstractMFGP.py:137) run in lock-step on one GPU.
 * h_lml (B); h_grad (B, P) or NULL (no gradient); h_info (B): 0, or the 1-based first non-positive pivot of
 * that vector's factorisation (the caller replays GPy's jitter schedule for it).  Returns 0 or <0. */
int mfgp_lml_grad_batch_max(void);   /* vectors per launch (larger B is processed in slices) */
int mfgp_lml_grad_batch(mfgp_handle_t h, int kind, const double* d_X, const double* d_y, int N, int D, int d,
                        const double* h_thetas, int P, int B, double jitter, double* h_lml, double* h_grad,
                        int* h_info);

/* Bordered update at FIXED theta (SURVEY.md section 8f rank 3): one training point appended, as the
 * adaptation loop does once per step (src/abstractMFGP.py:320,354), in O(N^2) instead of refactorising:
 *   l = W k, L[N] = [l, l_nn], l_nn = sqrt(K(a,a) + noise + 1e-8 + jitter - |l|^2),
 *   W[N] = [-(W^T l)/l_nn, 1/l_nn], alpha = W^T (W y).
 * d_X (N+1, D) and d_y (N+1): the new point is row N; N is the OLD count.  d_A, d_W, d_alpha are sized
 * for the N+1 points, Npad' = mfgp_padded_n(N+1): when N is a multiple of 128 the caller first moves
 * the factors into buffers one 128-tile larger (identity on the new pad diagonal, zeros elsewhere).
 * d_W must hold L^-1 of the N points; a_holds_L != 0 iff d_A holds L (after mfgp_factorize; after mfgp_lml_grad it holds K^-1): row N
 * of L is then written and h_out[0..1] = {LML, logdet} of the N+1 points, else they are NaN.
 * h_out[2] = y^T alpha, h_out[3] = l_nn.  Returns N+1 if the new pivot is not positive. */
int mfgp_append_point(mfgp_handle_t h, int kind, const double* d_X, const double* d_y, int N, int D,
                      int d, const double* h_theta, int P, double jitter, double* d_A, double* d_W,
                      double* d_alpha, int a_holds_L, double* h_out);

/* Building blocks exposed for the parity tests (LAPACK names, lower, row-major, n multiple of 128). */
int mfgp_potrf(mfgp_handle_t h, double* d_A, double* d_W, int npad);   /* A -> L; W diag blocks -> leaf inverses */
int mfgp_trtri(mfgp_handle_t h, const double* d_L, double* d_W, int npad); /* completes W = L^-1 (after mfgp_potrf) */
int mfgp_lauum(mfgp_handle_t h, const double* d_W, double* d_Kinv, int npad); /* Kinv(lower) = W^T W */

/* K6 -- prediction.  Replaces GP.predict -> Posterior._raw_predict (src/MFDataFusion.py:156,
 * src/abstractMFGP.py:104): mean = Kx^T alpha; var = max(Kxx - |W Kx|^2, 1e-15) (+ noise).
 * d_Xnew: (M, D).  d_var may be NULL (mean only, no W needed).  d_ws/ws_bytes: caller scratch for
 * the cross-covariance chunk, at least mfgp_predict_ws_bytes(N, 128). */
size_t mfgp_predict_ws_bytes(int N, long long cols);
int mfgp_predict(mfgp_handle_t h, const mfgp_level_t* gp, const double* d_Xnew, long long M,
                 double* d_mean, double* d_var, int include_noise, double* d_ws, size_t ws_bytes);

/* K6d -- predictive gradients.  Replaces GPy's GP.predictive_gradients [GPy-recall]: for the query rows q_c of d_Xnew
 * (M, D), dmean[c][j] = d mu(q_c) / d q_j = sum_k alpha_k dk(q_c, X_k)/dq_j and dvar[c][j] = d var / d q_j =
 * -2 sum_k u_kc dk(q_c, X_k)/dq_j with u_c = K_y^-1 k_c (k(q, q) is constant for both kernels).  dvar is the
 * derivative of the UNCLIPPED latent variance; the noise is a constant.  Both (M, D) row-major.
 * By-products (optional, NULL to skip): d_mean and d_var are mfgp_predict's outputs (var clipped at 1e-15, plus the
 * noise if include_noise), equal to them to round-off (other summation orders), so that an optimiser gets f and g
 * from one call.  d_dvar == NULL: mean-only mode -- no W, no scratch (d_ws may be NULL), d_var must be NULL.
 * Otherwise d_ws holds W^T and the per-chunk blocks: at least mfgp_predictive_gradients_ws_bytes(N, 128); chunks
 * are sized from ws_bytes.  A query's outputs do not depend on the chunk size or on the other queries of the call.
 * Asynchronous on the handle's stream, like mfgp_predict. */
size_t mfgp_predictive_gradients_ws_bytes(int N, long long cols);
int mfgp_predictive_gradients(mfgp_handle_t h, const mfgp_level_t* gp, const double* d_Xnew, long long M,
                              double* d_dmean /* (M, D) */, double* d_dvar /* (M, D) or NULL */,
                              double* d_mean /* (M) or NULL */, double* d_var /* (M) or NULL */,
                              int include_noise, double* d_ws, size_t ws_bytes);

/* K6, latency path: M <= mfgp_predict_small_max_rows() query rows given in HOST memory, results to HOST memory,
 * one or two launches and ONE synchronisation (query rows and results travel through pinned host memory
 * mapped into the device).  This is what a single objective evaluation of the reference's default acquisition
 * costs: scipydirect calls model_predict(x[None]) up to 20 000 times in sequence
 * (src/adaptation_maximizers/scipydirect_wrapper.py:22-26), each an __augment_Data + hf_model.predict
 * (src/MFDataFusion.py:153-156).  hf->N <= 2048.  lf == NULL: h_X holds augmented rows (M, hf->D).
 * lf != NULL (data-driven low fidelity): h_X holds plain inputs (M, lf->D) and the rows are augmented with
 * the LF posterior mean at x + o_e tau first (h_offsets: HOST (E, lf->D), hf->D == lf->D + E).
 * Same formulas as mfgp_predict; the summation orders differ, so results agree to round-off, not bit for bit. */
int mfgp_predict_small_max_rows(void);
int mfgp_predict_small(mfgp_handle_t h, const mfgp_level_t* hf, const mfgp_level_t* lf, const double* h_X,
                       int M, const double* h_offsets, int E, double tau, int include_noise, double* h_mean,
                       double* h_var);

/* K6, resident form of the latency path ("point service").  The reference's default acquisition asks for up to
 * 20 000 single-point predicts in sequence, each answer deciding the next question
 * (src/adaptation_maximizers/scipydirect_wrapper.py:22-26 -> src/MFDataFusion.py:153-156).  _start puts ONE CTA
 * on the device that stays resident and answers questions posted through mapped pinned host memory; _eval posts
 * one row (lf != NULL at _start: plain inputs (lf->D); lf == NULL: an augmented row (hf->D)) and spins on the
 * answer (h_out[0] = mean, h_out[1] = variance; bit-identical to mfgp_predict_small); _stop releases the SM.
 * No launch and no stream synchronisation per question.  The kernel leaves by itself after idle_ms (<= 0: 20 ms)
 * without a question and is relaunched transparently by the next _eval (_relaunches counts these).  The factors
 * of hf / lf must not change between _start and _stop.  One service per handle; _eval is not re-entrant. */
int mfgp_point_service_start(mfgp_handle_t h, const mfgp_level_t* hf, const mfgp_level_t* lf,
                             const double* h_offsets, int E, double tau, int include_noise, double idle_ms);
int mfgp_point_service_eval(mfgp_handle_t h, const double* h_x, double* h_out);
int mfgp_point_service_stop(mfgp_handle_t h);
long long mfgp_point_service_relaunches(mfgp_handle_t h);

/* A1 with a data-driven low-fidelity level.  Replaces __augment_Data (src/MFDataFusion.py:177-208)
 * when f_low is lf_model.predict(.)[0] (src/abstractMFGP.py:104):
 * Xaug[i] = [x_i, mu_l(x_i + o_0 tau), ..., mu_l(x_i + o_{E-1} tau)].  h_offsets: HOST (E, d). */
int mfgp_augment(mfgp_handle_t h, const mfgp_level_t* lf, const double* d_X, long long M,
                 const double* h_offsets, int E, double tau, double* d_Xaug, double* d_ws,
                 size_t ws_bytes);

/* K7 -- Monte-Carlo propagation of the low-fidelity posterior (extension; README.md:13).
 * For every test point m (global index m0 + m) and sample s: z = mu_l + sd_l * eps,
 * (mu_s, v_s) = HF predict at [x, z]; mean = mean_s mu_s; var = mean_s v_s + var_s(mu_s).
 * d_eps: (M, S) standard normals, or NULL -> Philox4x32-10 keyed by seed, counter = (m0+m)*S+s.
 * d_weights: optional (M,) quadrature weights; h_wsum[0] += sum_m w_m mean_m (PCE mean).
 * E = 1 (NARGP: offsets = {0}) only; mfgp_predict_mc_delays handles E > 1. */
/* Recommended scratch for mfgp_predict_mc / mfgp_predict_mc_chain.  N_up = the largest training-set size among
 * the upper levels.  Upper levels with N <= 64 -- the reference's own sizes, src/gpc/mfgp_gpc.py:10,18-20 -- run a
 * fused generator + contraction kernel that keeps no cross-covariance row, so the scratch then holds three
 * doubles per (point, sample) column and whole batches go through in one launch; otherwise a chunk is four
 * 128-column tiles per SM of (padded N_up + d + 4) doubles per column.  Results never depend on the size. */
size_t mfgp_predict_mc_ws_bytes(int N_l, int N_up, int d, long long M, int S);
int mfgp_predict_mc(mfgp_handle_t h, const mfgp_level_t* lf, const mfgp_level_t* hf,
                    const double* d_Xtest, long long M, int S, const double* d_eps,
                    unsigned long long seed, long long m0, int include_lf_noise,
                    int include_hf_noise, const double* d_weights, double* d_mean, double* d_var,
                    double* h_wsum, double* d_ws, size_t ws_bytes);

/* K7 through a chain of L >= 2 fidelity levels (recursive NARGP, README.md:13 / Perdikaris et al. 2017 eq. 2.9-2.10;
 * SURVEY.md section 8f rank 4): levels[0] is a GP on x (D = d), every levels[t >= 1] a GP on [x, z] (D = d + 1).
 *   z_1 = mu_0(x) + sd_0(x) eps_1;   (mu_t, v_t) = level t at [x, z_t];   z_{t+1} = mu_t + sqrt(v_t) eps_{t+1}
 * per sample, and mean = mean_s mu_{L-1,s}, var = mean_s v_{L-1,s} + var_s mu_{L-1,s}.  L = 2 is mfgp_predict_mc.
 * d_eps: (L-1, M, S) standard normals or NULL -> Philox4x32-10, key seed + (j-1) * 0x9E3779B97F4A7C15 for the j-th
 * sampling, counter (m0+m)*S+s (so j = 1 draws what mfgp_predict_mc draws).  include_lower_noise: the sampled
 * variances v_t (t < L-1) include that level's noise variance; include_top_noise: the returned one does. */
int mfgp_predict_mc_chain(mfgp_handle_t h, const mfgp_level_t* const* levels, int L, const double* d_Xtest,
                          long long M, int S, const double* d_eps, unsigned long long seed, long long m0,
                          int include_lower_noise, int include_top_noise, const double* d_weights,
                          double* d_mean, double* d_var, double* h_wsum, double* d_ws, size_t ws_bytes);

/* K7 with the low-fidelity posterior sampled JOINTLY across the test points (SURVEY.md section 8f rank 4,
 * "full-covariance LF sampling for small M"; E = 1 models, M <= 16384):
 *   Sigma_l = K_l(X*, X*) - (W_l K_l*)^T (W_l K_l*) + ((include_lf_noise ? noise_l : 0) + lf_jitter) I   (M x M),
 *   z_s = mu_l + chol(Sigma_l) eps_s,   eps: d_eps (M, S) or NULL -> Philox counter m*S+s,
 * so that every sample s is one coherent low-fidelity function; mean / var aggregate as in mfgp_predict_mc
 * (their expectation is the same -- they only depend on the marginals), and d_path_wsum (S, DEVICE, may be
 * NULL) receives the per-path functional sum_m w_m mu_s(x_m): the distribution of the PCE mean over
 * low-fidelity function draws.  Returns >0 (1-based pivot) if Sigma_l is not positive definite: raise lf_jitter.
 * Not sharded: all M points belong to one covariance.  Scratch: mfgp_predict_mc_joint_ws_bytes. */
size_t mfgp_predict_mc_joint_ws_bytes(int N_l, int N_h, long long M, int S);
int mfgp_predict_mc_joint(mfgp_handle_t h, const mfgp_level_t* lf, const mfgp_level_t* hf,
                          const double* d_Xtest, long long M, int S, const double* d_eps,
                          unsigned long long seed, int include_lf_noise, int include_hf_noise,
                          double lf_jitter, const double* d_weights, double* d_mean, double* d_var,
                          double* d_path_wsum, double* d_ws, size_t ws_bytes);

/* K7 for models with delays (GPDF / GPDFC: E = n*d + 1 augmented columns, 1 <= E <= 8).  The
 * low-fidelity posterior at the E locations x + o_e tau of a test point is JOINT: mu_l in R^E,
 * Sigma_l = k(a,a') - (W k_a).(W k_a') in R^(E x E) (+ (noise + lf_jitter) I), z_s = mu_l + chol(Sigma_l) eps_s,
 * then (mu_s, v_s) = HF predict at [x, z_s] and the same aggregation as mfgp_predict_mc.
 * h_offsets: HOST (E, d) iterator offsets (src/augm_iterators/backward_augm_iterator.py:20-37).
 * d_eps: (M, S, E) standard normals, or NULL -> Philox counter ((m0+m)*S + s)*E + e.
 * Returns >0: 1-based global index of the first test point whose Sigma_l is not positive definite
 * (raise lf_jitter, as np.linalg.cholesky would raise LinAlgError in the NumPy restatement). */
int mfgp_predict_mc_delays(mfgp_handle_t h, const mfgp_level_t* lf, const mfgp_level_t* hf,
                           const double* d_Xtest, long long M, const double* h_offsets, int E,
                           double tau, int S, const double* d_eps, unsigned long long seed,
                           long long m0, int include_lf_noise, int include_hf_noise, double lf_jitter,
                           const double* d_weights, double* d_mean, double* d_var, double* h_wsum,
                           double* d_ws, size_t ws_bytes);

/* the eps the in-kernel generator uses, for the parity tests: out[i] = N(0,1) of counter first+i */
int mfgp_fill_normal(mfgp_handle_t h, unsigned long long seed, long long first, long long count,
                     double* d_out);

/* K8 -- acquisition.  Replaces AbstractMaximizer.maximize's objective scan
 * (src/adaptation_maximizers/scipydirect_wrapper.py:22-26) by a candidate-set argmax:
 * h_val[0] = max_i v[i], h_idx[0] = lowest i attaining it (np.argmax semantics). */
int mfgp_argmax(mfgp_handle_t h, const double* d_v, long long C, double* h_val, long long* h_idx);

/* K8b -- greedy batch acquisition: q high-fidelity points per adaptation step instead of one
 * (src/abstractMFGP.py:317-359 acquires one per step and refits).  At fixed theta the predictive variance does not
 * depend on the targets, so the q points that q sequential steps (arg-max, append at fixed theta) would pick are a
 * pivoted partial Cholesky of the posterior covariance over the candidate set:
 *   v_0(c) = k(c, c) - |W k_c|^2 (unclipped),  s^2 = noise + 1e-8 + jitter (the diagonal mfgp_append_point adds),
 *   pick p_i = argmax_c max(v_i(c), 1e-15) (+ noise), lowest index on ties,
 *   R[i][c] = (k(c, a_i) - k_c^T K_y^-1 k(X, a_i) - sum_{l<i} R[l][c] R[l][p_i]) / sqrt(v_i(p_i) + s^2),
 *   v_{i+1}(c) = v_i(c) - R[i][c]^2,   a_i = d_cands[p_i] (augmented row).
 * Step-wise protocol, so that the same calls serve one GPU and candidates sharded over ranks:
 *   _begin computes v_0 (the pass mfgp_predict makes) and returns the LOCAL winner of pick 0;
 *   _step(i) conditions on pick i, given by its record h_rec_in (the GLOBAL winner's; on one GPU the record the
 *   previous call returned), and returns the local winner of pick i + 1.
 * Record (1 + D + q doubles): [v_i(p) unclipped, a (D values), R[0..i)[p], zeros].  h_val[0] = the winner's reported
 * variance max(v, 1e-15) (+ noise), h_idx[0] = its index in [0, C).  One synchronisation per call.
 * 1 <= q <= MFGP_ACQ_MAX_Q, C >= 1, 0 <= i < q.  jitter: the level's factorisation jitter.  d_ws (at least
 * mfgp_acq_batch_ws_bytes(N, C, q), of which the part beyond the fixed regions holds the prediction chunk) carries
 * state from call to call and must not be touched between the calls of one batch.
 * _step returns i + 1 (LAPACK-style) if v_i(p_i) + s^2 <= 0. */
#define MFGP_ACQ_MAX_Q 64
size_t mfgp_acq_batch_ws_bytes(int N, long long C, int q);
int mfgp_acq_batch_begin(mfgp_handle_t h, const mfgp_level_t* gp, const double* d_cands, long long C, int q,
                         int include_noise, double* d_ws, size_t ws_bytes, double* h_val, long long* h_idx,
                         double* h_rec);
int mfgp_acq_batch_step(mfgp_handle_t h, const mfgp_level_t* gp, const double* d_cands, long long C, int q,
                        int include_noise, double jitter, int i, const double* h_rec_in, double* d_ws,
                        size_t ws_bytes, double* h_val, long long* h_idx, double* h_rec);

/* K8c -- integrated-variance (ALC, "active learning Cohn") acquisition: how much acquiring candidate c lowers the
 * weighted latent predictive variance over a reference set, at the level's current theta.  With
 * Tt[x][i] = sum_{k<=i} k(x, X_k) W[i][k] for candidates c and references r (augmented rows, D columns):
 *   k_n(c, r) = k(c, r) - sum_i Tt[c][i] Tt[r][i],   v_n(c) = k(c, c) - sum_i Tt[c][i]^2 (unclipped),
 *   s^2 = noise + 1e-8 + jitter (the diagonal mfgp_append_point adds),
 *   d_alc[c] = sum_r w_r k_n(c, r)^2 / (v_n(c) + s^2),  -inf where v_n(c) + s^2 <= 0.
 * In exact arithmetic d_alc[c] = sum_r w_r (v_n(r) - v_{n+c}(r)) with v_{n+c} the latent variance after appending
 * c at the same theta.  d_w (R) holds w_r >= 0, or NULL for w_r = 1/R; d_cands (C, D), d_ref (R, D), d_alc (C):
 * DEVICE.  C >= 1, R >= 1; jitter: the level's factorisation jitter.  d_ws holds K(ref, X) and Tt_R plus per
 * candidate chunk K(cands, X), Tt_C and G = Tt_C Tt_R^T: at least the fixed part plus one 128-column chunk
 * (mfgp_alc_ws_bytes(N, 1, R)); chunks are sized from ws_bytes.  A candidate's value depends on nothing but the
 * candidate, the reference set and the level: not on the chunk size or the other candidates of the call.
 * Asynchronous on the handle's stream, like mfgp_predict; the arg-max is mfgp_argmax on d_alc.
 * mfgp_alc_ws_bytes: the scratch for C candidates (chunk capped at 1 GiB), 0 for invalid arguments. */
size_t mfgp_alc_ws_bytes(int N, long long C, long long R);
int mfgp_alc(mfgp_handle_t h, const mfgp_level_t* gp, const double* d_cands, long long C, const double* d_ref,
             long long R, const double* d_w, double jitter, double* d_alc, double* d_ws, size_t ws_bytes);

/* K9 -- polynomial-chaos projection on a quadrature grid (SURVEY.md section 8f rank 2).  Replaces
 * cp.fit_quadrature / cp.E / cp.Var as src/gpc/chaospy_wrapper.py:18-29 uses them, for independent
 * uniform inputs on the box [lb, ub] (tests/test_mfgp_adapt_4d.py:40) and the orthonormal Legendre basis:
 *   coeff[k] = sum_q w_q f_q prod_i sqrt(2 k_i + 1) P_{k_i}(2 (x_qi - lb_i)/(ub_i - lb_i) - 1)
 * so that mean = coeff[0] (the all-zero multi-index first) and variance = sum_{k>0} coeff[k]^2.
 * d_nodes (Q, d), d_weights (Q) (summing to 1), d_values (Q): DEVICE.  h_multi_index: HOST (P, d)
 * int32 degrees, each <= max_degree; P <= 4096.  d_coeff (P) DEVICE; h_coeff (P) HOST or NULL (when
 * given the call synchronises).  d_ws / ws_bytes: scratch of at least mfgp_pce_ws_bytes(d, P). */
size_t mfgp_pce_ws_bytes(int d, int P);
int mfgp_pce_project(mfgp_handle_t h, const double* d_nodes, const double* h_lb, const double* h_ub,
                     int d, const double* d_weights, const double* d_values, long long Q,
                     const int* h_multi_index, int P, int max_degree, double* d_coeff,
                     double* h_coeff, double* d_ws, size_t ws_bytes);

#ifdef __cplusplus
}
#endif
#endif /* MFGP_B200_H */

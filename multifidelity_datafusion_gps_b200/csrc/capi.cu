// extern "C" entry points declared in include/mfgp_b200.h: argument checks, scratch layout,
// chunk loops and stream ordering.  No torch types, no allocation outside mfgp_create.
#include <time.h>
#include "common.cuh"

// launchers defined in predict.cu
int solve_alpha_launch(mfgp_ctx* h, const double* L, const double* W, int npad, int N,
                       const double* y, double* v_tmp, double* alpha, double* d_out3, int ldl);
int cross_gen_launch(mfgp_ctx* h, const KParams& kp, const double* X, int N, int npad,
                     const double* alpha, const double* Xq, long long ncols, long long cols_pad,
                     double* Ks, double* mean);
int finish_var_launch(mfgp_ctx* h, const double* ss, long long n, double kdiag, double noise_add,
                      double* var, bool latent = false);
int acq_partials_doubles();
int kinv_apply_launch(mfgp_ctx* h, const double* W, int npad, int N, const double* k, double* l_tmp, double* u);
int acq_coef_launch(mfgp_ctx* h, const double* u, int N, int npad1, double* coef);
int acq_update_launch(mfgp_ctx* h, const double* kg, double* R, long long C, int i, const double* rp, double rho,
                      double* v, double noise_add, double* partials, double* best);
int acq_gather_launch(mfgp_ctx* h, const double* best, const double* v, const double* cands, int D,
                      const double* R, long long C, int nr, int q, double* out);
int build_locs_launch(mfgp_ctx* h, const double* X, long long rows, int d, const double* d_offs,
                      int E, double tau, double* out);
int concat_aug_launch(mfgp_ctx* h, const double* X, const double* vals, long long rows, int d, int E,
                      double* out);
int fill_normal_launch(mfgp_ctx* h, unsigned long long seed, long long first, long long count,
                       double* out);
int build_mc_rows_launch(mfgp_ctx* h, const double* Xtest, const double* mu_l, const double* sd_l,
                         const double* eps, unsigned long long seed, long long m_global0,
                         long long m_lo, long long ncols, int S, int d, double* out);
int cross_gen_mc_launch(mfgp_ctx* h, const KParams& kp, const double* X, int N, int npad,
                        const double* alpha, const double* Xtest, const double* mu_l,
                        const double* sd_l, const double* eps, unsigned long long seed,
                        long long m_global0, long long m_lo, long long npts, int S,
                        long long cols_pad, double* Ks, double* mu_c, const double* zcol, long long z_off,
                        long long ldz);
int sample_cols_launch(mfgp_ctx* h, const double* mu_c, const double* v_c, const double* eps,
                       unsigned long long key, long long m_global0, long long m_lo, long long ncols, int S,
                       double* z);
int fill_normal_padded_launch(mfgp_ctx* h, const double* eps, unsigned long long seed, long long M, int S,
                              long long rows, long long ldE, double* E);
int path_wsum_launch(mfgp_ctx* h, const double* mu_c, const double* w, long long m_lo, long long npts, int S,
                     double* path);
int append_point_launch(mfgp_ctx* h, const double* k, int N, int npad, double kaa, double* A, double* W,
                        int write_L, double* l_tmp, double* t_tmp, double* d_out2);
int mc_max_samples();
int predict_configure(mfgp_ctx* h);
int sqrt_launch(mfgp_ctx* h, double* v, long long n);
int mc_small_applies(int N);
int mc_small_launch(mfgp_ctx* h, const KParams& kp, const double* X, int N, int npad, const double* W,
                    const double* alpha, const double* Xtest, const double* mu_l, const double* sd_l,
                    const double* eps, unsigned long long seed, long long m_global0, long long m_lo,
                    long long npts, int S, double* mu_c, double* ss, const double* zcol, long long z_off,
                    long long ldz, int* took);
int mc_aggregate_launch(mfgp_ctx* h, const double* mu_c, const double* v_c, long long npts, int S,
                        double* mean, double* var);
int argmax_launch(mfgp_ctx* h, const double* v, long long n, double* d_val, long long* d_idx);
int group_gram_launch(mfgp_ctx* h, const double* T, int npad, long long ldt, long long npts, int E, double* G);
int joint_chol_launch(mfgp_ctx* h, const double* G, const double* d_kab, long long npts, int E,
                      double diag_add, long long p_global0, double* Lc);
int build_mc_rows_joint_launch(mfgp_ctx* h, const double* Xtest, const double* mu_l, const double* Lc,
                               const double* eps, unsigned long long seed, long long m_global0,
                               long long m_lo, long long ncols, int S, int d, int E, double* out);
int wdot_launch(mfgp_ctx* h, const double* w, const double* x, long long n, double* d_out);
int predict_small_max_n();
int point_service_launch(mfgp_ctx* h, const PointServiceArgs& a, PointServiceCtl* d_ctl, cudaStream_t stream);
int predict_small_launch(mfgp_ctx* h, const KParams& kh, const mfgp_level_t* hf, const KParams* kl,
                         const mfgp_level_t* lf, const double* Xq, int M, const double* d_offs, int E, double tau,
                         double* Xaug_tmp, double noise_add, double* out);

#define JITTER_CONST 1e-8   // GPy exact_gaussian_inference.py: diag.add(Ky, variance + 1e-8)
#define MFGP_SMALL 4096

static char g_err[256] = "invalid handle";

// Every entry point runs on the handle's device and leaves the caller's current device as it found it
// (torch's current device must not change under the caller).
struct DeviceGuard {
  int prev, dev;
  bool restore;
  explicit DeviceGuard(int d) : prev(-1), dev(d), restore(false) {
    if (cudaGetDevice(&prev) == cudaSuccess && prev != dev) restore = true;
    if (prev != dev) cudaSetDevice(dev);
  }
  ~DeviceGuard() {
    if (restore) cudaSetDevice(prev);
  }
};
#define ENTER(h)        \
  if (!(h)) return -1;  \
  DeviceGuard _device_guard((h)->device)

// -1 / (2 len^2), kept finite.  The optimiser's line search visits lengthscales down to the denormals
// (L-BFGS-B's first long steps on the reference's 1-D curve evaluate len = 5.6e-309): GPy then gets r = dist/len
// -> huge, exp(-r^2/2) -> 0 off the diagonal and K = variance * I, a perfectly valid (if useless) model whose
// finite LML steers the search back.  With an infinite coefficient the diagonal would be 0 * inf = NaN here and
// the evaluation would be reported as infeasible, which sends the optimiser somewhere else.  A coefficient of
// -1e300 gives exactly GPy's matrix: 0 on coincident points, underflow (< 4.5e-308) everywhere else.
static double inv_len2(double len) {
  const double a = -0.5 / (len * len);
  return a < -1e300 ? -1e300 : a;
}

// d/d len = S / len^3; below 1e-100 every off-diagonal covariance (and with it every term of S) has
// underflowed, and GPy's gradient is exactly 0 there (-r K G with K = 0) while S / len^3 would be 0 / 0
static double len_grad(double S, double len) { return len < 1e-100 ? 0.0 : S / (len * len * len); }

int make_kparams(mfgp_ctx* h, int kind, int D, int d, const double* theta, int P, KParams* kp) {
  ARG_CHECK(h, theta != nullptr);
  ARG_CHECK(h, D >= 1 && D <= MFGP_MAX_D && d >= 1 && d <= D);
  memset(kp, 0, sizeof(*kp));
  kp->kind = kind;
  kp->D = D;
  kp->d = d;
  if (kind == MFGP_KIND_COMPOSITE) {
    ARG_CHECK(h, P == 7 && d < D);
    for (int i = 0; i < 6; i++) ARG_CHECK(h, theta[i] > 0.0);
    kp->c12 = theta[0] * theta[2];
    kp->az = inv_len2(theta[1]);
    kp->ax = inv_len2(theta[3]);
    kp->s3 = theta[4];
    kp->a3 = inv_len2(theta[5]);
    kp->kdiag = theta[0] * theta[2] + theta[4];
  } else if (kind == MFGP_KIND_RBF) {
    ARG_CHECK(h, P == 3);
    ARG_CHECK(h, theta[0] > 0.0 && theta[1] > 0.0);
    kp->c12 = theta[0];
    kp->az = kp->ax = inv_len2(theta[1]);
    kp->s3 = 0.0;
    kp->a3 = 0.0;
    kp->kdiag = theta[0];
  } else {
    ARG_CHECK(h, kind == MFGP_KIND_RBF || kind == MFGP_KIND_COMPOSITE);
  }
  ARG_CHECK(h, theta[P - 1] >= 0.0);
  {  // exp2s() form (fastmath.cuh): coefficients in units of ln2/256, variances as additive logs
    const double U = 369.32993046757463;   // 256 / ln 2
    // The optimiser's line search visits absurd variances (softplus of a large negative number);
    // outside e^+-700 the log-variance is clamped: below, the term is < 1e-304 either way; above,
    // FP64 would overflow in GPy's form as well.
    double l12 = kind == MFGP_KIND_COMPOSITE ? log(theta[0]) + log(theta[2]) : log(theta[0]);
    double l3 = kp->s3 > 0.0 ? log(kp->s3) : 0.0;
    l12 = fmin(fmax(l12, -700.0), 700.0);
    l3 = fmin(fmax(l3, -700.0), 700.0);
    kp->uz = kp->az * U;
    kp->ux = kp->ax * U;
    kp->u3 = kp->a3 * U;
    kp->lc12 = l12 * U;
    kp->ls3 = l3 * U;
    kp->exp_tbl = h->d_exp_tbl;
  }
  kp->noise = theta[P - 1];
  for (int i = 0; i < P; i++) kp->theta[i] = theta[i];
  return 0;
}

// Up to this size the single-CTA kernel beats the multi-kernel chain (wall time per LML+gradient evaluation:
// N = 8: 66 vs 92 us, N = 30: 78 vs 108 us, N = 100: 147 vs 144 us; tools/fit_time.py)
#define MFGP_SMALL_N 96

static int fetch_scalars(mfgp_ctx* h, int ndoubles) {
  CUDA_TRY(h, cudaMemcpyAsync(h->h_pinned, h->d_scalars, ndoubles * sizeof(double),
                              cudaMemcpyDeviceToHost, h->stream));
  CUDA_TRY(h, cudaMemcpyAsync(h->h_info, h->d_info, 4 * sizeof(int), cudaMemcpyDeviceToHost,
                              h->stream));
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  return 0;
}

extern "C" {

int mfgp_version(void) { return 100; }

int mfgp_padded_n(int N) { return round_up(N < 1 ? 1 : N, MFGP_TILE); }

int mfgp_create(int device, mfgp_handle_t* out) {
  if (!out) return -1;
  *out = nullptr;
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) {
    snprintf(g_err, sizeof(g_err), "mfgp_create: no CUDA device (this library has no CPU fallback)");
    return -2;
  }
  if (device < 0 || device >= count) {
    snprintf(g_err, sizeof(g_err), "mfgp_create: device %d out of range (%d devices)", device, count);
    return -1;
  }
  cudaDeviceProp prop;
  if (cudaSetDevice(device) != cudaSuccess || cudaGetDeviceProperties(&prop, device) != cudaSuccess) {
    snprintf(g_err, sizeof(g_err), "mfgp_create: cannot select device %d", device);
    return -2;
  }
  if (prop.major != 10) {
    snprintf(g_err, sizeof(g_err), "mfgp_create: device is sm_%d%d; this library is built for sm_100a only",
             prop.major, prop.minor);
    return -3;
  }
  mfgp_ctx* h = new mfgp_ctx();
  memset(h, 0, sizeof(*h));
  h->device = device;
  h->stream = 0;
  bool ok = cudaMalloc(&h->d_partials, MFGP_PARTIALS * sizeof(double)) == cudaSuccess &&
            cudaMalloc(&h->d_scalars, MFGP_SMALL * sizeof(double)) == cudaSuccess &&
            cudaMalloc(&h->d_info, 4 * sizeof(int)) == cudaSuccess &&
            cudaMalloc(&h->d_exp_tbl, 256 * sizeof(double)) == cudaSuccess &&
            cudaMallocHost(&h->h_pinned, 64 * sizeof(double)) == cudaSuccess &&
            cudaMallocHost(&h->h_info, 4 * sizeof(int)) == cudaSuccess &&
            cudaHostAlloc(&h->h_batch, 16 * 16 * sizeof(double), cudaHostAllocMapped) == cudaSuccess &&
            cudaHostAlloc(&h->h_batch_info, 16 * sizeof(int), cudaHostAllocMapped) == cudaSuccess &&
            cudaHostGetDevicePointer((void**)&h->d_batch, h->h_batch, 0) == cudaSuccess &&
            cudaHostGetDevicePointer((void**)&h->d_batch_info, h->h_batch_info, 0) == cudaSuccess;
  for (int i = 0; ok && i < 8; i++) ok = cudaEventCreate(&h->ev[i]) == cudaSuccess;
  for (int i = 0; ok && i < 3 * 64 + 4; i++)
    ok = cudaEventCreateWithFlags(&h->ev_la[i], cudaEventDisableTiming) == cudaSuccess;
  if (ok) {
    int pr_least = 0, pr_greatest = 0;
    ok = cudaDeviceGetStreamPriorityRange(&pr_least, &pr_greatest) == cudaSuccess &&
         cudaStreamCreateWithPriority(&h->s_hi, cudaStreamNonBlocking, pr_greatest) == cudaSuccess &&
         cudaStreamCreateWithPriority(&h->s_mid, cudaStreamNonBlocking, (pr_least + pr_greatest) / 2) == cudaSuccess &&
         cudaStreamCreateWithPriority(&h->s_svc, cudaStreamNonBlocking, pr_greatest) == cudaSuccess &&
         cudaHostAlloc(&h->svc_h, sizeof(PointServiceCtl), cudaHostAllocMapped) == cudaSuccess &&
         cudaHostGetDevicePointer((void**)&h->svc_d, h->svc_h, 0) == cudaSuccess;
    if (ok) memset(h->svc_h, 0, sizeof(PointServiceCtl));
  }
  if (ok) ok = cudaMemset(h->d_info, 0, 4 * sizeof(int)) == cudaSuccess;
  if (ok) {   // 2^(j/256) rounded from 64-bit-mantissa long double
    double tbl[256];
    for (int j = 0; j < 256; j++) tbl[j] = (double)exp2l((long double)j / 256.0L);
    ok = cudaMemcpy(h->d_exp_tbl, tbl, sizeof(tbl), cudaMemcpyHostToDevice) == cudaSuccess;
  }
  if (!ok || small_gp_configure(h) != 0 || small_batch_configure(h) != 0 || linalg_configure(h) != 0 || assemble_configure(h) != 0 || predict_configure(h) != 0) {
    snprintf(g_err, sizeof(g_err), "mfgp_create: scratch allocation / kernel configuration failed: %s",
             cudaGetErrorString(cudaGetLastError()));
    delete h;
    return -100;
  }
  *out = h;
  return 0;
}

int mfgp_destroy(mfgp_handle_t h) {
  ENTER(h);
  cudaFree(h->d_partials);
  cudaFree(h->d_scalars);
  cudaFree(h->d_info);
  cudaFree(h->d_exp_tbl);
  cudaFreeHost(h->h_pinned);
  cudaFreeHost(h->h_info);
  cudaFreeHost(h->h_batch);
  cudaFreeHost(h->h_batch_info);
  for (int i = 0; i < 8; i++) cudaEventDestroy(h->ev[i]);
  for (int i = 0; i < 3 * 64 + 4; i++) cudaEventDestroy(h->ev_la[i]);
  if (h->s_hi) cudaStreamDestroy(h->s_hi);
  if (h->s_mid) cudaStreamDestroy(h->s_mid);
  if (h->svc_active) {
    h->svc_h->stop = 1;
    cudaStreamSynchronize(h->s_svc);
  }
  if (h->s_svc) cudaStreamDestroy(h->s_svc);
  if (h->svc_h) cudaFreeHost(h->svc_h);
  if (h->prof_ev) {
    for (int i = 0; i < MFGP_PROF_CLASSES * MFGP_PROF_POOL * 2; i++) cudaEventDestroy(h->prof_ev[i]);
    delete[] h->prof_ev;
  }
  delete h;
  return 0;
}

int mfgp_set_stream(mfgp_handle_t h, void* cuda_stream) {
  ENTER(h);
  h->stream = (cudaStream_t)cuda_stream;
  return 0;
}

const char* mfgp_last_error(mfgp_handle_t h) { return h ? h->err : g_err; }

long long mfgp_launch_count(mfgp_handle_t h) { return h ? h->launches : -1; }

int mfgp_profile_enable(mfgp_handle_t h, int on) {
  ENTER(h);
  if (on && !h->prof_ev) {
    const int n = MFGP_PROF_CLASSES * MFGP_PROF_POOL * 2;
    h->prof_ev = new cudaEvent_t[n];
    for (int i = 0; i < n; i++) CUDA_TRY(h, cudaEventCreate(&h->prof_ev[i]));
  }
  h->prof_on = on ? 1 : 0;
  for (int i = 0; i < 16; i++) h->prof_count[i] = 0;
  return 0;
}

int mfgp_profile_read(mfgp_handle_t h, double* h_ms, long long* h_count) {
  ENTER(h);
  ARG_CHECK(h, h_ms && h_count);
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  for (int cls = 0; cls < MFGP_PROF_CLASSES; cls++) {
    double total = 0.0;
    long long n = h->prof_count[cls] < MFGP_PROF_POOL ? h->prof_count[cls] : MFGP_PROF_POOL;
    for (long long i = 0; h->prof_ev && i < n; i++) {
      float ms = 0.f;
      CUDA_TRY(h, cudaEventElapsedTime(&ms, h->prof_ev[(cls * MFGP_PROF_POOL + i) * 2],
                                       h->prof_ev[(cls * MFGP_PROF_POOL + i) * 2 + 1]));
      total += ms;
    }
    h_ms[cls] = n > 0 ? total / (double)n : 0.0;   // average duration of the timed launches
    h_count[cls] = h->prof_count[cls];
  }
  return 0;
}

int mfgp_assemble(mfgp_handle_t h, int kind, const double* d_X, int N, int D, int d,
                  const double* h_theta, int P, double jitter, double* d_K, long long ldk, int uplo) {
  ENTER(h);
  ARG_CHECK(h, d_X && d_K && N >= 0 && ldk >= N);
  ARG_CHECK(h, uplo == MFGP_UPLO_LOWER || uplo == MFGP_UPLO_FULL);
  KParams kp;
  int rc = make_kparams(h, kind, D, d, h_theta, P, &kp);
  if (rc) return rc;
  if (N == 0) return 0;
  return assemble_launch(h, kp, d_X, N, kp.noise + JITTER_CONST + jitter, d_K, ldk, uplo, 0);
}

// shared by factorize / lml_grad: returns after enqueueing; scalars at d_scalars[0..2]
static int factor_enqueue(mfgp_ctx* h, const KParams& kp, const double* d_X, const double* d_y, int N,
                          double jitter, double* d_A, double* d_W, double* d_alpha,
                          cudaEvent_t* ev /* optional, 5 events */, bool defer_solve = false) {
  const int npad = mfgp_padded_n(N);
  ARG_CHECK(h, npad <= MFGP_PARTIALS);
  int rc;
  if (ev) CUDA_TRY(h, cudaEventRecord(ev[0], h->stream));
  if ((rc = assemble_launch(h, kp, d_X, N, kp.noise + JITTER_CONST + jitter, d_A, npad,
                            MFGP_UPLO_LOWER, npad)))
    return rc;
  if (ev) CUDA_TRY(h, cudaEventRecord(ev[1], h->stream));
  // (ev[2] sits where the factorisation is complete; part of the inverse may already have run by then)
  if ((rc = potrf_trtri_padded(h, d_A, d_W, npad, N, ev ? ev[2] : nullptr))) return rc;
  if (ev) CUDA_TRY(h, cudaEventRecord(ev[3], h->stream));
  if (defer_solve) return 0;
  if ((rc = solve_alpha_launch(h, d_A, d_W, npad, N, d_y, h->d_partials, d_alpha, h->d_scalars, npad)))
    return rc;
  if (ev) CUDA_TRY(h, cudaEventRecord(ev[4], h->stream));
  return 0;
}

int mfgp_factorize(mfgp_handle_t h, int kind, const double* d_X, const double* d_y, int N, int D,
                   int d, const double* h_theta, int P, double jitter, double* d_A, double* d_W,
                   double* d_alpha, double* h_out) {
  ENTER(h);
  ARG_CHECK(h, d_X && d_y && d_A && d_W && d_alpha && N >= 1);
  KParams kp;
  int rc = make_kparams(h, kind, D, d, h_theta, P, &kp);
  if (rc) return rc;
  if (N <= MFGP_SMALL_N) {
    if ((rc = small_gp_launch(h, kp, d_X, d_y, N, kp.noise + JITTER_CONST + jitter, d_A, d_W, d_alpha,
                              h->d_scalars, 0)))
      return rc;
  } else if ((rc = factor_enqueue(h, kp, d_X, d_y, N, jitter, d_A, d_W, d_alpha, nullptr))) {
    return rc;
  }
  if ((rc = fetch_scalars(h, 3))) return rc;
  if (h_out) {
    h_out[0] = h->h_pinned[0];
    h_out[1] = h->h_pinned[1];
    h_out[2] = h->h_pinned[2];
  }
  return h->h_info[0];
}

static void grads_from_sums(const KParams& kp, const double* S, double* g) {
  const double* th = kp.theta;
  if (kp.kind == MFGP_KIND_COMPOSITE) {
    g[0] = S[0] / th[0];
    g[1] = len_grad(S[1], th[1]);
    g[2] = S[0] / th[2];
    g[3] = len_grad(S[2], th[3]);
    g[4] = S[3] / th[4];
    g[5] = len_grad(S[4], th[5]);
    g[6] = S[5];
  } else {
    g[0] = S[0] / th[0];
    g[1] = len_grad(S[1] + S[2], th[1]);
    g[2] = S[5];
  }
}

int mfgp_lml_grad_timed(mfgp_handle_t h, int kind, const double* d_X, const double* d_y, int N,
                        int D, int d, const double* h_theta, int P, double jitter, double* d_A,
                        double* d_W, double* d_alpha, double* h_lml, double* h_grad, double* h_ms) {
  ENTER(h);
  ARG_CHECK(h, d_X && d_y && d_A && d_W && d_alpha && N >= 1);
  KParams kp;
  int rc = make_kparams(h, kind, D, d, h_theta, P, &kp);
  if (rc) return rc;
  const int npad = mfgp_padded_n(N);
  if (N <= MFGP_SMALL_N) {   // one fused launch; no per-stage times
    if ((rc = small_gp_launch(h, kp, d_X, d_y, N, kp.noise + JITTER_CONST + jitter, d_A, d_W, d_alpha,
                              h->d_scalars, 1)))
      return rc;
    if ((rc = fetch_scalars(h, 16))) return rc;
    if (h_lml) h_lml[0] = h->h_pinned[0];
    if (h_grad) grads_from_sums(kp, h->h_pinned + 8, h_grad);
    if (h_ms)
      for (int i = 0; i < 6; i++) h_ms[i] = 0.0;
    return h->h_info[0];
  }
  cudaEvent_t* ev = h_ms ? h->ev : nullptr;
  // Untimed (production) schedule: the O(N^2), HBM-bound solves (v = W y, alpha = W^T v, LML) run on the side stream
  // UNDER the tensor-bound K^-1 = W^T W -- both only read W.  With stage timing the schedule stays sequential so
  // that the six stage times add up.
  if (!ev && h->s_hi && npad >= 2048 && 2LL * npad <= MFGP_PARTIALS) {
    if ((rc = factor_enqueue(h, kp, d_X, d_y, N, jitter, d_A, d_W, d_alpha, nullptr, true))) return rc;
    cudaStream_t caller = h->stream;
    cudaEvent_t ev_fork = h->ev_la[3 * 64], ev_join = h->ev_la[3 * 64 + 1];
    // the log-determinant needs the diagonal of L, which K^-1 is about to overwrite: packed copy first
    double* diag = h->d_partials + npad;
    CUDA_TRY(h, cudaMemcpy2DAsync(diag, sizeof(double), d_A, (size_t)(npad + 1) * sizeof(double), sizeof(double),
                                  (size_t)N, cudaMemcpyDeviceToDevice, caller));
    CUDA_TRY(h, cudaEventRecord(ev_fork, caller));
    CUDA_TRY(h, cudaStreamWaitEvent(h->s_hi, ev_fork, 0));
    h->stream = h->s_hi;
    rc = solve_alpha_launch(h, diag, d_W, npad, N, d_y, h->d_partials, d_alpha, h->d_scalars, 0);
    h->stream = caller;
    if (rc) return rc;
    CUDA_TRY(h, cudaEventRecord(ev_join, h->s_hi));
    if ((rc = lauum_padded(h, d_W, d_A, npad))) return rc;
    CUDA_TRY(h, cudaStreamWaitEvent(caller, ev_join, 0));
  } else {
    if ((rc = factor_enqueue(h, kp, d_X, d_y, N, jitter, d_A, d_W, d_alpha, ev))) return rc;
    if ((rc = lauum_padded(h, d_W, d_A, npad))) return rc;
  }
  if (ev) CUDA_TRY(h, cudaEventRecord(ev[5], h->stream));
  if ((rc = grad_reduce_launch(h, kp, d_X, N, d_A, npad, d_alpha, h->d_scalars + 8))) return rc;
  if (ev) CUDA_TRY(h, cudaEventRecord(ev[6], h->stream));
  if ((rc = fetch_scalars(h, 16))) return rc;
  if (h_lml) h_lml[0] = h->h_pinned[0];
  if (h_grad) grads_from_sums(kp, h->h_pinned + 8, h_grad);
  if (h_ms) {
    for (int i = 0; i < 6; i++) {
      float ms = 0.f;
      CUDA_TRY(h, cudaEventElapsedTime(&ms, ev[i], ev[i + 1]));
      h_ms[i] = ms;
    }
  }
  return h->h_info[0];
}

int mfgp_lml_grad(mfgp_handle_t h, int kind, const double* d_X, const double* d_y, int N, int D,
                  int d, const double* h_theta, int P, double jitter, double* d_A, double* d_W,
                  double* d_alpha, double* h_lml, double* h_grad) {
  return mfgp_lml_grad_timed(h, kind, d_X, d_y, N, D, d, h_theta, P, jitter, d_A, d_W, d_alpha,
                             h_lml, h_grad, nullptr);
}

int mfgp_lml_grad_batch_max(void) { return small_batch_max(); }

int mfgp_lml_grad_batch(mfgp_handle_t h, int kind, const double* d_X, const double* d_y, int N, int D, int d,
                        const double* h_thetas, int P, int B, double jitter, double* h_lml, double* h_grad,
                        int* h_info) {
  ENTER(h);
  ARG_CHECK(h, d_X && d_y && h_thetas && h_lml && h_info && B >= 1 && N >= 1 && N <= MFGP_TILE);
  const int bmax = small_batch_max();
  KParams kps[16];
  double diag_add[16];
  for (int b0 = 0; b0 < B; b0 += bmax) {
    const int nb = B - b0 < bmax ? B - b0 : bmax;
    int rc;
    for (int b = 0; b < nb; b++) {
      if ((rc = make_kparams(h, kind, D, d, h_thetas + (long)(b0 + b) * P, P, &kps[b]))) return rc;
      diag_add[b] = kps[b].noise + JITTER_CONST + jitter;
    }
    // the kernel writes its scalars straight into mapped pinned host memory: one launch + one sync
    if ((rc = small_lml_batch_launch(h, kps, diag_add, nb, d_X, d_y, N, h->d_batch, h->d_batch_info,
                                     h_grad != nullptr)))
      return rc;
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    for (int b = 0; b < nb; b++) {
      h_lml[b0 + b] = h->h_batch[b * 16];
      h_info[b0 + b] = h->h_batch_info[b];
      if (h_grad) grads_from_sums(kps[b], h->h_batch + b * 16 + 8, h_grad + (long)(b0 + b) * P);
    }
  }
  return 0;
}

int mfgp_append_point(mfgp_handle_t h, int kind, const double* d_X, const double* d_y, int N, int D,
                      int d, const double* h_theta, int P, double jitter, double* d_A, double* d_W,
                      double* d_alpha, int a_holds_L, double* h_out) {
  ENTER(h);
  ARG_CHECK(h, d_X && d_y && d_A && d_W && d_alpha && N >= 1);
  KParams kp;
  int rc = make_kparams(h, kind, D, d, h_theta, P, &kp);
  if (rc) return rc;
  const int npad = mfgp_padded_n(N + 1);   // the buffers are sized for the N+1 points
  ARG_CHECK(h, 3LL * npad <= MFGP_PARTIALS);
  double* krow = h->d_partials;
  double* l_tmp = krow + npad;
  double* t_tmp = l_tmp + npad;
  CUDA_TRY(h, cudaMemsetAsync(h->d_info, 0, sizeof(int), h->stream));
  // k = K(x_new, X[0:N]) (zero on the pad); the new point is row N of d_X
  if ((rc = cross_gen_launch(h, kp, d_X, N, npad, d_alpha, d_X + (long long)N * D, 1, 1, krow, nullptr))) return rc;
  if ((rc = append_point_launch(h, krow, N, npad, kp.kdiag + kp.noise + JITTER_CONST + jitter, d_A, d_W,
                                a_holds_L, l_tmp, t_tmp, h->d_scalars + 32)))
    return rc;
  if ((rc = solve_alpha_launch(h, d_A, d_W, npad, N + 1, d_y, h->d_partials, d_alpha, h->d_scalars, npad))) return rc;
  if ((rc = fetch_scalars(h, 40))) return rc;
  if (h_out) {
    h_out[0] = a_holds_L ? h->h_pinned[0] : NAN;   // LML of the N+1 points
    h_out[1] = a_holds_L ? h->h_pinned[1] : NAN;   // logdet
    h_out[2] = h->h_pinned[2];                     // y^T alpha
    h_out[3] = h->h_pinned[32];                    // new diagonal entry of L
  }
  return h->h_info[0];
}

int mfgp_potrf(mfgp_handle_t h, double* d_A, double* d_W, int npad) {
  ENTER(h);
  ARG_CHECK(h, d_A && d_W);
  int rc = potrf_padded(h, d_A, d_W, npad, npad);
  if (rc) return rc;
  if ((rc = fetch_scalars(h, 1))) return rc;
  return h->h_info[0];
}

int mfgp_trtri(mfgp_handle_t h, const double* d_L, double* d_W, int npad) {
  ENTER(h);
  ARG_CHECK(h, d_L && d_W);
  return trtri_padded(h, d_L, d_W, npad);
}

int mfgp_lauum(mfgp_handle_t h, const double* d_W, double* d_Kinv, int npad) {
  ENTER(h);
  ARG_CHECK(h, d_W && d_Kinv && d_W != d_Kinv);
  return lauum_padded(h, d_W, d_Kinv, npad);
}

size_t mfgp_predict_ws_bytes(int N, long long cols) {
  const long long npad = mfgp_padded_n(N);
  const long long cp = (cols + 127) / 128 * 128;
  return (size_t)((npad + 1) * cp) * sizeof(double);
}

static int level_kparams(mfgp_ctx* h, const mfgp_level_t* gp, KParams* kp) {
  ARG_CHECK(h, gp != nullptr && gp->d_X != nullptr && gp->d_alpha != nullptr && gp->N >= 1);
  return make_kparams(h, gp->kind, gp->D, gp->d, gp->h_theta, gp->P, kp);
}

// Column chunks are sized in whole waves of 128-column tiles (one CTA per SM): a chunk of 149 tiles costs two
// waves, i.e. twice the time of 148 (found the hard way: a scratch that grew by 0.1 % doubled the
// low-fidelity stage of the MC sweep).  Results never depend on the chunk size.
static long long whole_waves(long long cols) {
  const long long wave = (long long)MFGP_NUM_SMS * 128;
  return cols > wave ? cols / wave * wave : cols;
}

// latent: d_var receives k(x, x) - |W k_x|^2 unclipped and without noise (the batch acquisition's v_0)
static int predict_impl(mfgp_ctx* h, const mfgp_level_t* gp, const KParams& kp, const double* d_Xnew,
                        long long M, double* d_mean, double* d_var, int include_noise, double* d_ws,
                        size_t ws_bytes, bool latent = false) {
  const int npad = mfgp_padded_n(gp->N);
  int rc;
  if (M <= 0) return 0;
  if (!d_var) {   // mean only: no cross-covariance is ever stored
    ARG_CHECK(h, d_mean != nullptr);
    return cross_gen_launch(h, kp, gp->d_X, gp->N, npad, gp->d_alpha, d_Xnew, M, M, nullptr, d_mean);
  }
  ARG_CHECK(h, gp->d_W != nullptr && d_ws != nullptr);
  const long long per_col = (long long)npad + 1;
  long long chunk = whole_waves((long long)(ws_bytes / sizeof(double)) / per_col / 128 * 128);
  ARG_CHECK(h, chunk >= 128);
  double* Ks = d_ws;
  double* ss = d_ws + chunk * npad;
  for (long long c0 = 0; c0 < M; c0 += chunk) {
    const long long ncols = (M - c0 < chunk) ? (M - c0) : chunk;
    const long long cols_pad = (ncols + 127) / 128 * 128;
    if ((rc = cross_gen_launch(h, kp, gp->d_X, gp->N, npad, gp->d_alpha, d_Xnew + c0 * kp.D, ncols,
                               cols_pad, Ks, d_mean ? d_mean + c0 : nullptr)))
      return rc;
    if ((rc = trmm_sumsq(h, gp->d_W, npad, Ks, cols_pad, ss))) return rc;
    if ((rc = finish_var_launch(h, ss, ncols, kp.kdiag, include_noise ? kp.noise : 0.0, d_var + c0, latent)))
      return rc;
  }
  return 0;
}

int mfgp_predict(mfgp_handle_t h, const mfgp_level_t* gp, const double* d_Xnew, long long M,
                 double* d_mean, double* d_var, int include_noise, double* d_ws, size_t ws_bytes) {
  ENTER(h);
  KParams kp;
  int rc = level_kparams(h, gp, &kp);
  if (rc) return rc;
  ARG_CHECK(h, d_Xnew != nullptr || M == 0);
  return predict_impl(h, gp, kp, d_Xnew, M, d_mean, d_var, include_noise, d_ws, ws_bytes);
}

// ---- K6d predictive gradients (math: assemble.cu, cross_grad_kernel) -------------------------------------------
// Scratch: W^T (npad^2) | per chunk Ks, reused for Ut = Ks K_y^-1 (chunk x npad) | Tt (chunk x npad).
size_t mfgp_predictive_gradients_ws_bytes(int N, long long cols) {
  const long long npad = mfgp_padded_n(N);
  const long long cp = ((cols < 1 ? 1 : cols) + 127) / 128 * 128;
  return (size_t)(npad * npad + 2 * npad * cp) * sizeof(double);
}

int mfgp_predictive_gradients(mfgp_handle_t h, const mfgp_level_t* gp, const double* d_Xnew, long long M,
                              double* d_dmean, double* d_dvar, double* d_mean, double* d_var, int include_noise,
                              double* d_ws, size_t ws_bytes) {
  ENTER(h);
  KParams kp;
  int rc = level_kparams(h, gp, &kp);
  if (rc) return rc;
  ARG_CHECK(h, M >= 0 && (d_Xnew != nullptr || M == 0) && d_dmean != nullptr);
  ARG_CHECK(h, d_dvar != nullptr || d_var == nullptr);   // the variance needs W, as its gradient does
  const int N = gp->N, D = gp->D, npad = mfgp_padded_n(N);
  long long chunk = M;
  double *Wt = nullptr, *Ks = nullptr, *Tt = nullptr;
  if (d_dvar) {
    ARG_CHECK(h, gp->d_W != nullptr && d_ws != nullptr);
    ARG_CHECK(h, ws_bytes >= mfgp_predictive_gradients_ws_bytes(N, 128));
    const long long avail = (long long)(ws_bytes / sizeof(double)) - (long long)npad * npad;
    chunk = whole_waves(avail / (2LL * npad) / 128 * 128);
    Wt = d_ws;
    Ks = Wt + (long long)npad * npad;
    Tt = Ks + chunk * npad;
  }
  if (M == 0) return 0;
  if (d_dvar && (rc = transpose_launch(h, gp->d_W, npad, Wt))) return rc;
  for (long long c0 = 0; c0 < M; c0 += chunk) {
    const long long ncols = (M - c0 < chunk) ? (M - c0) : chunk;
    const long long cols_pad = (ncols + 127) / 128 * 128;
    const double* Xq = d_Xnew + c0 * D;
    if (d_dvar) {
      if ((rc = cross_gen_launch(h, kp, gp->d_X, N, npad, gp->d_alpha, Xq, ncols, cols_pad, Ks, nullptr))) return rc;
      if ((rc = kinv_rows(h, gp->d_W, Wt, npad, Ks, cols_pad, Tt, Ks))) return rc;
    }
    if ((rc = cross_grad_launch(h, kp, gp->d_X, N, gp->d_alpha, d_dvar ? Ks : nullptr, npad, Xq, ncols,
                                d_dmean + c0 * D, d_dvar ? d_dvar + c0 * D : nullptr, d_mean ? d_mean + c0 : nullptr,
                                d_var ? d_var + c0 : nullptr)))
      return rc;
    if (d_var && (rc = finish_var_launch(h, d_var + c0, ncols, kp.kdiag, include_noise ? kp.noise : 0.0, d_var + c0,
                                         false)))
      return rc;
  }
  return 0;
}

int mfgp_predict_small_max_rows(void) { return 16; }

int mfgp_predict_small(mfgp_handle_t h, const mfgp_level_t* hf, const mfgp_level_t* lf, const double* h_X,
                       int M, const double* h_offsets, int E, double tau, int include_noise, double* h_mean,
                       double* h_var) {
  ENTER(h);
  KParams kh, kl;
  int rc;
  if ((rc = level_kparams(h, hf, &kh))) return rc;
  ARG_CHECK(h, hf->d_W != nullptr && h_X && h_mean && h_var && M >= 1 && M <= mfgp_predict_small_max_rows());
  ARG_CHECK(h, hf->N <= predict_small_max_n());
  // staging in the mapped pinned block (16 x 16 doubles): [0, 128) query rows, [128, 160) results,
  // [160, 224) augmented rows are kept on the device side of d_scalars instead (no host visibility needed)
  const int width = lf ? lf->D : hf->D;
  ARG_CHECK(h, M * width <= 128 && M * hf->D <= 1024);
  double* d_offs = h->d_scalars + 64;
  double* d_aug = h->d_scalars + 2048;
  if (lf) {
    if ((rc = level_kparams(h, lf, &kl))) return rc;
    ARG_CHECK(h, h_offsets && E >= 1 && E <= MFGP_MAX_E && hf->D == lf->D + E && E * lf->D <= 96);
    // the offsets travel as kernel-visible data through the same mapped block (after the query rows)
    memcpy(h->h_batch + 160, h_offsets, (size_t)E * lf->D * sizeof(double));
    d_offs = h->d_batch + 160;
  }
  memcpy(h->h_batch, h_X, (size_t)M * width * sizeof(double));
  if ((rc = predict_small_launch(h, kh, hf, lf ? &kl : nullptr, lf, h->d_batch, M, d_offs, E, tau, d_aug,
                                 include_noise ? kh.noise : 0.0, h->d_batch + 128)))
    return rc;
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  for (int m = 0; m < M; m++) {
    h_mean[m] = h->h_batch[128 + 2 * m];
    h_var[m] = h->h_batch[128 + 2 * m + 1];
  }
  return 0;
}

// ---- point service (see point_service_kernel) ----------------------------------------------------------
static int point_service_relaunch(mfgp_ctx* h) {
  h->svc_h->alive = 1;
  h->svc_args.start_seq = h->svc_h->ack_seq;
  __sync_synchronize();
  return point_service_launch(h, h->svc_args, h->svc_d, h->s_svc);
}

int mfgp_point_service_stop(mfgp_handle_t h) {
  ENTER(h);
  if (!h->svc_active) return 0;
  h->svc_h->stop = 1;
  __sync_synchronize();
  CUDA_TRY(h, cudaStreamSynchronize(h->s_svc));
  h->svc_active = 0;
  return 0;
}

int mfgp_point_service_start(mfgp_handle_t h, const mfgp_level_t* hf, const mfgp_level_t* lf,
                             const double* h_offsets, int E, double tau, int include_noise, double idle_ms) {
  ENTER(h);
  int rc;
  if (h->svc_active && (rc = mfgp_point_service_stop(h))) return rc;
  PointServiceArgs& a = h->svc_args;
  memset(&a, 0, sizeof(a));
  if ((rc = level_kparams(h, hf, &a.kh))) return rc;
  ARG_CHECK(h, hf->d_W != nullptr && hf->N >= 1 && hf->N <= predict_small_max_n() && hf->D <= 64);
  a.Xh = hf->d_X; a.Nh = hf->N; a.npad_h = mfgp_padded_n(hf->N); a.alpha_h = hf->d_alpha; a.Wh = hf->d_W;
  a.noise_add = include_noise ? a.kh.noise : 0.0;
  a.has_lf = lf != nullptr;
  h->svc_width = hf->D;
  if (lf) {
    if ((rc = level_kparams(h, lf, &a.kl))) return rc;
    ARG_CHECK(h, h_offsets && E >= 1 && E <= MFGP_MAX_E && hf->D == lf->D + E && E * lf->D <= 96 && lf->d_alpha);
    a.Xl = lf->d_X; a.Nl = lf->N; a.alpha_l = lf->d_alpha; a.d = lf->D; a.E = E; a.tau = tau;
    memcpy(a.offs, h_offsets, (size_t)E * lf->D * sizeof(double));
    h->svc_width = lf->D;
  }
  if (!(idle_ms > 0.0)) idle_ms = 20.0;
  a.idle_ns = (unsigned long long)(idle_ms * 1e6);
  // the factors may still be in flight on the caller's stream
  CUDA_TRY(h, cudaEventRecord(h->ev_la[3 * 64 + 3], h->stream));
  CUDA_TRY(h, cudaStreamWaitEvent(h->s_svc, h->ev_la[3 * 64 + 3], 0));
  h->svc_h->stop = 0;
  h->svc_seq = h->svc_h->ack_seq = h->svc_h->req_seq;
  h->svc_relaunches = -1;     // the first launch is not a relaunch
  if ((rc = point_service_relaunch(h))) return rc;
  h->svc_relaunches = 0;
  h->svc_active = 1;
  return 0;
}

// One question: h_x (width doubles: plain inputs with a low-fidelity level, augmented row without) -> out[0] = mean,
// out[1] = variance.  Spins on the mapped acknowledgement; relaunches the kernel if it left on its idle limit.
int mfgp_point_service_eval(mfgp_handle_t h, const double* h_x, double* h_out) {
  if (!h) return -1;
  ARG_CHECK(h, h->svc_active && h_x && h_out);
  PointServiceCtl* c = h->svc_h;
  for (int i = 0; i < h->svc_width; i++) c->x[i] = h_x[i];
  __sync_synchronize();
  const unsigned long long seq = ++h->svc_seq;
  c->req_seq = seq;
  __sync_synchronize();
  struct timespec t0;
  clock_gettime(CLOCK_MONOTONIC, &t0);
  for (unsigned long long spin = 1;; spin++) {
    if (c->ack_seq == seq) break;
    if (!c->alive) {
      DeviceGuard guard(h->device);
      cudaStreamSynchronize(h->s_svc);          // the old kernel has decided to leave; let it finish
      if (c->ack_seq == seq) break;             // it answered on its way out
      int rc = point_service_relaunch(h);
      if (rc) return rc;
      h->svc_relaunches++;
    }
    if ((spin & 0xffff) == 0) {
      struct timespec t1;
      clock_gettime(CLOCK_MONOTONIC, &t1);
      if ((t1.tv_sec - t0.tv_sec) + 1e-9 * (t1.tv_nsec - t0.tv_nsec) > 10.0) {
        cudaError_t e = cudaStreamQuery(h->s_svc);
        snprintf(h->err, sizeof(h->err), "point service: no answer within 10 s (stream state: %s)", cudaGetErrorString(e));
        return -102;
      }
    }
  }
  __sync_synchronize();
  h_out[0] = c->out[0];
  h_out[1] = c->out[1];
  return 0;
}

long long mfgp_point_service_relaunches(mfgp_handle_t h) { return h ? h->svc_relaunches : -1; }

int mfgp_augment(mfgp_handle_t h, const mfgp_level_t* lf, const double* d_X, long long M,
                 const double* h_offsets, int E, double tau, double* d_Xaug, double* d_ws,
                 size_t ws_bytes) {
  ENTER(h);
  KParams kp;
  int rc = level_kparams(h, lf, &kp);
  if (rc) return rc;
  const int d = lf->D;
  ARG_CHECK(h, h_offsets && E >= 1 && E <= MFGP_MAX_E && d + E <= MFGP_MAX_D && E * d <= MFGP_SMALL - 64);
  ARG_CHECK(h, d_X && d_Xaug && d_ws);
  if (M <= 0) return 0;
  double* d_offs = h->d_scalars + 64;
  CUDA_TRY(h, cudaMemcpyAsync(d_offs, h_offsets, (size_t)E * d * sizeof(double),
                              cudaMemcpyHostToDevice, h->stream));
  const long long per_row = (long long)E * (d + 1);
  long long chunk = (long long)(ws_bytes / sizeof(double)) / per_row;
  ARG_CHECK(h, chunk >= 1);
  if (chunk > M) chunk = M;
  double* locs = d_ws;
  double* vals = d_ws + chunk * E * d;
  const int npad = mfgp_padded_n(lf->N);
  for (long long r0 = 0; r0 < M; r0 += chunk) {
    const long long rows = (M - r0 < chunk) ? (M - r0) : chunk;
    if ((rc = build_locs_launch(h, d_X + r0 * d, rows, d, d_offs, E, tau, locs))) return rc;
    if ((rc = cross_gen_launch(h, kp, lf->d_X, lf->N, npad, lf->d_alpha, locs, rows * E, rows * E,
                               nullptr, vals)))
      return rc;
    if ((rc = concat_aug_launch(h, d_X + r0 * d, vals, rows, d, E, d_Xaug + r0 * (d + E)))) return rc;
  }
  return 0;
}

// K7 through a chain of L >= 2 levels; L = 2 is mfgp_predict_mc.  levels[0]: GP on x (D = d); levels[t >= 1]:
// GP on [x, z] (D = d + 1).  Sampling #j (the value level j-1 hands to level j) draws from Philox key
// seed + (j-1) * golden-ratio increment with counter (m0 + m) S + s, or from d_eps[(j-1) M S + m S + s].
#define MFGP_MAX_LEVELS 8
static int mc_chain_impl(mfgp_ctx* h, const mfgp_level_t* const* levels, int L, const double* d_Xtest,
                         long long M, int S, const double* d_eps, unsigned long long seed, long long m0,
                         int include_lower_noise, int include_top_noise, const double* d_weights,
                         double* d_mean, double* d_var, double* h_wsum, double* d_ws, size_t ws_bytes) {
  ARG_CHECK(h, levels && L >= 2 && L <= MFGP_MAX_LEVELS);
  KParams kp[MFGP_MAX_LEVELS];
  int rc;
  for (int t = 0; t < L; t++) {
    ARG_CHECK(h, levels[t] != nullptr);
    if ((rc = level_kparams(h, levels[t], &kp[t]))) return rc;
    ARG_CHECK(h, levels[t]->d_W != nullptr);
  }
  const mfgp_level_t* lf = levels[0];
  const int d = lf->D;
  int npad_max = 0;
  for (int t = 1; t < L; t++) {
    // E = 1: NARGP (composite kernel on [x, z]) or GPDF without delays (one RBF over [x, z]: az == ax, so
    // the same code runs with the split at d)
    ARG_CHECK(h, levels[t]->D == d + 1 && (levels[t]->d == d || levels[t]->kind == MFGP_KIND_RBF));
    kp[t].d = d;
    const int np_t = mfgp_padded_n(levels[t]->N);
    if (np_t > npad_max) npad_max = np_t;
  }
  ARG_CHECK(h, d_Xtest && d_mean && d_var && d_ws && S >= 1 && M >= 0);
  ARG_CHECK(h, L == 2 || S <= mc_max_samples());
  if (M == 0) return 0;
  const long long wsd = (long long)(ws_bytes / sizeof(double));
  ARG_CHECK(h, wsd > 2 * M);
  double* mu_l = d_ws;
  double* sd_l = d_ws + M;
  double* rest = d_ws + 2 * M;
  const long long restd = wsd - 2 * M;
  // low-fidelity posterior marginals at the test points (kept out of the per-class profile so that
  // the trmm_sumsq / cross_gen classes hold the high-fidelity launches only)
  const int prof_saved = h->prof_on;
  h->prof_on = 0;
  rc = predict_impl(h, lf, kp[0], d_Xtest, M, mu_l, sd_l, include_lower_noise, rest,
                    (size_t)restd * sizeof(double));
  h->prof_on = prof_saved;
  if (rc) return rc;
  if ((rc = sqrt_launch(h, sd_l, M))) return rc;
  // upper levels over (point, sample) columns
  const int D = d + 1;
  // when every upper level takes the fused small-level kernel no cross-covariance row is ever stored: a column
  // needs its mean, sum of squares and sample only, and a chunk is as many points as the scratch holds
  bool all_small = true;
  for (int t = 1; t < L; t++) all_small = all_small && mc_small_applies(levels[t]->N);
  const long long per_col = all_small ? 3 : (long long)npad_max + D + 3;
  long long max_cols = all_small ? (restd - 384) / per_col : whole_waves(restd / per_col / 128 * 128);
  ARG_CHECK(h, max_cols >= (all_small ? S : 128));
  long long pm = max_cols / S;
  ARG_CHECK(h, pm >= 1);   // the scratch must hold all S samples of at least one point
  if (pm > M) pm = M;
  const long long cp_max = (pm * S + 127) / 128 * 128;
  double* Xq = rest;                 // (cp_max, D): rows [x, z] when S exceeds the generator's sample limit
  double* mu_c = Xq + (all_small ? 0 : cp_max * D);
  double* ss = mu_c + cp_max;
  double* zcol = ss + cp_max;
  double* Ks = zcol + cp_max;
  for (long long m_lo = 0; m_lo < M; m_lo += pm) {
    const long long npts = (M - m_lo < pm) ? (M - m_lo) : pm;
    const long long ncols = npts * S;
    const long long cols_pad = (ncols + 127) / 128 * 128;
    for (int t = 1; t < L; t++) {
      const mfgp_level_t* lv = levels[t];
      const int npad = mfgp_padded_n(lv->N);
      const unsigned long long key = seed + (unsigned long long)(t - 1) * 0x9E3779B97F4A7C15ULL;
      const double* eps_t = d_eps ? d_eps + (long long)(t - 1) * M * S : nullptr;
      int fused = 0;
      if (t == 1) {
        if ((rc = mc_small_launch(h, kp[1], lv->d_X, lv->N, npad, lv->d_W, lv->d_alpha, d_Xtest, mu_l, sd_l, eps_t, key,
                                  m0, m_lo, npts, S, mu_c, ss, nullptr, 0, 0, &fused)))
          return rc;
        if (fused) {
        } else if (S <= mc_max_samples()) {
          // one CTA per test point: x-dependent kernel factors shared by its S samples (1 exp / element)
          if ((rc = cross_gen_mc_launch(h, kp[1], lv->d_X, lv->N, npad, lv->d_alpha, d_Xtest, mu_l, sd_l, eps_t,
                                        key, m0, m_lo, npts, S, cols_pad, Ks, mu_c, nullptr, 0, 0)))
            return rc;
        } else {
          if ((rc = build_mc_rows_launch(h, d_Xtest, mu_l, sd_l, eps_t, key, m0, m_lo, ncols, S, d, Xq)))
            return rc;
          if ((rc = cross_gen_launch(h, kp[1], lv->d_X, lv->N, npad, lv->d_alpha, Xq, ncols, cols_pad, Ks, mu_c)))
            return rc;
        }
      } else {
        // z = mu + sqrt(v) eps of the level below, per (point, sample) column, then this level at [x, z]
        if ((rc = sample_cols_launch(h, mu_c, ss, eps_t, key, m0, m_lo, ncols, S, zcol))) return rc;
        if ((rc = mc_small_launch(h, kp[t], lv->d_X, lv->N, npad, lv->d_W, lv->d_alpha, d_Xtest, nullptr, nullptr,
                                  nullptr, 0, m0, m_lo, npts, S, mu_c, ss, zcol, 0, S, &fused)))
          return rc;
        if (!fused &&
            (rc = cross_gen_mc_launch(h, kp[t], lv->d_X, lv->N, npad, lv->d_alpha, d_Xtest, nullptr, nullptr,
                                      nullptr, 0, m0, m_lo, npts, S, cols_pad, Ks, mu_c, zcol, 0, S)))
          return rc;
      }
      if (!fused && (rc = trmm_sumsq(h, lv->d_W, npad, Ks, cols_pad, ss))) return rc;
      const int with_noise = (t == L - 1) ? include_top_noise : include_lower_noise;
      if ((rc = finish_var_launch(h, ss, ncols, kp[t].kdiag, with_noise ? kp[t].noise : 0.0, ss))) return rc;
    }
    if ((rc = mc_aggregate_launch(h, mu_c, ss, npts, S, d_mean + m_lo, d_var + m_lo))) return rc;
  }
  if (h_wsum) {
    if ((rc = wdot_launch(h, d_weights, d_mean, M, h->d_scalars + 20))) return rc;
    if ((rc = fetch_scalars(h, 24))) return rc;
    h_wsum[0] += h->h_pinned[20];
  }
  return 0;
}

size_t mfgp_predict_mc_ws_bytes(int N_l, int N_up, int d, long long M, int S) {
  const long long npl = mfgp_padded_n(N_l), npu = mfgp_padded_n(N_up);
  const long long tiles4 = (long long)MFGP_NUM_SMS * 128 * 4;
  const long long lf_need = (npl + 1) * 128 * 8, lf_want = (npl + 1) * tiles4 * 8;
  long long up_need, up_want;
  if (mc_small_applies(N_up)) {
    const long long cols = M * (long long)S;
    up_need = ((long long)S + 256) * 24;
    up_want = (cols < (1LL << 28) ? cols : (1LL << 28)) * 24 + 8192;
  } else {
    const long long per_col = (npu + d + 4) * 8;
    up_need = ((long long)S + 256) * per_col;
    up_want = tiles4 * per_col;
  }
  const long long need = 16 * M + (lf_need > up_need ? lf_need : up_need) + 4096;
  long long want = 16 * M + (lf_want > up_want ? lf_want : up_want) + 4096;
  if (want > (12LL << 30)) want = 12LL << 30;
  return (size_t)(want > need ? want : need);
}

int mfgp_predict_mc(mfgp_handle_t h, const mfgp_level_t* lf, const mfgp_level_t* hf,
                    const double* d_Xtest, long long M, int S, const double* d_eps,
                    unsigned long long seed, long long m0, int include_lf_noise,
                    int include_hf_noise, const double* d_weights, double* d_mean, double* d_var,
                    double* h_wsum, double* d_ws, size_t ws_bytes) {
  ENTER(h);
  const mfgp_level_t* levels[2] = {lf, hf};
  return mc_chain_impl(h, levels, 2, d_Xtest, M, S, d_eps, seed, m0, include_lf_noise, include_hf_noise,
                       d_weights, d_mean, d_var, h_wsum, d_ws, ws_bytes);
}

int mfgp_predict_mc_chain(mfgp_handle_t h, const mfgp_level_t* const* levels, int L, const double* d_Xtest,
                          long long M, int S, const double* d_eps, unsigned long long seed, long long m0,
                          int include_lower_noise, int include_top_noise, const double* d_weights,
                          double* d_mean, double* d_var, double* h_wsum, double* d_ws, size_t ws_bytes) {
  ENTER(h);
  return mc_chain_impl(h, levels, L, d_Xtest, M, S, d_eps, seed, m0, include_lower_noise, include_top_noise,
                       d_weights, d_mean, d_var, h_wsum, d_ws, ws_bytes);
}

size_t mfgp_predict_mc_joint_ws_bytes(int N_l, int N_h, long long M, int S) {
  const long long npl = mfgp_padded_n(N_l), nph = mfgp_padded_n(N_h);
  const long long Mp = (M + 127) / 128 * 128, Sp = ((long long)S + 127) / 128 * 128;
  const long long fixed = Mp + 2 * Mp * Mp + 2 * Mp * npl + 2 * Mp * Sp;
  const long long cols = (Mp * (long long)S < 148LL * 128 * 4 ? Mp * (long long)S : 148LL * 128 * 4) + 256 + S;
  return (size_t)(fixed + cols * (nph + 3)) * sizeof(double);
}

// K7 with the low-fidelity posterior sampled JOINTLY across the test points (small M): z_s = mu_l + chol(Sigma_l) eps_s
// with the full M x M predictive covariance Sigma_l = K(X*, X*) - (W_l K_l*)^T (W_l K_l*) (+ (noise + jitter) I),
// so that every sample s is one coherent low-fidelity function draw and per-path functionals
// (d_path_wsum[s] = sum_m w_m mu_s(x_m), the PCE mean of path s) are meaningful.
int mfgp_predict_mc_joint(mfgp_handle_t h, const mfgp_level_t* lf, const mfgp_level_t* hf,
                          const double* d_Xtest, long long M, int S, const double* d_eps,
                          unsigned long long seed, int include_lf_noise, int include_hf_noise,
                          double lf_jitter, const double* d_weights, double* d_mean, double* d_var,
                          double* d_path_wsum, double* d_ws, size_t ws_bytes) {
  ENTER(h);
  KParams kl, kh;
  int rc;
  if ((rc = level_kparams(h, lf, &kl))) return rc;
  if ((rc = level_kparams(h, hf, &kh))) return rc;
  const int d = lf->D;
  ARG_CHECK(h, hf->D == d + 1 && (hf->d == d || hf->kind == MFGP_KIND_RBF));
  kh.d = d;
  ARG_CHECK(h, lf->d_W && hf->d_W && d_Xtest && d_mean && d_var && d_ws);
  ARG_CHECK(h, S >= 1 && S <= mc_max_samples() && M >= 1 && M <= 16384);
  ARG_CHECK(h, ws_bytes >= mfgp_predict_mc_joint_ws_bytes(lf->N, hf->N, M, S));
  const int npl = mfgp_padded_n(lf->N), nph = mfgp_padded_n(hf->N);
  const long long Mp = (M + 127) / 128 * 128, Sp = ((long long)S + 127) / 128 * 128;
  double* mu_l = d_ws;                      // (Mp)
  double* Sigma = mu_l + Mp;                // (Mp, Mp) -> chol(Sigma_l), lower
  double* Wt = Sigma + Mp * Mp;             // (Mp, Mp) leaf inverses (scratch of the factorisation)
  double* Ksl = Wt + Mp * Mp;               // (Mp, npl)
  double* T = Ksl + Mp * npl;               // (npl, Mp)
  double* E = T + Mp * npl;                 // (Mp, Sp) standard normals
  double* Z = E + Mp * Sp;                  // (Mp, Sp) chol(Sigma_l) E
  double* rest = Z + Mp * Sp;
  const long long restd = (long long)(ws_bytes / sizeof(double)) - (rest - d_ws);
  const int prof_saved = h->prof_on;
  h->prof_on = 0;
  // joint low-fidelity posterior
  if ((rc = cross_gen_launch(h, kl, lf->d_X, lf->N, npl, lf->d_alpha, d_Xtest, M, Mp, Ksl, mu_l))) return rc;
  if ((rc = trmm_store(h, lf->d_W, npl, Ksl, Mp, T))) return rc;
  if ((rc = assemble_launch(h, kl, d_Xtest, (int)M, (include_lf_noise ? kl.noise : 0.0) + lf_jitter, Sigma, Mp,
                            MFGP_UPLO_LOWER, (int)Mp)))
    return rc;
  if ((rc = syrk_tn_sub(h, T, Mp, npl, Sigma, (int)Mp))) return rc;       // Sigma(lower) -= T^T T
  if ((rc = potrf_padded(h, Sigma, Wt, (int)Mp, (int)M))) return rc;
  if ((rc = fetch_scalars(h, 1))) return rc;
  if (h->h_info[0] != 0) {
    h->prof_on = prof_saved;
    return h->h_info[0];                    // joint covariance not positive definite: raise lf_jitter
  }
  if ((rc = fill_normal_padded_launch(h, d_eps, seed, M, S, Mp, Sp, E))) return rc;
  if ((rc = trmm_right_store(h, Sigma, (int)Mp, E, Sp, Z))) return rc;     // Z = chol(Sigma_l) E
  h->prof_on = prof_saved;
  if (d_path_wsum) CUDA_TRY(h, cudaMemsetAsync(d_path_wsum, 0, (size_t)S * sizeof(double), h->stream));
  // high-fidelity level over (point, sample) columns
  const long long per_col = (long long)nph + 3;
  long long max_cols = whole_waves(restd / per_col / 128 * 128);
  ARG_CHECK(h, max_cols >= 128);
  long long pm = max_cols / S;
  ARG_CHECK(h, pm >= 1);
  if (pm > M) pm = M;
  const long long cp_max = (pm * S + 127) / 128 * 128;
  double* mu_c = rest;
  double* ss = mu_c + cp_max;
  double* Ks = ss + cp_max;
  for (long long m_lo = 0; m_lo < M; m_lo += pm) {
    const long long npts = (M - m_lo < pm) ? (M - m_lo) : pm;
    const long long ncols = npts * S, cols_pad = (ncols + 127) / 128 * 128;
    if ((rc = cross_gen_mc_launch(h, kh, hf->d_X, hf->N, nph, hf->d_alpha, d_Xtest, mu_l, nullptr, nullptr, 0, 0,
                                  m_lo, npts, S, cols_pad, Ks, mu_c, Z, m_lo, Sp)))
      return rc;
    if ((rc = trmm_sumsq(h, hf->d_W, nph, Ks, cols_pad, ss))) return rc;
    if ((rc = finish_var_launch(h, ss, ncols, kh.kdiag, include_hf_noise ? kh.noise : 0.0, ss))) return rc;
    if ((rc = mc_aggregate_launch(h, mu_c, ss, npts, S, d_mean + m_lo, d_var + m_lo))) return rc;
    if (d_path_wsum && (rc = path_wsum_launch(h, mu_c, d_weights, m_lo, npts, S, d_path_wsum))) return rc;
  }
  return 0;
}

int mfgp_predict_mc_delays(mfgp_handle_t h, const mfgp_level_t* lf, const mfgp_level_t* hf,
                           const double* d_Xtest, long long M, const double* h_offsets, int E,
                           double tau, int S, const double* d_eps, unsigned long long seed,
                           long long m0, int include_lf_noise, int include_hf_noise, double lf_jitter,
                           const double* d_weights, double* d_mean, double* d_var, double* h_wsum,
                           double* d_ws, size_t ws_bytes) {
  ENTER(h);
  KParams kl, kh;
  int rc;
  if ((rc = level_kparams(h, lf, &kl))) return rc;
  if ((rc = level_kparams(h, hf, &kh))) return rc;
  const int d = lf->D;
  ARG_CHECK(h, lf->kind == MFGP_KIND_RBF);              // the reference's low-fidelity GP: RBF(d)
  ARG_CHECK(h, h_offsets && E >= 1 && E <= 8 && hf->D == d + E && (hf->d == d || hf->kind == MFGP_KIND_RBF));
  ARG_CHECK(h, lf->d_W && hf->d_W && d_Xtest && d_mean && d_var && d_ws && S >= 1 && M >= 0);
  ARG_CHECK(h, E * d + E * E <= MFGP_SMALL - 1024);
  if (M == 0) return 0;
  // prior covariance between the E locations of one point (depends on the offsets only)
  double h_kab[64];
  for (int a = 0; a < E; a++)
    for (int b = 0; b < E; b++) {
      double r2 = 0.0;
      for (int dd = 0; dd < d; dd++) {
        const double t = (h_offsets[a * d + dd] - h_offsets[b * d + dd]) * tau;
        r2 += t * t;
      }
      h_kab[a * E + b] = kl.c12 * exp(kl.ax * r2);
    }
  double* d_offs = h->d_scalars + 64;
  double* d_kab = h->d_scalars + 1024;
  CUDA_TRY(h, cudaMemcpyAsync(d_offs, h_offsets, (size_t)E * d * sizeof(double), cudaMemcpyHostToDevice, h->stream));
  CUDA_TRY(h, cudaMemcpyAsync(d_kab, h_kab, (size_t)E * E * sizeof(double), cudaMemcpyHostToDevice, h->stream));
  CUDA_TRY(h, cudaMemsetAsync(h->d_info + 1, 0x7f, sizeof(int), h->stream));
  const int npl = mfgp_padded_n(lf->N), nph = mfgp_padded_n(hf->N);
  const int D = d + E, NP = E * (E + 1) / 2;
  // scratch per test point (doubles); both stages reuse the same region, 2 x 128 columns of slack
  const long long lf_pp = (long long)E * (d + 2LL * npl + 1) + NP;
  const long long hf_pp = (long long)S * (D + nph + 2);
  const long long keep_pp = (long long)E + E * E;                       // mu_l, Lc survive into the HF stage
  const long long slack = 256LL * (2LL * npl + nph + D + 4);
  const long long wsd = (long long)(ws_bytes / sizeof(double));
  // Two chunk levels: the low-fidelity stage runs over pmL points at a time (its scratch per point is small
  // and its kernels want many columns), the high-fidelity stage over pmH <= pmL points of that chunk
  // (S columns per point); mu_l / Lc of the pmL points survive in between.  Results do not depend on
  // either size (fixed-order reductions per point).
  long long pmL = (wsd - slack) / (keep_pp + lf_pp);
  if (pmL > M) pmL = M;
  if (pmL < 1 || wsd - pmL * keep_pp - slack < hf_pp)
    pmL = (wsd - slack) / (keep_pp + (lf_pp > hf_pp ? lf_pp : hf_pp));   // one level: both stages fit per point
  ARG_CHECK(h, pmL >= 1);
  if (pmL > M) pmL = M;
  if (pmL * E > (1LL << 30) / 4) pmL = (1LL << 28) / E;
  long long pmH = (wsd - pmL * keep_pp - slack) / hf_pp;
  ARG_CHECK(h, pmH >= 1);
  if (pmH > pmL) pmH = pmL;
  double* mu_l = d_ws;                    // (pmL, E)
  double* Lc = mu_l + pmL * E;            // (pmL, E, E)
  double* rest = Lc + pmL * E * E;
  const int prof_saved = h->prof_on;
  for (long long mL = 0; mL < M; mL += pmL) {
    const long long nL = (M - mL < pmL) ? (M - mL) : pmL;
    {  // low-fidelity level: joint posterior at the nL*E locations
      const long long cols = nL * E, cols_pad = (cols + 127) / 128 * 128;
      double* locs = rest;                          // (cols, d)
      double* Ks = locs + cols_pad * d;             // (cols_pad, npl)
      double* T = Ks + cols_pad * npl;              // (npl, cols_pad)
      double* G = T + cols_pad * npl;               // (nL, NP)
      h->prof_on = 0;
      if ((rc = build_locs_launch(h, d_Xtest + mL * d, nL, d, d_offs, E, tau, locs))) return rc;
      if ((rc = cross_gen_launch(h, kl, lf->d_X, lf->N, npl, lf->d_alpha, locs, cols, cols_pad, Ks, mu_l)))
        return rc;
      if ((rc = trmm_store(h, lf->d_W, npl, Ks, cols_pad, T))) return rc;
      if ((rc = group_gram_launch(h, T, npl, cols_pad, nL, E, G))) return rc;
      if ((rc = joint_chol_launch(h, G, d_kab, nL, E, (include_lf_noise ? kl.noise : 0.0) + lf_jitter,
                                  m0 + mL, Lc)))
        return rc;
      h->prof_on = prof_saved;
    }
    for (long long mH = mL; mH < mL + nL; mH += pmH) {   // high-fidelity level over (point, sample) columns
      const long long npts = (mL + nL - mH < pmH) ? (mL + nL - mH) : pmH;
      const long long ncols = npts * S, cols_pad = (ncols + 127) / 128 * 128;
      double* Xq = rest;                            // (cols_pad, D)
      double* mu_c = Xq + cols_pad * D;
      double* ss = mu_c + cols_pad;
      double* Ks = ss + cols_pad;                   // (cols_pad, nph)
      if ((rc = build_mc_rows_joint_launch(h, d_Xtest, mu_l + (mH - mL) * E, Lc + (mH - mL) * E * E, d_eps, seed,
                                           m0, mH, ncols, S, d, E, Xq)))
        return rc;
      if ((rc = cross_gen_launch(h, kh, hf->d_X, hf->N, nph, hf->d_alpha, Xq, ncols, cols_pad, Ks, mu_c)))
        return rc;
      if ((rc = trmm_sumsq(h, hf->d_W, nph, Ks, cols_pad, ss))) return rc;
      if ((rc = finish_var_launch(h, ss, ncols, kh.kdiag, include_hf_noise ? kh.noise : 0.0, ss))) return rc;
      if ((rc = mc_aggregate_launch(h, mu_c, ss, npts, S, d_mean + mH, d_var + mH))) return rc;
    }
  }
  if (h_wsum) {
    if ((rc = wdot_launch(h, d_weights, d_mean, M, h->d_scalars + 20))) return rc;
  }
  if ((rc = fetch_scalars(h, 24))) return rc;
  if (h_wsum) h_wsum[0] += h->h_pinned[20];
  const int bad = h->h_info[1];
  return (bad > 0 && bad < 0x7f7f7f7f) ? bad : 0;   // 1-based global index of the first non-PD joint covariance
}

int mfgp_fill_normal(mfgp_handle_t h, unsigned long long seed, long long first, long long count,
                     double* d_out) {
  ENTER(h);
  ARG_CHECK(h, d_out != nullptr && count >= 0);
  return fill_normal_launch(h, seed, first, count, d_out);
}

int mfgp_argmax(mfgp_handle_t h, const double* d_v, long long C, double* h_val, long long* h_idx) {
  ENTER(h);
  ARG_CHECK(h, d_v != nullptr && C >= 1 && h_val && h_idx);
  int rc = argmax_launch(h, d_v, C, h->d_scalars + 16, reinterpret_cast<long long*>(h->d_scalars + 17));
  if (rc) return rc;
  if ((rc = fetch_scalars(h, 24))) return rc;
  h_val[0] = h->h_pinned[16];
  memcpy(h_idx, h->h_pinned + 17, sizeof(long long));
  return 0;
}

// ---- K8b greedy batch acquisition (math: predict.cu, acq_update_kernel) -----------------------------------------
// Scratch layout in the caller's d_ws, every region on a 128-double boundary: v (C) | kg (C) | R (q, C) |
// X' = [X; a] ((N+1) x MFGP_MAX_D) | k(X, a), W k, u / coefficients (Npad(N+1) each) | pivot record (128) |
// arg-max partials | winner (2) | the prediction chunk for v_0 (the rest).  v and R carry over from call to call.
struct AcqLayout {
  double *v, *kg, *R, *Xp, *krow, *l, *coef, *rec, *partials, *best, *chunk;
  long long chunk_doubles;
};

static long long acq_fixed_doubles(int N, long long C, int q, AcqLayout* L, double* base) {
  const long long np1 = mfgp_padded_n(N + 1);
  long long off = 0;
  auto take = [&](long long n) {
    double* p = base ? base + off : nullptr;
    off += (n + 127) / 128 * 128;
    return p;
  };
  double* v = take(C);
  double* kg = take(C);
  double* R = take((long long)q * C);
  double* Xp = take((long long)(N + 1) * MFGP_MAX_D);
  double* krow = take(np1);
  double* l = take(np1);
  double* coef = take(np1);
  double* rec = take(128);
  double* partials = take(acq_partials_doubles());
  double* best = take(2);
  if (L) *L = AcqLayout{v, kg, R, Xp, krow, l, coef, rec, partials, best, base ? base + off : nullptr, 0};
  return off;
}

static int acq_prepare(mfgp_ctx* h, const mfgp_level_t* gp, const double* d_cands, long long C, int q,
                       double* d_ws, size_t ws_bytes, const double* h_val, const long long* h_idx,
                       const double* h_rec, KParams* kp, AcqLayout* L) {
  int rc = level_kparams(h, gp, kp);
  if (rc) return rc;
  ARG_CHECK(h, gp->d_W != nullptr && d_cands && d_ws && h_val && h_idx && h_rec);
  ARG_CHECK(h, C >= 1 && q >= 1 && q <= MFGP_ACQ_MAX_Q);
  const long long fixed = acq_fixed_doubles(gp->N, C, q, L, d_ws);
  const long long have = (long long)(ws_bytes / sizeof(double));
  ARG_CHECK(h, have >= fixed);
  L->chunk_doubles = have - fixed;
  return 0;
}

// one synchronisation: the winner's value, index and record arrive through mapped pinned memory
static int acq_finish(mfgp_ctx* h, const AcqLayout& L, const double* d_cands, int D, long long C, int nr, int q,
                      double* h_val, long long* h_idx, double* h_rec) {
  int rc = acq_gather_launch(h, L.best, L.v, d_cands, D, L.R, C, nr, q, h->d_batch + 128);
  if (rc) return rc;
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  const double* out = h->h_batch + 128;
  long long idx;
  memcpy(&idx, out + 1, sizeof(idx));
  if (idx < 0) {
    snprintf(h->err, sizeof(h->err), "batch acquisition: no candidate has a comparable variance (NaN)");
    return -1;
  }
  h_val[0] = out[0];
  h_idx[0] = idx;
  memcpy(h_rec, out + 2, (size_t)(1 + D + q) * sizeof(double));
  return 0;
}

size_t mfgp_acq_batch_ws_bytes(int N, long long C, int q) {
  if (N < 1 || C < 1 || q < 1 || q > MFGP_ACQ_MAX_Q) return 0;
  size_t chunk = mfgp_predict_ws_bytes(N, C);          // what mfgp_predict's callers size for C rows, capped
  if (chunk > ((size_t)1 << 30)) chunk = (size_t)1 << 30;
  const size_t least = mfgp_predict_ws_bytes(N, 128);
  if (chunk < least) chunk = least;
  return (size_t)acq_fixed_doubles(N, C, q, nullptr, nullptr) * sizeof(double) + chunk;
}

int mfgp_acq_batch_begin(mfgp_handle_t h, const mfgp_level_t* gp, const double* d_cands, long long C, int q,
                         int include_noise, double* d_ws, size_t ws_bytes, double* h_val, long long* h_idx,
                         double* h_rec) {
  ENTER(h);
  KParams kp;
  AcqLayout L;
  int rc = acq_prepare(h, gp, d_cands, C, q, d_ws, ws_bytes, h_val, h_idx, h_rec, &kp, &L);
  if (rc) return rc;
  // v_0 through mfgp_predict's own chunk loop (same generator, same DMMA contraction, kg as the mean's scratch),
  // finished latent: the clip and the noise are applied only where values are reported or compared
  if ((rc = predict_impl(h, gp, kp, d_cands, C, L.kg, L.v, 0, L.chunk, (size_t)L.chunk_doubles * sizeof(double),
                         true)))
    return rc;
  if ((rc = acq_update_launch(h, nullptr, L.R, C, 0, nullptr, 1.0, L.v, include_noise ? kp.noise : 0.0, L.partials,
                              L.best)))
    return rc;
  return acq_finish(h, L, d_cands, gp->D, C, 0, q, h_val, h_idx, h_rec);
}

int mfgp_acq_batch_step(mfgp_handle_t h, const mfgp_level_t* gp, const double* d_cands, long long C, int q,
                        int include_noise, double jitter, int i, const double* h_rec_in, double* d_ws,
                        size_t ws_bytes, double* h_val, long long* h_idx, double* h_rec) {
  ENTER(h);
  KParams kp;
  AcqLayout L;
  int rc = acq_prepare(h, gp, d_cands, C, q, d_ws, ws_bytes, h_val, h_idx, h_rec, &kp, &L);
  if (rc) return rc;
  ARG_CHECK(h, h_rec_in && i >= 0 && i < q);
  const int N = gp->N, D = gp->D;
  const int npad = mfgp_padded_n(N), npad1 = mfgp_padded_n(N + 1);
  const double rho2 = h_rec_in[0] + kp.noise + JITTER_CONST + jitter;   // v_i(p_i) + s^2
  if (!(rho2 > 0.0)) return i + 1;
  // the pivot's record (a, R[0..i)[p]) to the device through the pinned staging block
  const int nrec = 1 + D + q;
  memcpy(h->h_batch, h_rec_in, (size_t)nrec * sizeof(double));
  CUDA_TRY(h, cudaMemcpyAsync(L.rec, h->h_batch, (size_t)nrec * sizeof(double), cudaMemcpyHostToDevice, h->stream));
  CUDA_TRY(h, cudaMemcpyAsync(L.Xp, gp->d_X, (size_t)N * D * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
  CUDA_TRY(h, cudaMemcpyAsync(L.Xp + (long long)N * D, L.rec + 1, (size_t)D * sizeof(double),
                              cudaMemcpyDeviceToDevice, h->stream));
  // u = K_y^-1 k(X, a), then k(c, a) - k_c^T u for every candidate in one mean-mode pass over X' = [X; a]
  if ((rc = cross_gen_launch(h, kp, gp->d_X, N, npad, gp->d_alpha, L.Xp + (long long)N * D, 1, 1, L.krow, nullptr)))
    return rc;
  if ((rc = kinv_apply_launch(h, gp->d_W, npad, N, L.krow, L.l, L.coef))) return rc;
  if ((rc = acq_coef_launch(h, L.coef, N, npad1, L.coef))) return rc;
  if ((rc = cross_gen_launch(h, kp, L.Xp, N + 1, npad1, L.coef, d_cands, C, C, nullptr, L.kg))) return rc;
  if ((rc = acq_update_launch(h, L.kg, L.R, C, i, L.rec + 1 + D, sqrt(rho2), L.v, include_noise ? kp.noise : 0.0,
                              L.partials, L.best)))
    return rc;
  return acq_finish(h, L, d_cands, D, C, i + 1, q, h_val, h_idx, h_rec);
}

// ---- K8c integrated-variance (ALC) acquisition (math: assemble.cu, alc_reduce_kernel) ---------------------------
// Scratch: Ks_R | Tt_R (Rpad x npad each) | per chunk Ks, Tt_C (chunk x npad each) | G (chunk x Rpad).
constexpr long long ALC_MAX_R = (1LL << 31) - 128;   // Rpad is a GEMM extent (int)

static long long alc_fixed_doubles(int N, long long R) {
  return 2LL * ((R + 127) / 128 * 128) * mfgp_padded_n(N);
}
static long long alc_col_doubles(int N, long long R) { return 2LL * mfgp_padded_n(N) + (R + 127) / 128 * 128; }

size_t mfgp_alc_ws_bytes(int N, long long C, long long R) {
  if (N < 1 || C < 1 || R < 1 || R > ALC_MAX_R) return 0;
  const unsigned long long cap = 1ULL << 30, per_col = 8ULL * alc_col_doubles(N, R);
  const unsigned long long cpad = (unsigned long long)((C + 127) / 128 * 128);
  unsigned long long chunk = cpad > cap / per_col ? cap : per_col * cpad;   // what C columns need, capped
  if (chunk < 128 * per_col) chunk = 128 * per_col;                          // at least one 128-column chunk
  return (size_t)(8ULL * alc_fixed_doubles(N, R) + chunk);
}

int mfgp_alc(mfgp_handle_t h, const mfgp_level_t* gp, const double* d_cands, long long C, const double* d_ref,
             long long R, const double* d_w, double jitter, double* d_alc, double* d_ws, size_t ws_bytes) {
  ENTER(h);
  KParams kp;
  int rc = level_kparams(h, gp, &kp);
  if (rc) return rc;
  ARG_CHECK(h, gp->d_W != nullptr && d_cands && d_ref && d_alc && d_ws);
  ARG_CHECK(h, C >= 1 && R >= 1 && R <= ALC_MAX_R && std::isfinite(jitter) && jitter >= 0.0);
  const int N = gp->N, npad = mfgp_padded_n(N);
  const long long rpad = (R + 127) / 128 * 128, fixed = alc_fixed_doubles(N, R), per_col = alc_col_doubles(N, R);
  const long long have = (long long)(ws_bytes / sizeof(double));
  ARG_CHECK(h, have >= fixed + 128 * per_col);
  long long chunk = whole_waves((have - fixed) / per_col / 128 * 128);
  const long long max_chunk = whole_waves(1LL << 30);   // keeps the chunk a GEMM extent (int) whatever ws_bytes is
  if (chunk > max_chunk) chunk = max_chunk;
  double* KsR = d_ws;
  double* TtR = KsR + rpad * npad;
  double* Ks = TtR + rpad * npad;
  double* TtC = Ks + chunk * npad;
  double* G = TtC + chunk * npad;
  const double s2 = kp.noise + JITTER_CONST + jitter;
  if ((rc = cross_gen_launch(h, kp, gp->d_X, N, npad, gp->d_alpha, d_ref, R, rpad, KsR, nullptr))) return rc;
  if ((rc = trmm_rows(h, gp->d_W, npad, KsR, rpad, TtR))) return rc;
  for (long long c0 = 0; c0 < C; c0 += chunk) {
    const long long ncols = (C - c0 < chunk) ? (C - c0) : chunk;
    const long long cols_pad = (ncols + 127) / 128 * 128;
    const double* Xc = d_cands + c0 * gp->D;
    if ((rc = cross_gen_launch(h, kp, gp->d_X, N, npad, gp->d_alpha, Xc, ncols, cols_pad, Ks, nullptr))) return rc;
    if ((rc = trmm_rows(h, gp->d_W, npad, Ks, cols_pad, TtC))) return rc;
    if ((rc = gemm_nt(h, TtC, npad, TtR, npad, G, rpad, cols_pad, rpad, npad))) return rc;
    if ((rc = alc_reduce_launch(h, kp, d_ref, R, d_w, 1.0 / (double)R, G, rpad, TtC, npad, Xc, ncols, s2,
                                d_alc + c0)))
      return rc;
  }
  return 0;
}

}  // extern "C"

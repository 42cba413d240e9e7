// Shared declarations for the sm_100a kernels behind include/mfgp_b200.h.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <math.h>
#include "../../include/mfgp_b200.h"

#define MFGP_TILE 128            // factor buffers are padded to multiples of this
#define MFGP_NUM_SMS 148

// Kernel hyper-parameters folded into the coefficients the device code needs.
//   K(a,b) = c12 * exp(az * |z_a-z_b|^2 + ax * |x_a-x_b|^2) + s3 * exp(a3 * |x_a-x_b|^2)
// COMPOSITE: c12 = var1*var2, az = -1/(2 len1^2), ax = -1/(2 len2^2), s3 = var3, a3 = -1/(2 len3^2)
// RBF      : c12 = var, az = ax = -1/(2 len^2), s3 = 0   (x = first d columns, z = the rest)
// The device kernels evaluate both exponentials with fastmath.cuh's exp2s(), whose argument is in
// units of ln2/256 and carries the variance as an additive constant:
//   K(a,b) = exp2s(uz*|dz|^2 + ux*|dx|^2 + lc12) + exp2s(u3*|dx|^2 + ls3)      (second term iff s3 != 0)
//   uz = az*256/ln2, ux = ax*256/ln2, u3 = a3*256/ln2, lc12 = log(c12)*256/ln2, ls3 = log(s3)*256/ln2
struct KParams {
  int kind, d, D;
  double c12, az, ax, s3, a3;
  double uz, ux, u3, lc12, ls3;
  double kdiag;   // K(a,a)
  double noise;   // Gaussian_noise.variance
  double theta[8];
  const double* exp_tbl;   // device, 256 doubles: 2^(j/256) (mfgp_ctx::d_exp_tbl)
};

// Point service (predict.cu: point_service_kernel).  Control block in mapped pinned host memory; every flag on its
// own 64-byte line.
struct PointServiceCtl {
  volatile unsigned long long req_seq;   // host -> device: sequence number of the posted question
  unsigned long long pad0[7];
  volatile unsigned long long ack_seq;   // device -> host: last answered question
  unsigned long long pad1[7];
  volatile int stop;                     // host -> device: leave
  int pad2[15];
  volatile int alive;                    // 1 while a service kernel is (being) launched; the kernel clears it on exit
  int pad3[15];
  volatile double x[64];                 // question: query row
  volatile double out[8];                // answer: mean, variance
};
struct PointServiceArgs {
  KParams kh;
  const double* Xh;
  int Nh, npad_h;
  const double* alpha_h;
  const double* Wh;
  int has_lf;
  KParams kl;
  const double* Xl;
  int Nl;
  const double* alpha_l;
  int d, E;
  double tau;
  double offs[96];
  double noise_add;
  unsigned long long idle_ns;
  unsigned long long start_seq;
};

struct mfgp_ctx {
  int device;
  cudaStream_t stream;
  char err[512];
  long long launches;
  // fixed scratch (allocated once in mfgp_create)
  double* d_partials;     // MFGP_PARTIALS doubles: per-block partial sums
  double* d_scalars;      // 64 doubles: results staged for the host
  int* d_info;            // 4 ints: [0] first bad pivot (1-based, 0 = ok)
  double* d_exp_tbl;      // 256 doubles: 2^(j/256), correctly rounded on the host
  double* h_pinned;       // 64 doubles pinned
  int* h_info;            // 4 ints pinned
  // batched objective (mfgp_lml_grad_batch): results are written by the kernel straight into mapped pinned
  // host memory (no copy to enqueue): 16 x 16 doubles + 16 ints, and their device-side addresses
  double* h_batch;
  int* h_batch_info;
  double* d_batch;
  int* d_batch_info;
  cudaEvent_t ev[8];
  // look-ahead Cholesky: a high-priority side stream for the panel (critical-path) kernels and
  // per-panel events ordering it against the caller's stream
  cudaStream_t s_hi;
  cudaStream_t s_mid;                   // medium priority: the bulk updates when the caller's stream carries the
                                        // overlapped triangular inverse (potrf_trtri_padded)
  cudaEvent_t ev_la[3 * 64 + 4];
  // point service (mfgp_point_service_*)
  cudaStream_t s_svc;
  PointServiceCtl* svc_h;               // mapped pinned
  PointServiceCtl* svc_d;               // its device-side address
  PointServiceArgs svc_args;            // kept for relaunches
  int svc_active, svc_width;
  unsigned long long svc_seq;
  long long svc_relaunches;
  // optional per-kernel-class timing (mfgp_profile_enable): event pairs around launches
  int prof_on;
  cudaEvent_t* prof_ev;                 // [MFGP_PROF_CLASSES][MFGP_PROF_POOL][2]
  long long prof_count[16];             // launches seen per class since enable/reset
};

#define MFGP_PROF_CLASSES 10
#define MFGP_PROF_POOL 512
enum { PC_ASSEMBLE = 0, PC_LEAF, PC_GEMM, PC_SOLVE, PC_LAUUM, PC_GRAD, PC_CROSSGEN, PC_TRMM_SUMSQ, PC_MISC, PC_ARGMAX };

static inline void prof_begin(mfgp_ctx* h, int cls) {
  if (!h->prof_on) return;
  long long c = h->prof_count[cls];
  if (c < MFGP_PROF_POOL) cudaEventRecord(h->prof_ev[(cls * MFGP_PROF_POOL + c) * 2], h->stream);
}
static inline void prof_end(mfgp_ctx* h, int cls) {
  if (!h->prof_on) return;
  long long c = h->prof_count[cls]++;
  if (c < MFGP_PROF_POOL) cudaEventRecord(h->prof_ev[(cls * MFGP_PROF_POOL + c) * 2 + 1], h->stream);
}

#define MFGP_PARTIALS (1 << 16)

#define CUDA_TRY(h, expr)                                                          \
  do {                                                                             \
    cudaError_t _e = (expr);                                                       \
    if (_e != cudaSuccess) {                                                       \
      snprintf((h)->err, sizeof((h)->err), "%s:%d %s: %s", __FILE__, __LINE__, #expr, \
               cudaGetErrorString(_e));                                            \
      return -100;                                                                 \
    }                                                                              \
  } while (0)

#define ARG_CHECK(h, cond)                                                         \
  do {                                                                             \
    if (!(cond)) {                                                                 \
      snprintf((h)->err, sizeof((h)->err), "%s:%d bad argument: %s", __FILE__, __LINE__, #cond); \
      return -1;                                                                   \
    }                                                                              \
  } while (0)

#define LAUNCH_CHECK(h)                                                            \
  do {                                                                             \
    (h)->launches++;                                                               \
    cudaError_t _e = cudaGetLastError();                                           \
    if (_e != cudaSuccess) {                                                       \
      snprintf((h)->err, sizeof((h)->err), "%s:%d launch: %s", __FILE__, __LINE__, \
               cudaGetErrorString(_e));                                            \
      return -101;                                                                 \
    }                                                                              \
  } while (0)

static inline int round_up(int n, int m) { return (n + m - 1) / m * m; }

int make_kparams(mfgp_ctx* h, int kind, int D, int d, const double* theta, int P, KParams* kp);

// ---- linalg.cu ---------------------------------------------------------------------------
int linalg_configure(mfgp_ctx* h);
int potrf_padded(mfgp_ctx* h, double* A, double* W, int npad, int nreal);   // nreal <= npad: rest is identity pad
int trtri_padded(mfgp_ctx* h, const double* L, double* W, int npad);
// potrf_padded followed by trtri_padded, with the inverse of the LEADING half started while the factorisation's
// serial tail leaves SMs idle; ev_mid (optional) is recorded where the factorisation is complete
int potrf_trtri_padded(mfgp_ctx* h, double* A, double* W, int npad, int nreal, cudaEvent_t ev_mid);
int lauum_padded(mfgp_ctx* h, const double* W, double* Kinv, int npad);
// tmp = W[:, :]*Ks^T with fused column sum of squares:  out_ss[c] = sum_i (sum_k W[i][k] Ks[c][k])^2
int trmm_sumsq(mfgp_ctx* h, const double* W, int npad, const double* Ks, long long cols_pad,
               double* out_ss);

int small_gp_launch(mfgp_ctx* h, const KParams& kp, const double* X, const double* y, int N, double diag_add,
                    double* A, double* W, double* alpha, double* d_out, int want_grad);
int small_gp_configure(mfgp_ctx* h);
int small_batch_configure(mfgp_ctx* h);
int small_batch_max();
int small_lml_batch_launch(mfgp_ctx* h, const KParams* kps, const double* diag_add, int B, const double* X,
                           const double* y, int N, double* d_out, int* d_info, int want_grad);
int trmm_store(mfgp_ctx* h, const double* W, int npad, const double* Ks, long long cols_pad, double* T);
// Tt = Ks W^T for the rows of Ks (cols_pad x npad, like Tt): the first product of kinv_rows
int trmm_rows(mfgp_ctx* h, const double* W, int npad, const double* Ks, long long cols_pad, double* Tt);
// C (m x n, ld ldc) = A B^T for A (m x k, ld lda) and B (n x k, ld ldb); m, n multiples of 128, k of LEAF
int gemm_nt(mfgp_ctx* h, const double* A, long long lda, const double* B, long long ldb, double* C, long long ldc,
            long long m, long long n, int k);
// Ut = Ks K_y^-1 for the rows of Ks (cols_pad x npad, like Ut and the scratch Tt), Wt = W^T (npad x npad)
int kinv_rows(mfgp_ctx* h, const double* W, const double* Wt, int npad, const double* Ks, long long cols_pad,
              double* Tt, double* Ut);
int transpose_launch(mfgp_ctx* h, const double* A, int n, double* At);   // At = A^T, n x n, n multiple of 32
// C(lower, n x n, ld = n) -= T^T T for T (k x n, ld = ldt); n, k multiples of 128
int syrk_tn_sub(mfgp_ctx* h, const double* T, long long ldt, int k, double* C, int n);
// Z[i][c] = sum_{k<=i} L[i][k] E[k][c]   (L: n x n lower with explicit zeros above the diagonal inside its
// diagonal 128-blocks; E, Z: n x ldc row-major, ldc multiple of 128)
int trmm_right_store(mfgp_ctx* h, const double* L, int n, const double* E, long long ldc, double* Z);

// ---- assemble.cu -------------------------------------------------------------------------
int assemble_configure(mfgp_ctx* h);
int assemble_launch(mfgp_ctx* h, const KParams& kp, const double* X, int N, double diag_add,
                    double* K, long long ldk, int uplo, int npad_identity);
int cross_tile_launch(mfgp_ctx* h, const KParams& kp, const double* X, int N, int npad, const double* alpha,
                      const double* Xq, long long ncols, long long cols_pad, double* Ks, double* mean);
int cross_grad_launch(mfgp_ctx* h, const KParams& kp, const double* X, int N, const double* alpha, const double* Ut,
                      long long ldu, const double* Xq, long long ncols, double* dmean, double* dvar, double* mean,
                      double* quad);
int alc_reduce_launch(mfgp_ctx* h, const KParams& kp, const double* Xr, long long R, const double* w, double w_def,
                      const double* G, long long ldg, const double* Tt, int npad, const double* Xc, long long ncols,
                      double s2, double* alc);
int grad_reduce_launch(mfgp_ctx* h, const KParams& kp, const double* X, int N, const double* Kinv,
                       long long ld, const double* alpha, double* d_out8);

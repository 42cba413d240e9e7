// Blocked FP64 Cholesky (K2), triangular inverse, K^-1 = W^T W (K4) and the O(N^2) solves (K3).
// Replaces GPy.util.linalg.pdinv / dpotrs / dpotri (LAPACK on the CPU) as reached from
// GPRegression construction and every optimiser step (reference src/MFDataFusion.py:93-100,
// src/abstractMFGP.py:131-137).  Everything is lower / row-major on an npad x npad buffer whose
// pad block is the identity (npad multiple of 128).
//
// Recursive formulation so that almost all flops are large DMMA GEMMs (gemm.cuh):
//   potrf(n):  potrf(A11); A21 <- A21 L11^-T (recursive TRSM, leaf = multiply by the 128x128 leaf
//              inverse); A22 -= A21 A21^T (SYRK, lower tiles); potrf(A22)
//   trtri(n):  trtri(11), trtri(22); W21 = -W22 L21 W11
//   lauum:     Kinv = W^T W, one launch over the lower tiles with k >= row0
#include "gemm.cuh"
#include "fastmath.cuh"

namespace {

constexpr int LEAF = 128;
constexpr int LEAF_LD = LEAF + 1;

// One CTA factorises a 128x128 diagonal block and inverts the factor, with the whole block
// REGISTER-resident: thread (ty,tx) of the 16x16 thread grid owns the 2-D cyclic 8x8 element set
// (i = ty+16a, j = tx+16b).  Positions with j <= i hold A -> L; positions with j > i hold the
// accumulators of W = L^-1 transposed (position (r,c), r < c, works on W[c][r]).  Per elimination
// step only column k of that packed matrix goes through shared memory (double-buffered, one
// __syncthreads per step for factor AND inverse); the rank-1 updates are pure register FMAs.
constexpr int LT = 16;   // thread grid edge; 8 = LEAF / LT elements per thread and dimension

// One elimination step does both jobs with ONE barrier: column k of the packed matrix is published
// whole -- rows >= k carry the (unscaled) column of L, rows < k the finished accumulators of W[k][.]
// (contributions to W[k][r] come from steps < k only) -- then every thread applies the Cholesky
// rank-1 update to its lower positions (i, j > k) and the inverse update
//   acc(W[c][r]) += L[c][k] * W[k][r],  W[k][r] = -acc(k,r) / L[k][k]  (r < k),  W[k][k] = 1 / L[k][k]
// to its upper positions (r <= k < c).  128 barriers per leaf instead of 256.
template <int KB>
__device__ __forceinline__ void leaf_fused_block(double (&t)[8][8], double (*col)[LEAF], double* dinv,
                                                 int tx, int ty, int* info, int j0, int nvalid) {
  // columns >= nvalid belong to the identity pad: L = W = I there already, no step needed
  const int kend = min(LT, nvalid - KB * LT);
  for (int ko = 0; ko < kend; ko++) {
    const int k = KB * LT + ko;
    double* buf = col[k & 1];
    if (tx == ko) {   // owners of column k of the packed matrix
#pragma unroll
      for (int a = 0; a < 8; a++) buf[ty + LT * a] = t[a][KB];
    }
    __syncthreads();
    double p = buf[k];
    if (!(p > 0.0)) {   // also catches NaN
      if (tx == 0 && ty == 0 && info[0] == 0) info[0] = j0 + k + 1;
      p = 1.0;
    }
    const double rinv = rsqrt(p);
    if (tx == ko) {   // owners keep the scaled column = column k of L (rows < k keep the W accumulators)
#pragma unroll
      for (int a = KB; a < 8; a++) {
        const int i = ty + LT * a;
        if (i > k) t[a][KB] *= rinv;
        else if (i == k) { t[a][KB] = p * rinv; dinv[k] = rinv; }
      }
    }
    double li[8], lj[8], wr[8];
#pragma unroll
    for (int a = KB; a < 8; a++) li[a] = buf[ty + LT * a] * rinv;       // L[i][k], rows i > k
#pragma unroll
    for (int b = KB; b < 8; b++) lj[b] = buf[tx + LT * b] * rinv;       // L[j][k], columns j > k
#pragma unroll
    for (int a = 0; a <= KB; a++) {                                     // W[k][r], rows r <= k
      const int r = ty + LT * a;
      wr[a] = (r == k) ? rinv : -rinv * buf[r];
    }
#pragma unroll
    for (int a = KB; a < 8; a++) {                                      // Cholesky: lower positions
      if (a == KB && ty <= ko) continue;          // row i <= k
#pragma unroll
      for (int b = KB; b <= a; b++) {
        if (b == KB && tx <= ko) continue;        // column j <= k
        if (a == b && tx > ty) continue;          // strictly upper position
        t[a][b] = fma(-li[a], lj[b], t[a][b]);
      }
    }
#pragma unroll
    for (int a = 0; a <= KB; a++) {                                     // inverse: upper positions r <= k < c
      if (a == KB && ty > ko) continue;           // row r > k
#pragma unroll
      for (int b = KB; b < 8; b++) {
        if (b == KB && tx <= ko) continue;        // column c <= k
        t[a][b] = fma(lj[b], wr[a], t[a][b]);     // acc(W[c][r]) += L[c][k] * W[k][r]
      }
    }
  }
}

__global__ void __launch_bounds__(256, 1)
    leaf_potrf_inv_kernel(double* A, long lda, double* W, long ldw, int* info, int j0, int nvalid) {
  extern __shared__ double S[];   // LEAF x LEAF_LD staging for the coalesced write-out
  __shared__ double col[2][LEAF];
  __shared__ double dinv[LEAF];
  const int tid = threadIdx.x;
  const int tx = tid & (LT - 1), ty = tid >> 4;
  double t[8][8];
#pragma unroll
  for (int a = 0; a < 8; a++)
#pragma unroll
    for (int b = 0; b < 8; b++) {
      const int i = ty + LT * a, j = tx + LT * b;
      t[a][b] = (j <= i) ? A[(long)i * lda + j] : 0.0;
    }
  if (tid < LEAF) dinv[tid] = 1.0;     // pad columns: 1 / L[i][i] = 1
  __syncthreads();
  leaf_fused_block<0>(t, col, dinv, tx, ty, info, j0, nvalid);
  leaf_fused_block<1>(t, col, dinv, tx, ty, info, j0, nvalid);
  leaf_fused_block<2>(t, col, dinv, tx, ty, info, j0, nvalid);
  leaf_fused_block<3>(t, col, dinv, tx, ty, info, j0, nvalid);
  leaf_fused_block<4>(t, col, dinv, tx, ty, info, j0, nvalid);
  leaf_fused_block<5>(t, col, dinv, tx, ty, info, j0, nvalid);
  leaf_fused_block<6>(t, col, dinv, tx, ty, info, j0, nvalid);
  leaf_fused_block<7>(t, col, dinv, tx, ty, info, j0, nvalid);
  __syncthreads();   // dinv complete; col buffers free
  // stage the packed matrix, then write L and W with coalesced rows
#pragma unroll
  for (int a = 0; a < 8; a++)
#pragma unroll
    for (int b = 0; b < 8; b++) S[(ty + LT * a) * LEAF_LD + tx + LT * b] = t[a][b];
  __syncthreads();
  for (int idx = tid; idx < LEAF * LEAF; idx += 256) {
    const int i = idx >> 7, j = idx & 127;
    double l, w;
    if (j < i) {
      l = S[i * LEAF_LD + j];
      w = -dinv[i] * S[j * LEAF_LD + i];   // W[i][j] = -acc(j,i) / L[i][i]
    } else if (j == i) {
      l = S[i * LEAF_LD + i];
      w = dinv[i];
    } else {
      l = 0.0;
      w = 0.0;
    }
    A[(long)i * lda + j] = l;
    W[(long)i * ldw + j] = w;
  }
}


// ---- N <= 128: the whole LML (+ gradient) evaluation in ONE kernel -----------------------------------
// The reference's own problems are tiny (5-30 high-fidelity points, src/gpc/mfgp_gpc.py:10,18-20, refitted
// by up to 7 L-BFGS-B runs per adaptation step), where the chain assemble -> leaf -> solves -> W^T W ->
// gradient reduction -> reduce was eight launches of ~10 us each plus their gaps.  One CTA does it all:
// K_y is assembled straight into the leaf's register tile, factorised and inverted there (steps over
// the identity pad skipped), and alpha, log det, K^-1 = W^T W and the six gradient sums come out of
// shared memory.  Same arithmetic per element as the large-N kernels (exp2s, direct-form distances).
constexpr int SMALL_SMEM_FIXED = (fm::EXP_TBL_DOUBLES + LEAF * LEAF_LD + 6 * LEAF + 64) * 8;

__device__ __forceinline__ void small_kernel_parts(const KParams& kp, const double* sX, int i, int j, unsigned tbl,
                                                   double& rx, double& rz, double& k12, double& k3) {
  rx = 0.0;
  rz = 0.0;
  for (int dd = 0; dd < kp.D; dd++) {
    const double t = sX[dd * LEAF + i] - sX[dd * LEAF + j];
    if (dd < kp.d) rx = fma(t, t, rx);
    else rz = fma(t, t, rz);
  }
  k12 = fm::exp2s(fma(kp.uz, rz, fma(kp.ux, rx, kp.lc12)), tbl);
  k3 = kp.s3 != 0.0 ? fm::exp2s(fma(kp.u3, rx, kp.ls3), tbl) : 0.0;
}

__global__ void __launch_bounds__(256, 1)
    small_gp_kernel(KParams kp, const double* __restrict__ X, const double* __restrict__ y, int N,
                    double diag_add, double* __restrict__ A, double* __restrict__ W,
                    double* __restrict__ alpha, double* __restrict__ out, int* info, int want_grad) {
  extern __shared__ __align__(16) double sm[];
  double* stbl = sm;                                   // exp table (32 KB)
  double* S = stbl + fm::EXP_TBL_DOUBLES;              // [128][129] packed matrix
  double* dinv = S + LEAF * LEAF_LD;                   // [128]
  double* sy = dinv + LEAF;                            // [128]
  double* sv = sy + LEAF;                              // [128]
  double* sal = sv + LEAF;                             // [128]
  double (*col)[LEAF] = reinterpret_cast<double (*)[LEAF]>(sal + LEAF);   // [2][128]... uses 2*LEAF
  double* red = sal + LEAF + 2 * LEAF;                 // [64]
  double* sX = red + 64;                               // [D][128]
  const int tid = threadIdx.x, tx = tid & (LT - 1), ty = tid >> 4;
  const int lane = tid & 31, warp = tid >> 5;
  fm::load_exp_table(stbl, kp.exp_tbl);
  const unsigned tbl = fm::lane_table(stbl);
  for (int idx = tid; idx < LEAF * kp.D; idx += 256) {
    const int r = idx / kp.D, dd = idx - r * kp.D;
    sX[dd * LEAF + r] = r < N ? X[idx] : 0.0;
  }
  if (tid < LEAF) {
    sy[tid] = tid < N ? y[tid] : 0.0;
    dinv[tid] = 1.0;
  }
  __syncthreads();
  // K_y into the packed register tile (lower positions; identity on the pad)
  double t[8][8];
#pragma unroll
  for (int a = 0; a < 8; a++)
#pragma unroll
    for (int b = 0; b < 8; b++) {
      const int i = ty + LT * a, j = tx + LT * b;
      double v = 0.0;
      if (j <= i) {
        if (i < N) {
          double rx, rz, k12, k3;
          small_kernel_parts(kp, sX, i, j, tbl, rx, rz, k12, k3);
          v = k12 + k3 + (i == j ? diag_add : 0.0);
        } else {
          v = (i == j) ? 1.0 : 0.0;
        }
      }
      t[a][b] = v;
    }
  leaf_fused_block<0>(t, col, dinv, tx, ty, info, 0, N);
  leaf_fused_block<1>(t, col, dinv, tx, ty, info, 0, N);
  leaf_fused_block<2>(t, col, dinv, tx, ty, info, 0, N);
  leaf_fused_block<3>(t, col, dinv, tx, ty, info, 0, N);
  leaf_fused_block<4>(t, col, dinv, tx, ty, info, 0, N);
  leaf_fused_block<5>(t, col, dinv, tx, ty, info, 0, N);
  leaf_fused_block<6>(t, col, dinv, tx, ty, info, 0, N);
  leaf_fused_block<7>(t, col, dinv, tx, ty, info, 0, N);
  __syncthreads();
#pragma unroll
  for (int a = 0; a < 8; a++)
#pragma unroll
    for (int b = 0; b < 8; b++) S[(ty + LT * a) * LEAF_LD + tx + LT * b] = t[a][b];
  __syncthreads();
  // upper positions: accumulators -> W itself, S[j][i] = W[i][j] (j < i); then L and W go to global memory
  for (int idx = tid; idx < LEAF * LEAF; idx += 256) {
    const int i = idx >> 7, j = idx & 127;
    if (j < i) S[j * LEAF_LD + i] *= -dinv[i];
  }
  __syncthreads();
  for (int idx = tid; idx < LEAF * LEAF; idx += 256) {
    const int i = idx >> 7, j = idx & 127;
    double l = 0.0, w = 0.0;
    if (j < i) { l = S[i * LEAF_LD + j]; w = S[j * LEAF_LD + i]; }
    else if (j == i) { l = S[i * LEAF_LD + i]; w = dinv[i]; }
    if (!want_grad) A[(long)i * LEAF + j] = l;       // with the gradient, A receives K^-1 below
    W[(long)i * LEAF + j] = w;
  }
  // v = W y, alpha = W^T v (threads 0..127, one row / column each; conflict-free strides)
  if (tid < LEAF) {
    double acc = 0.0;
    if (tid < N) {
      for (int k = 0; k < tid; k++) acc = fma(S[k * LEAF_LD + tid], sy[k], acc);
      acc = fma(dinv[tid], sy[tid], acc);
    }
    sv[tid] = acc;
  }
  __syncthreads();
  if (tid < LEAF) {
    double acc = 0.0;
    if (tid < N) {
      acc = dinv[tid] * sv[tid];
      for (int i = tid + 1; i < N; i++) acc = fma(S[tid * LEAF_LD + i], sv[i], acc);
    }
    sal[tid] = acc;
    alpha[tid] = acc;
  }
  __syncthreads();
  if (warp == 0) {   // log det and y^T alpha, fixed order
    double ld = 0.0, ya = 0.0;
    for (int i = lane; i < N; i += 32) {
      ld -= log(dinv[i]);
      ya = fma(sy[i], sal[i], ya);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      ld += __shfl_xor_sync(0xffffffffu, ld, o);
      ya += __shfl_xor_sync(0xffffffffu, ya, o);
    }
    if (lane == 0) {
      const double logdet = 2.0 * ld;
      out[1] = logdet;
      out[2] = ya;
      out[0] = 0.5 * (-(double)N * 1.8378770664093453 - logdet - ya);
    }
  }
  if (!want_grad) return;
  // K^-1 = W^T W on the lower positions and the six gradient sums in the same sweep
  double G6[6] = {0, 0, 0, 0, 0, 0};
#pragma unroll 1
  for (int a = 0; a < 8; a++) {
    const int i = ty + LT * a;
#pragma unroll 1
    for (int b = 0; b <= a; b++) {
      const int j = tx + LT * b;
      double kin = 0.0;
      if (j <= i) {
        if (i < N) {
          // sum_{k > i} W[k][i] W[k][j] + W[i][i] W[i][j]
          double acc = dinv[i] * (j < i ? S[j * LEAF_LD + i] : dinv[i]);
          for (int k = i + 1; k < N; k++) acc = fma(S[i * LEAF_LD + k], S[j * LEAF_LD + k], acc);
          kin = acc;
          double rx, rz, k12, k3;
          small_kernel_parts(kp, sX, i, j, tbl, rx, rz, k12, k3);
          const double wgt = (i == j) ? 0.5 : 1.0;      // G = 0.5 (aa^T - K^-1); off-diagonal counted twice
          const double G = wgt * fma(sal[i], sal[j], -kin);
          const double gk = G * k12, g3 = G * k3;
          G6[0] += gk;
          G6[1] = fma(gk, rz, G6[1]);
          G6[2] = fma(gk, rx, G6[2]);
          G6[3] += g3;
          G6[4] = fma(g3, rx, G6[4]);
          if (i == j) G6[5] += G;
        } else {
          kin = (i == j) ? 1.0 : 0.0;
        }
        A[(long)i * LEAF + j] = kin;
      } else {
        A[(long)i * LEAF + j] = 0.0;
      }
    }
  }
  // upper blocks of A that the loop above did not visit (b > a) are left as they were: only the lower
  // triangle of K^-1 is defined, as after the large-N path
#pragma unroll
  for (int q = 0; q < 6; q++) {
    double v = G6[q];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0) red[warp * 6 + q] = v;
  }
  __syncthreads();
  if (tid < 6) {
    double v = 0.0;
    for (int w = 0; w < 8; w++) v += red[w * 6 + tid];
    out[8 + tid] = v;
  }
}

// ---- batched-theta objective for N <= 128: one CTA per hyper-parameter vector, only scalars come back ----
// What the optimiser needs from an evaluation is (LML, gradient) -- not the factors.  The reference refits 5-30
// high-fidelity points with 1 + 6 L-BFGS-B runs per adaptation step (src/abstractMFGP.py:131-137,
// src/gpc/mfgp_gpc.py:17-20); the 6 restarts are independent, so their evaluations are batched: B vectors
// in ONE launch (gp.GPRegression drives the restarts in lock-step).  Compared with small_gp_kernel the
// register tile, the staging matrix and every loop are sized by NB = ceil(N / 16) at compile time, the
// exponential uses a plain 2 KB table, and nothing N x N is written to global memory (small_gp_kernel
// writes two full 128 x 128 matrices per evaluation whatever N is).  Same arithmetic per element.
struct SmallTheta {
  double uz, ux, u3, lc12, ls3, s3, diag_add, pad;
};
constexpr int SMALL_BATCH_MAX = 16;
struct SmallBatch {
  SmallTheta th[SMALL_BATCH_MAX];
};

template <int KB, int NB>
__device__ __forceinline__ void small_fused_block(double (&t)[NB][NB], double* col0, double* col1, double* dinv,
                                                  int tx, int ty, int* bad, int nvalid) {
  const int kend = min(LT, nvalid - KB * LT);
  for (int ko = 0; ko < kend; ko++) {
    const int k = KB * LT + ko;
    double* buf = (k & 1) ? col1 : col0;
    if (tx == ko) {
#pragma unroll
      for (int a = 0; a < NB; a++) buf[ty + LT * a] = t[a][KB];
    }
    __syncthreads();
    double p = buf[k];
    if (!(p > 0.0)) {   // also catches NaN
      if (tx == 0 && ty == 0 && bad[0] == 0) bad[0] = k + 1;
      p = 1.0;
    }
    const double rinv = rsqrt(p);
    if (tx == ko) {
#pragma unroll
      for (int a = KB; a < NB; a++) {
        const int i = ty + LT * a;
        if (i > k) t[a][KB] *= rinv;
        else if (i == k) { t[a][KB] = p * rinv; dinv[k] = rinv; }
      }
    }
    double li[NB], lj[NB], wr[NB];
#pragma unroll
    for (int a = KB; a < NB; a++) li[a] = buf[ty + LT * a] * rinv;
#pragma unroll
    for (int b = KB; b < NB; b++) lj[b] = buf[tx + LT * b] * rinv;
#pragma unroll
    for (int a = 0; a <= KB; a++) {
      const int r = ty + LT * a;
      wr[a] = (r == k) ? rinv : -rinv * buf[r];
    }
#pragma unroll
    for (int a = KB; a < NB; a++) {
      if (a == KB && ty <= ko) continue;
#pragma unroll
      for (int b = KB; b <= a; b++) {
        if (b == KB && tx <= ko) continue;
        if (a == b && tx > ty) continue;
        t[a][b] = fma(-li[a], lj[b], t[a][b]);
      }
    }
#pragma unroll
    for (int a = 0; a <= KB; a++) {
      if (a == KB && ty > ko) continue;
#pragma unroll
      for (int b = KB; b < NB; b++) {
        if (b == KB && tx <= ko) continue;
        t[a][b] = fma(lj[b], wr[a], t[a][b]);
      }
    }
  }
}

template <int KB, int NB>
__device__ __forceinline__ void small_eliminate(double (&t)[NB][NB], double* col0, double* col1, double* dinv,
                                                int tx, int ty, int* bad, int nvalid) {
  if constexpr (KB < NB) {
    small_fused_block<KB, NB>(t, col0, col1, dinv, tx, ty, bad, nvalid);
    small_eliminate<KB + 1, NB>(t, col0, col1, dinv, tx, ty, bad, nvalid);
  }
}

template <int NB>
constexpr int small_batch_smem_doubles(int D) {
  return 256 + (NB * 16) * (NB * 16 + 1) + 6 * (NB * 16) + 64 + D * (NB * 16);
}

template <int NB>
__global__ void __launch_bounds__(256, 1)
    small_lml_batch_kernel(SmallBatch params, int D, int d, const double* __restrict__ X,
                           const double* __restrict__ y, int N, const double* __restrict__ gtbl,
                           double* __restrict__ out /* (B, 16) */, int* __restrict__ info /* (B) */,
                           int want_grad) {
  constexpr int NP = NB * 16, LD = NP + 1;
  extern __shared__ __align__(16) double sm[];
  __shared__ int s_bad;
  double* stbl = sm;                 // [256] 2^(j/256)
  double* S = stbl + 256;            // [NP][LD] packed matrix
  double* dinv = S + NP * LD;        // [NP]
  double* sy = dinv + NP;
  double* sv = sy + NP;
  double* sal = sv + NP;
  double* col0 = sal + NP;
  double* col1 = col0 + NP;
  double* red = col1 + NP;           // [64]
  double* sX = red + 64;             // [D][NP]
  const SmallTheta th = params.th[blockIdx.x];
  const int tid = threadIdx.x, tx = tid & (LT - 1), ty = tid >> 4;
  const int lane = tid & 31, warp = tid >> 5;
  stbl[tid] = gtbl[tid];
  for (int idx = tid; idx < NP * D; idx += 256) {
    const int r = idx / D, dd = idx - r * D;
    sX[dd * NP + r] = r < N ? X[idx] : 0.0;
  }
  if (tid < NP) {
    sy[tid] = tid < N ? y[tid] : 0.0;
    dinv[tid] = 1.0;
  }
  if (tid == 0) s_bad = 0;
  __syncthreads();
  const unsigned tbl = (unsigned)__cvta_generic_to_shared(stbl);
  const bool has3 = th.s3 != 0.0;
  auto parts = [&](int i, int j, double& rx, double& rz, double& k12, double& k3) {
    rx = 0.0;
    rz = 0.0;
    for (int dd = 0; dd < D; dd++) {
      const double q = sX[dd * NP + i] - sX[dd * NP + j];
      if (dd < d) rx = fma(q, q, rx);
      else rz = fma(q, q, rz);
    }
    k12 = fm::exp2s_flat(fma(th.uz, rz, fma(th.ux, rx, th.lc12)), tbl);
    k3 = has3 ? fm::exp2s_flat(fma(th.u3, rx, th.ls3), tbl) : 0.0;
  };
  double t[NB][NB];
#pragma unroll
  for (int a = 0; a < NB; a++)
#pragma unroll
    for (int b = 0; b < NB; b++) {
      const int i = ty + LT * a, j = tx + LT * b;
      double v = 0.0;
      if (j <= i) {
        if (i < N) {
          double rx, rz, k12, k3;
          parts(i, j, rx, rz, k12, k3);
          v = k12 + k3 + (i == j ? th.diag_add : 0.0);
        } else {
          v = (i == j) ? 1.0 : 0.0;
        }
      }
      t[a][b] = v;
    }
  small_eliminate<0, NB>(t, col0, col1, dinv, tx, ty, &s_bad, N);
  __syncthreads();
#pragma unroll
  for (int a = 0; a < NB; a++)
#pragma unroll
    for (int b = 0; b < NB; b++) S[(ty + LT * a) * LD + tx + LT * b] = t[a][b];
  __syncthreads();
  // upper positions: accumulators -> W itself, S[j][i] = W[i][j] (j < i)
  for (int idx = tid; idx < NP * NP; idx += 256) {
    const int i = idx / NP, j = idx - i * NP;
    if (j < i) S[j * LD + i] *= -dinv[i];
  }
  __syncthreads();
  if (tid < NP) {   // v = W y
    double acc = 0.0;
    if (tid < N) {
      for (int k = 0; k < tid; k++) acc = fma(S[k * LD + tid], sy[k], acc);
      acc = fma(dinv[tid], sy[tid], acc);
    }
    sv[tid] = acc;
  }
  __syncthreads();
  if (tid < NP) {   // alpha = W^T v
    double acc = 0.0;
    if (tid < N) {
      acc = dinv[tid] * sv[tid];
      for (int i = tid + 1; i < N; i++) acc = fma(S[tid * LD + i], sv[i], acc);
    }
    sal[tid] = acc;
  }
  __syncthreads();
  double* o = out + (long)blockIdx.x * 16;
  if (warp == 0) {   // log det and y^T alpha, fixed order
    double ld = 0.0, ya = 0.0;
    for (int i = lane; i < N; i += 32) {
      ld -= log(dinv[i]);
      ya = fma(sy[i], sal[i], ya);
    }
#pragma unroll
    for (int q = 16; q > 0; q >>= 1) {
      ld += __shfl_xor_sync(0xffffffffu, ld, q);
      ya += __shfl_xor_sync(0xffffffffu, ya, q);
    }
    if (lane == 0) {
      const double logdet = 2.0 * ld;
      o[1] = logdet;
      o[2] = ya;
      o[0] = 0.5 * (-(double)N * 1.8378770664093453 - logdet - ya);
      info[blockIdx.x] = s_bad;
    }
  }
  if (!want_grad) return;
  double G6[6] = {0, 0, 0, 0, 0, 0};
#pragma unroll 1
  for (int a = 0; a < NB; a++) {
    const int i = ty + LT * a;
#pragma unroll 1
    for (int b = 0; b <= a; b++) {
      const int j = tx + LT * b;
      if (j <= i && i < N) {
        // K^-1[i][j] = sum_{k > i} W[k][i] W[k][j] + W[i][i] W[i][j]
        double acc = dinv[i] * (j < i ? S[j * LD + i] : dinv[i]);
        for (int k = i + 1; k < N; k++) acc = fma(S[i * LD + k], S[j * LD + k], acc);
        double rx, rz, k12, k3;
        parts(i, j, rx, rz, k12, k3);
        const double wgt = (i == j) ? 0.5 : 1.0;      // G = 0.5 (aa^T - K^-1); off-diagonal counted twice
        const double G = wgt * fma(sal[i], sal[j], -acc);
        const double gk = G * k12, g3 = G * k3;
        G6[0] += gk;
        G6[1] = fma(gk, rz, G6[1]);
        G6[2] = fma(gk, rx, G6[2]);
        G6[3] += g3;
        G6[4] = fma(g3, rx, G6[4]);
        if (i == j) G6[5] += G;
      }
    }
  }
#pragma unroll
  for (int q = 0; q < 6; q++) {
    double v = G6[q];
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) v += __shfl_xor_sync(0xffffffffu, v, s);
    if (lane == 0) red[warp * 6 + q] = v;
  }
  __syncthreads();
  if (tid < 6) {
    double v = 0.0;
    for (int w = 0; w < 8; w++) v += red[w * 6 + tid];
    o[8 + tid] = v;
  }
}

template <class T>
int tile_count(const dg::GemmParams& p) {
  const int tm = p.M / T::BM, tn = p.N / T::BN;
  return (p.lower_only ? tm * (tm + 1) / 2 : tm * tn) * (p.batch > 1 ? p.batch : 1);
}

// ---- TMA descriptors (cuTensorMapEncodeTiled through the runtime's driver entry point: no -lcuda) --------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_tiled() {
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

// row-major (rows x inner) FP64 matrix, leading dimension ld: boxes of {16 doubles, 128 rows}, 128-byte swizzle
static bool make_map(CUtensorMap* m, const double* base, unsigned long long inner, unsigned long long rows,
                     unsigned long long ld) {
  EncodeTiledFn fn = encode_tiled();
  if (!fn) return false;
  cuuint64_t dims[2] = {inner, rows};
  cuuint64_t strides[1] = {ld * sizeof(double)};
  cuuint32_t box[2] = {dg::tma::BOXK, 128};
  cuuint32_t estr[2] = {1, 1};
  return fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, const_cast<double*>(base), dims, strides, box, estr,
            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// NT product through the TMA kernel (k-contiguous operands, full 128 x 128 tiles on at least one wave).
// Returns 1 if it took the launch.  Measured r02 against the cp.async kernels at N = 16384: potrf 53.8 -> 51.6 ms,
// trtri 44.7 -> 43.6, same bits.
static int try_gemm_tma(mfgp_ctx* h, const dg::GemmParams& p, int cls) {
  const int nodes = p.batch > 1 ? p.batch : 1;
  // operand views: A is (M + node shifts) x K, B is (N + node shifts) x K; the leading dimension bounds k
  const long shift = nodes > 1 ? p.batch_stride : 0;      // elements per node along the diagonal: n * (ld + 1)
  long a_rows_shift = 0, a_k_shift = 0, b_rows_shift = 0, b_k_shift = 0, c_stride = 0;
  if (nodes > 1) {
    // batch_stride = n * (ld + 1) for all three operands (equal leading dimensions): n rows down, n columns right
    if (p.lda != p.ldb || p.lda != p.ldc) return 0;
    const long n = shift / (p.lda + 1);
    if (n * (p.lda + 1) != shift) return 0;
    a_rows_shift = b_rows_shift = a_k_shift = b_k_shift = n;
    c_stride = shift;
  }
  CUtensorMap tmA, tmB;
  const unsigned long long a_rows = (unsigned long long)p.M + (nodes - 1) * a_rows_shift;
  const unsigned long long b_rows = (unsigned long long)p.N + (nodes - 1) * b_rows_shift;
  const unsigned long long kext = (unsigned long long)p.K + (nodes - 1) * a_k_shift;
  if (!make_map(&tmA, p.A, kext, a_rows, p.lda) || !make_map(&tmB, p.B, kext, b_rows, p.ldb)) return 0;
  dg::GemmTmaParams q;
  memset(&q, 0, sizeof(q));
  q.C = p.C; q.ldc = p.ldc; q.M = p.M; q.N = p.N; q.K = p.K; q.alpha = p.alpha; q.beta = p.beta;
  q.lower_only = p.lower_only; q.kb_row = p.kb_row; q.kb_col = p.kb_col; q.ke_row = p.ke_row; q.ke_col = p.ke_col;
  q.batch = p.batch; q.c_batch_stride = c_stride;
  q.a_batch_rows = (int)a_rows_shift; q.a_batch_k = (int)a_k_shift;
  q.b_batch_rows = (int)b_rows_shift; q.b_batch_k = (int)b_k_shift;
  q.neg_init = p.alpha == -1.0 && p.beta == 1.0;
  prof_begin(h, cls);
  dg::gemm_tma_kernel<dg::Big16><<<tile_count<dg::Big16>(p), dg::Big16::THREADS, dg::tma::SMEM_BYTES, h->stream>>>(
      tmA, tmB, q);
  prof_end(h, cls);
  return 1;
}

// row-major FP64 matrix read as an m-contiguous operand X(m, k) = X[k * ld + m]: boxes of {16 m values, 32 k rows}
static bool make_map_mc(CUtensorMap* m, const double* base, unsigned long long m_extent, unsigned long long k_rows,
                        unsigned long long ld) {
  EncodeTiledFn fn = encode_tiled();
  if (!fn) return false;
  cuuint64_t dims[2] = {m_extent, k_rows};
  cuuint64_t strides[1] = {ld * sizeof(double)};
  cuuint32_t box[2] = {16, 32};
  cuuint32_t estr[2] = {1, 1};
  return fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, const_cast<double*>(base), dims, strides, box, estr,
            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// Products with at least one m-contiguous operand (first product of the triangular inverse, K^-1 = W^T W,
// the Gram / right-multiply helpers of the delayed-input MC path) through gemm_tma_mc_kernel.  Returns 1 if it
// took the launch.
template <bool A_KC, bool B_KC>
static int try_gemm_tma_mc(mfgp_ctx* h, const dg::GemmParams& p, int cls) {
  const int nodes = p.batch > 1 ? p.batch : 1;
  long n_shift = 0, c_stride = 0;
  if (nodes > 1) {
    if (p.lda != p.ldb || p.lda != p.ldc) return 0;
    n_shift = p.batch_stride / (p.lda + 1);
    if (n_shift * (p.lda + 1) != p.batch_stride) return 0;
    c_stride = p.batch_stride;
  }
  const unsigned long long a_m = (unsigned long long)p.M + (nodes - 1) * n_shift;
  const unsigned long long b_n = (unsigned long long)p.N + (nodes - 1) * n_shift;
  const unsigned long long kext = (unsigned long long)p.K + (nodes - 1) * n_shift;
  CUtensorMap tmA, tmB;
  const bool okA = A_KC ? make_map(&tmA, p.A, kext, a_m, p.lda) : make_map_mc(&tmA, p.A, a_m, kext, p.lda);
  const bool okB = B_KC ? make_map(&tmB, p.B, kext, b_n, p.ldb) : make_map_mc(&tmB, p.B, b_n, kext, p.ldb);
  if (!okA || !okB) return 0;
  dg::GemmTmaParams q;
  memset(&q, 0, sizeof(q));
  q.C = p.C; q.ldc = p.ldc; q.M = p.M; q.N = p.N; q.K = p.K; q.alpha = p.alpha; q.beta = p.beta;
  q.lower_only = p.lower_only; q.kb_row = p.kb_row; q.kb_col = p.kb_col; q.ke_row = p.ke_row; q.ke_col = p.ke_col;
  q.batch = p.batch; q.c_batch_stride = c_stride;
  q.a_batch_rows = q.a_batch_k = q.b_batch_rows = q.b_batch_k = (int)n_shift;
  prof_begin(h, cls);
  dg::gemm_tma_mc_kernel<dg::Big16, A_KC, B_KC>
      <<<tile_count<dg::Big16>(p), dg::Big16::THREADS, dg::tma::SMEM_BYTES, h->stream>>>(tmA, tmB, q);
  prof_end(h, cls);
  return 1;
}

// Narrow GEMMs (fewer 128x128 tiles than SMs) sit on the critical path of the recursion: run them
// with 64x64 tiles so that four times as many SMs share the work.
// Narrow products of the Cholesky panel (row solves, in-panel updates: fewer 128 x 128 tiles than SMs).  With many
// rows below the panel the bulk update hides the panel, and what these products cost is MACHINE time: full 128 x 128
// TMA tiles (one CTA per 128 rows) do the same flops on a quarter of the SM time of the 64 x 64 / 32 x 128 latency
// tiles, which are kept for the chain-bound tail.  NARROW_BIG_ROWS = rows from which the big tiles are used; measured
// r02 at N = 16384: potrf 50.3 -> 48.7 ms (8192: 49.0, 4096: 48.9, 2048: 49.5, 0: 50.0).
constexpr int NARROW_BIG_ROWS = 6144;

template <bool A_KC, bool B_KC>
int launch_gemm(mfgp_ctx* h, const dg::GemmParams& p, int cls = PC_GEMM) {
  const int big_tiles = tile_count<dg::Big16>(p);
  if (big_tiles <= 0) return 0;
  if (A_KC && B_KC && (big_tiles >= MFGP_NUM_SMS || (p.batch <= 1 && p.M >= NARROW_BIG_ROWS)) &&
      try_gemm_tma(h, p, cls)) {
    LAUNCH_CHECK(h);
    return 0;
  }
  if constexpr (!(A_KC && B_KC)) {
    if (big_tiles >= MFGP_NUM_SMS && try_gemm_tma_mc<A_KC, B_KC>(h, p, cls)) {
      LAUNCH_CHECK(h);
      return 0;
    }
  }
  prof_begin(h, cls);
  if (big_tiles < MFGP_NUM_SMS) {
    dg::gemm_kernel<dg::Small, A_KC, B_KC>
        <<<tile_count<dg::Small>(p), dg::Small::THREADS, dg::Small::SMEM_BYTES, h->stream>>>(p);
  } else {
    dg::gemm_kernel<dg::Big16, A_KC, B_KC>
        <<<big_tiles, dg::Big16::THREADS, dg::Big16::SMEM_BYTES, h->stream>>>(p);
  }
  prof_end(h, cls);
  LAUNCH_CHECK(h);
  return 0;
}

// X <- X * Wl^T in place (X: m x 128, Wl: 128 x 128): every CTA must own all 128 columns of its rows
int launch_trsm_leaf(mfgp_ctx* h, const dg::GemmParams& p) {
  // (in place is safe with the TMA kernel too: a CTA owns all 128 columns of its rows and stores after its last slab)
  if (p.M >= NARROW_BIG_ROWS && try_gemm_tma(h, p, PC_GEMM)) {
    LAUNCH_CHECK(h);
    return 0;
  }
  prof_begin(h, PC_GEMM);
  if (p.M / 128 < MFGP_NUM_SMS) {
    dg::gemm_kernel<dg::Row32, true, true>
        <<<tile_count<dg::Row32>(p), dg::Row32::THREADS, dg::Row32::SMEM_BYTES, h->stream>>>(p);
  } else {
    dg::gemm_kernel<dg::Big16, true, true>
        <<<tile_count<dg::Big16>(p), dg::Big16::THREADS, dg::Big16::SMEM_BYTES, h->stream>>>(p);
  }
  prof_end(h, PC_GEMM);
  LAUNCH_CHECK(h);
  return 0;
}

dg::GemmParams gp(const double* A, long lda, const double* B, long ldb, double* C, long ldc, int m,
                  int n, int k, double alpha, double beta) {
  dg::GemmParams p;
  memset(&p, 0, sizeof(p));
  p.A = A; p.lda = lda; p.B = B; p.ldb = ldb; p.C = C; p.ldc = ldc;
  p.M = m; p.N = n; p.K = k;
  p.alpha = alpha; p.beta = beta;
  return p;
}

inline int split(int n) { return (n / LEAF / 2) * LEAF; }   // first half, multiple of the leaf

// X (m x n at A[r0][j0]) <- X * L^-T, L = A[j0:j0+n, j0:j0+n]; leaf inverses are in W's diagonal blocks
int trsm_rec(mfgp_ctx* h, double* A, double* W, long ld, int r0, int m, int j0, int n) {
  if (n == LEAF) {
    double* X = A + (long)r0 * ld + j0;
    const double* Wl = W + (long)j0 * ld + j0;
    // X[r][c] = sum_k X[r][k] * Wl[c][k]; in place is safe: a CTA owns all 128 columns of its rows
    return launch_trsm_leaf(h, gp(X, ld, Wl, ld, X, ld, m, LEAF, LEAF, 1.0, 0.0));
  }
  int n1 = split(n), n2 = n - n1, rc;
  if ((rc = trsm_rec(h, A, W, ld, r0, m, j0, n1))) return rc;
  // X2 -= X1 * L21^T,  L21 = A[j0+n1 : j0+n, j0 : j0+n1]
  rc = launch_gemm<true, true>(h, gp(A + (long)r0 * ld + j0, ld, A + (long)(j0 + n1) * ld + j0, ld,
                                     A + (long)r0 * ld + j0 + n1, ld, m, n2, n1, -1.0, 1.0));
  if (rc) return rc;
  return trsm_rec(h, A, W, ld, r0, m, j0 + n1, n2);
}

// nreal: rows/columns below it are the identity pad (leaf steps there are skipped)
int potrf_rec(mfgp_ctx* h, double* A, double* W, long ld, int j0, int n, int nreal) {
  if (n == LEAF) {
    const int smem = LEAF * LEAF_LD * 8;
    prof_begin(h, PC_LEAF);
    const int nvalid = nreal - j0 < 0 ? 0 : (nreal - j0 > LEAF ? LEAF : nreal - j0);
    leaf_potrf_inv_kernel<<<1, 256, smem, h->stream>>>(A + (long)j0 * ld + j0, ld,
                                                       W + (long)j0 * ld + j0, ld, h->d_info, j0, nvalid);
    prof_end(h, PC_LEAF);
    LAUNCH_CHECK(h);
    return 0;
  }
  int n1 = split(n), n2 = n - n1, rc;
  if ((rc = potrf_rec(h, A, W, ld, j0, n1, nreal))) return rc;
  if ((rc = trsm_rec(h, A, W, ld, j0 + n1, n2, j0, n1))) return rc;
  // A22 -= L21 L21^T on the lower tiles
  {
    const double* L21 = A + (long)(j0 + n1) * ld + j0;
    dg::GemmParams p = gp(L21, ld, L21, ld, A + (long)(j0 + n1) * ld + j0 + n1, ld, n2, n2, n1, -1.0, 1.0);
    p.lower_only = 1;
    if ((rc = launch_gemm<true, true>(h, p))) return rc;
  }
  return potrf_rec(h, A, W, ld, j0 + n1, n2, nreal);
}

int trtri_rec(mfgp_ctx* h, const double* L, double* W, long ld, int j0, int n) {
  if (n == LEAF) return 0;   // leaf inverse already written by potrf
  int n1 = split(n), n2 = n - n1, rc;
  if ((rc = trtri_rec(h, L, W, ld, j0, n1))) return rc;
  if ((rc = trtri_rec(h, L, W, ld, j0 + n1, n2))) return rc;
  const double* W11 = W + (long)j0 * ld + j0;
  const double* W22 = W + (long)(j0 + n1) * ld + j0 + n1;
  const double* L21 = L + (long)(j0 + n1) * ld + j0;
  double* Tt = W + (long)j0 * ld + j0 + n1;          // n1 x n2 scratch in W's (unused) upper block
  double* W21 = W + (long)(j0 + n1) * ld + j0;
  // Tt[c][r] = sum_{k>=c} W11[k][c] * L21[r][k]         (Tt = (L21 W11)^T)
  {
    dg::GemmParams p = gp(W11, ld, L21, ld, Tt, ld, n1, n2, n1, 1.0, 0.0);
    p.kb_row = 1;
    if ((rc = launch_gemm<false, true>(h, p))) return rc;
  }
  // W21[r][c] = -sum_{k<=r} W22[r][k] * Tt[c][k]
  {
    dg::GemmParams p = gp(W22, ld, Tt, ld, W21, ld, n2, n1, n2, -1.0, 0.0);
    p.ke_row = 1;
    if ((rc = launch_gemm<true, true>(h, p))) return rc;
  }
  return 0;
}

}  // namespace

template <class T, bool A_KC, bool B_KC>
static int configure_gemm(mfgp_ctx* h) {
  CUDA_TRY(h, cudaFuncSetAttribute(dg::gemm_kernel<T, A_KC, B_KC>,
                                   cudaFuncAttributeMaxDynamicSharedMemorySize, T::SMEM_BYTES));
  return 0;
}

int linalg_configure(mfgp_ctx* h) {
  int rc = 0;
  rc |= configure_gemm<dg::Small, true, false>(h);
  rc |= configure_gemm<dg::Big16, true, false>(h);
  rc |= configure_gemm<dg::Small, true, true>(h);
  rc |= configure_gemm<dg::Small, false, true>(h);
  rc |= configure_gemm<dg::Small, false, false>(h);
  rc |= configure_gemm<dg::Row32, true, true>(h);
  if (rc) return -100;
  CUDA_TRY(h, cudaFuncSetAttribute(dg::trmm_sumsq_kernel<dg::Big16>,
                                   cudaFuncAttributeMaxDynamicSharedMemorySize, dg::Big16::SMEM_BYTES));
  CUDA_TRY(h, cudaFuncSetAttribute(dg::trmm_sumsq_tma_kernel<dg::Big16>,
                                   cudaFuncAttributeMaxDynamicSharedMemorySize, dg::tma::SMEM_BYTES));
  CUDA_TRY(h, cudaFuncSetAttribute(dg::gemm_tma_kernel<dg::Big16>,
                                   cudaFuncAttributeMaxDynamicSharedMemorySize, dg::tma::SMEM_BYTES));
  CUDA_TRY(h, cudaFuncSetAttribute(dg::gemm_tma_mc_kernel<dg::Big16, false, true>,
                                   cudaFuncAttributeMaxDynamicSharedMemorySize, dg::tma::SMEM_BYTES));
  CUDA_TRY(h, cudaFuncSetAttribute(dg::gemm_tma_mc_kernel<dg::Big16, false, false>,
                                   cudaFuncAttributeMaxDynamicSharedMemorySize, dg::tma::SMEM_BYTES));
  CUDA_TRY(h, cudaFuncSetAttribute(dg::gemm_tma_mc_kernel<dg::Big16, true, false>,
                                   cudaFuncAttributeMaxDynamicSharedMemorySize, dg::tma::SMEM_BYTES));
  rc |= configure_gemm<dg::Big16, true, true>(h);
  rc |= configure_gemm<dg::Big16, false, true>(h);
  rc |= configure_gemm<dg::Big16, false, false>(h);
  if (rc) return -100;
  CUDA_TRY(h, cudaFuncSetAttribute(leaf_potrf_inv_kernel,
                                   cudaFuncAttributeMaxDynamicSharedMemorySize, LEAF * LEAF_LD * 8));
  return 0;
}

// Right-looking panels with look-ahead on top of the recursion.  Panel p (NB columns) is factorised
// and its rows solved on the high-priority stream (the latency-bound chain of leaf kernels and narrow
// GEMMs), which then applies panel p to the NEXT panel's block column only; the bulk of panel p's
// trailing update runs on the caller's stream and overlaps the critical path of panel p+1.
//   la[p]   (s_hi)  : A[next block column] -= L21 L21[next rows]^T      waits bulk[p-1] (same tiles)
//   bulk[p] (s_main): A[beyond next block column, lower] -= L21 L21^T   waits trsm[p]
constexpr int LA_MIN = 4096;    // below this the plain recursion is as fast
constexpr int LA_MAXP = 64;
// Panel width, measured at N = 16384: 512 -> 55.1 ms, 768 -> 55.4, 1024 -> 56.3, 2048 -> 61.2 (profiles/r01_notes.md)
// (r02, with the big-tile policy for hidden panels: N = 16384: 512 -> 49.0 ms, 640 -> 49.0, 768 -> 49.4, 1024 -> 50.0;
//  N = 32768: 512 -> 353.6 ms, 1024 -> 344.8)
static int la_nb(int npad) { return npad < 24576 ? 512 : 1024; }
// The panels run to the last column.  Handing the remaining columns to the plain recursion was measured at
// N = 16384 (profiles/r02_potrf_tail.txt), by the number of remaining columns: never -> 53.8 ms, 2048 -> 53.9,
// 4096 -> 54.6, 6144 -> 56.0, 8192 -> 57.8: the recursion loses at every size (its half-size TRSM / SYRK expose
// MORE serial leaf chain, not less).

// The panel's critical path, 128 columns at a time (left-looking inside the panel): leaf -> ONE in-place
// multiply of ALL rows below by the leaf inverse -> ONE update of the next 128-column block by the panel
// columns factorised so far.  12 launches per 512-column panel against 20 for potrf_rec + trsm_rec (whose
// recursion buys nothing here: every one of its GEMMs is narrower than the machine, so each costs a launch
// latency whatever its size), i.e. a shorter serial chain wherever the bulk update no longer hides it.
static int panel_chain(mfgp_ctx* h, double* A, double* W, long ld, int c0, int w, int npad, int nreal) {
  int rc = 0;
  for (int j = 0; j < w && rc == 0; j += LEAF) {
    const int cj = c0 + j;
    if ((rc = potrf_rec(h, A, W, ld, cj, LEAF, nreal))) break;
    const int r0 = cj + LEAF, mr = npad - r0;
    if (mr <= 0) break;
    double* X = A + (long)r0 * ld + cj;
    if ((rc = launch_trsm_leaf(h, gp(X, ld, W + (long)cj * ld + cj, ld, X, ld, mr, LEAF, LEAF, 1.0, 0.0)))) break;
    if (j + LEAF < w) {
      // A[r0:, r0:r0+128] -= A[r0:, c0:r0] * A[r0:r0+128, c0:r0]^T   (K = j + 128)
      const double* P = A + (long)r0 * ld + c0;
      rc = launch_gemm<true, true>(h, gp(P, ld, P, ld, A + (long)r0 * ld + r0, ld, mr, LEAF, j + LEAF, -1.0, 1.0));
    }
  }
  return rc;
}

// s_bulk: stream of the bulk updates (the caller's, or s_mid when the caller's stream is to carry other work
// meanwhile -- then `join` is false and the caller of this function orders its stream after ev_la[3*LA_MAXP+1]
// (chain) and ev_la[3*LA_MAXP+2] (bulk) itself).
static int potrf_lookahead(mfgp_ctx* h, double* A, double* W, int npad, int nreal, cudaStream_t s_bulk = nullptr,
                           bool join = true) {
  const long ld = npad;
  cudaStream_t s_caller = h->stream, s_hi = h->s_hi;
  cudaStream_t s_main = s_bulk ? s_bulk : s_caller;
  cudaEvent_t* ev_trsm = h->ev_la;
  cudaEvent_t* ev_bulk = h->ev_la + LA_MAXP;
  cudaEvent_t ev_start = h->ev_la[3 * LA_MAXP], ev_end = h->ev_la[3 * LA_MAXP + 1];
  const int LA_NB = la_nb(npad);
  int rc = 0;
  bool bulk_pending = false;
  CUDA_TRY(h, cudaEventRecord(ev_start, s_caller));
  CUDA_TRY(h, cudaStreamWaitEvent(s_hi, ev_start, 0));
  if (s_main != s_caller) CUDA_TRY(h, cudaStreamWaitEvent(s_main, ev_start, 0));
  const int P = (npad + LA_NB - 1) / LA_NB;
  for (int p = 0; p < P && rc == 0; p++) {
    const int c0 = p * LA_NB;
    const int w = (npad - c0 < LA_NB) ? npad - c0 : LA_NB;
    const int m = npad - c0 - w;
    h->stream = s_hi;
    if ((rc = panel_chain(h, A, W, ld, c0, w, npad, nreal))) break;
    if (m > 0) {
      CUDA_TRY(h, cudaEventRecord(ev_trsm[p], s_hi));
      const int w2 = m < LA_NB ? m : LA_NB;
      const double* L21 = A + (long)(c0 + w) * ld + c0;
      if (bulk_pending) CUDA_TRY(h, cudaStreamWaitEvent(s_hi, ev_bulk[p - 1], 0));
      // look-ahead: rows c0+w.., columns [c0+w, c0+w+w2)
      rc = launch_gemm<true, true>(h, gp(L21, ld, L21, ld, A + (long)(c0 + w) * ld + c0 + w, ld, m, w2, w,
                                         -1.0, 1.0));
      if (rc) break;
      const int m2 = m - w2;
      bulk_pending = false;
      if (m2 > 0) {
        h->stream = s_main;
        CUDA_TRY(h, cudaStreamWaitEvent(s_main, ev_trsm[p], 0));
        const double* L2 = A + (long)(c0 + w + w2) * ld + c0;
        dg::GemmParams q = gp(L2, ld, L2, ld, A + (long)(c0 + w + w2) * ld + c0 + w + w2, ld, m2, m2, w, -1.0, 1.0);
        q.lower_only = 1;
        rc = launch_gemm<true, true>(h, q);
        if (rc) break;
        CUDA_TRY(h, cudaEventRecord(ev_bulk[p], s_main));
        bulk_pending = true;
      }
    }
  }
  h->stream = s_caller;
  cudaEventRecord(ev_end, s_hi);
  if (s_main != s_caller) cudaEventRecord(h->ev_la[3 * LA_MAXP + 2], s_main);
  if (join || rc) {
    cudaStreamWaitEvent(s_caller, ev_end, 0);
    if (s_main != s_caller) cudaStreamWaitEvent(s_caller, h->ev_la[3 * LA_MAXP + 2], 0);
  }
  return rc;
}

int potrf_padded(mfgp_ctx* h, double* A, double* W, int npad, int nreal) {
  ARG_CHECK(h, npad > 0 && npad % LEAF == 0);
  CUDA_TRY(h, cudaMemsetAsync(h->d_info, 0, 4 * sizeof(int), h->stream));
  if (h->s_hi && npad >= LA_MIN && npad <= la_nb(npad) * LA_MAXP) {
    cudaStream_t caller = h->stream;
    const int rc = potrf_lookahead(h, A, W, npad, nreal);
    h->stream = caller;   // also on the error paths inside
    return rc;
  }
  return potrf_rec(h, A, W, npad, 0, npad, nreal);
}

// Level-synchronous form of trtri_rec for npad = 128 * 2^q: the nodes of one level are independent and
// equally shaped, so each level is TWO launches over all of its nodes (14 launches at N = 16384
// instead of 254); the deep levels, whose single nodes fill only a fraction of the SMs, then run as
// one grid.
// Levels n_first .. nsub of the nodes inside the diagonal block [off, off + nsub) (ld = npad).
static int trtri_levels_range(mfgp_ctx* h, const double* L, double* W, int npad, int off, int nsub, int n_first) {
  const long ld = npad;
  const long o = (long)off * (ld + 1);
  int rc;
  for (int n = n_first; n <= nsub; n *= 2) {
    const int n1 = n / 2, nodes = nsub / n;
    const long stride = (long)n * (ld + 1);
    const double* W11 = W + o;
    const double* W22 = W + o + (long)n1 * ld + n1;
    const double* L21 = L + o + (long)n1 * ld;
    double* Tt = W + o + n1;              // n1 x n1 scratch in W's (unused) upper block
    double* W21 = W + o + (long)n1 * ld;
    {  // Tt[c][r] = sum_{k>=c} W11[k][c] * L21[r][k]
      dg::GemmParams p = gp(W11, ld, L21, ld, Tt, ld, n1, n1, n1, 1.0, 0.0);
      p.kb_row = 1;
      p.batch = nodes;
      p.batch_stride = stride;
      if ((rc = launch_gemm<false, true>(h, p))) return rc;
    }
    {  // W21[r][c] = -sum_{k<=r} W22[r][k] * Tt[c][k]
      dg::GemmParams p = gp(W22, ld, Tt, ld, W21, ld, n1, n1, n1, -1.0, 0.0);
      p.ke_row = 1;
      p.batch = nodes;
      p.batch_stride = stride;
      if ((rc = launch_gemm<true, true>(h, p))) return rc;
    }
  }
  return 0;
}

static int trtri_levels(mfgp_ctx* h, const double* L, double* W, int npad) {
  return trtri_levels_range(h, L, W, npad, 0, npad, 2 * LEAF);
}

int trtri_padded(mfgp_ctx* h, const double* L, double* W, int npad) {
  ARG_CHECK(h, npad > 0 && npad % LEAF == 0);
  const int m = npad / LEAF;
  if ((m & (m - 1)) == 0) return trtri_levels(h, L, W, npad);
  return trtri_rec(h, L, W, npad, 0, npad);
}

// Factorise and invert with the inverse of the leading half overlapped with the factorisation's tail.  The last
// ~6000 columns of the look-ahead Cholesky are bound by the serial panel chain (profiles/r02_potrf_experiments.txt):
// the trailing updates no longer fill the machine.  The triangular inverse of the LEADING half only needs
// L[0:n/2, 0:n/2], final once the panel ending at n/2 has been solved, so its GEMMs (1/8 of the inverse's flops
// at n = 16384) go to the caller's stream -- lowest priority -- right behind that panel's event, while the bulk
// updates move to a medium-priority stream and the chain keeps the high-priority one.  Same products on the same
// data as potrf_padded + trtri_padded; a level batched over half of the matrix may fall below one wave of tiles
// and then takes another GEMM kernel than the level batched over the whole matrix, so the two schedules agree to
// round-off.
int potrf_trtri_padded(mfgp_ctx* h, double* A, double* W, int npad, int nreal, cudaEvent_t ev_mid) {
  const int m = npad / LEAF;
  int rc;
  const bool la = h->s_hi && npad >= LA_MIN && npad <= la_nb(npad) * LA_MAXP;
  const int half = npad / 2;
  if (!(la && h->s_mid && (m & (m - 1)) == 0 && npad >= 8192 && half % la_nb(npad) == 0)) {
    if ((rc = potrf_padded(h, A, W, npad, nreal))) return rc;
    if (ev_mid) CUDA_TRY(h, cudaEventRecord(ev_mid, h->stream));
    return trtri_padded(h, A, W, npad);
  }
  ARG_CHECK(h, npad > 0 && npad % LEAF == 0);
  CUDA_TRY(h, cudaMemsetAsync(h->d_info, 0, 4 * sizeof(int), h->stream));
  cudaStream_t caller = h->stream;
  rc = potrf_lookahead(h, A, W, npad, nreal, h->s_mid, false);
  h->stream = caller;
  if (rc) return rc;
  // leading half: its last panel is panel half / NB - 1, whose chain (and row solves) end at ev_trsm of that panel
  const int p_half = half / la_nb(npad) - 1;
  CUDA_TRY(h, cudaStreamWaitEvent(caller, h->ev_la[p_half], 0));
  if ((rc = trtri_levels_range(h, A, W, npad, 0, half, 2 * LEAF))) return rc;
  CUDA_TRY(h, cudaStreamWaitEvent(caller, h->ev_la[3 * LA_MAXP + 1], 0));
  CUDA_TRY(h, cudaStreamWaitEvent(caller, h->ev_la[3 * LA_MAXP + 2], 0));
  if (ev_mid) CUDA_TRY(h, cudaEventRecord(ev_mid, caller));
  if ((rc = trtri_levels_range(h, A, W, npad, half, half, 2 * LEAF))) return rc;
  return trtri_levels_range(h, A, W, npad, 0, npad, npad);
}

int lauum_padded(mfgp_ctx* h, const double* W, double* Kinv, int npad) {
  ARG_CHECK(h, npad > 0 && npad % LEAF == 0);
  // Kinv[i][j] = sum_{k >= max(i,j)} W[k][i] * W[k][j]; lower tiles have row0 >= col0
  dg::GemmParams p = gp(W, npad, W, npad, Kinv, npad, npad, npad, npad, 1.0, 0.0);
  p.lower_only = 1;
  p.kb_row = 1;
  return launch_gemm<false, false>(h, p, PC_LAUUM);
}

// T[i][c] = sum_{k<=i} W[i][k] * Ks[c][k]   (T: npad x cols_pad, row-major, ld = cols_pad)
int trmm_store(mfgp_ctx* h, const double* W, int npad, const double* Ks, long long cols_pad, double* T) {
  ARG_CHECK(h, npad % LEAF == 0 && cols_pad % dg::Big16::BN == 0 && cols_pad < (1LL << 31));
  if (cols_pad == 0) return 0;
  dg::GemmParams p = gp(W, npad, Ks, npad, T, cols_pad, npad, (int)cols_pad, npad, 1.0, 0.0);
  p.ke_row = 1;
  return launch_gemm<true, true>(h, p, PC_MISC);
}

// Both products are NT (k-contiguous operands): the cp.async and TMA kernels that launch_gemm picks between share
// one accumulation order, so a row's result does not depend on how many rows share the call.  (U = W^T T as a TT
// product would go through gemm_tma_mc_kernel from one wave of tiles on, whose k order differs.)
//   Tt[c][i] = sum_{k<=i} Ks[c][k] W[i][k],   Ut[c][k] = sum_{i>=k} Tt[c][i] Wt[k][i]
int trmm_rows(mfgp_ctx* h, const double* W, int npad, const double* Ks, long long cols_pad, double* Tt) {
  ARG_CHECK(h, npad % LEAF == 0 && cols_pad % dg::Big16::BM == 0 && cols_pad < (1LL << 31));
  if (cols_pad == 0) return 0;
  dg::GemmParams p = gp(Ks, npad, W, npad, Tt, npad, (int)cols_pad, npad, npad, 1.0, 0.0);
  p.ke_col = 1;
  return launch_gemm<true, true>(h, p, PC_MISC);
}

int kinv_rows(mfgp_ctx* h, const double* W, const double* Wt, int npad, const double* Ks, long long cols_pad,
              double* Tt, double* Ut) {
  int rc = trmm_rows(h, W, npad, Ks, cols_pad, Tt);
  if (rc || cols_pad == 0) return rc;
  dg::GemmParams p = gp(Tt, npad, Wt, npad, Ut, npad, (int)cols_pad, npad, npad, 1.0, 0.0);
  p.kb_col = 1;
  return launch_gemm<true, true>(h, p, PC_MISC);
}

// C[r][c] = sum_k A[r][k] B[c][k]: a plain NT product, so an entry depends only on its two operand rows
int gemm_nt(mfgp_ctx* h, const double* A, long long lda, const double* B, long long ldb, double* C, long long ldc,
            long long m, long long n, int k) {
  ARG_CHECK(h, m % dg::Big16::BM == 0 && n % dg::Big16::BN == 0 && k % LEAF == 0);
  ARG_CHECK(h, m < (1LL << 31) && n < (1LL << 31));
  if (m == 0 || n == 0) return 0;
  return launch_gemm<true, true>(h, gp(A, (long)lda, B, (long)ldb, C, (long)ldc, (int)m, (int)n, k, 1.0, 0.0),
                                 PC_GEMM);
}

__global__ void transpose_kernel(const double* __restrict__ A, int n, double* __restrict__ At) {
  __shared__ double t[32][33];
  const long bx = (long)blockIdx.x * 32, by = (long)blockIdx.y * 32;
  for (int r = threadIdx.y; r < 32; r += 8) t[r][threadIdx.x] = A[(by + r) * n + bx + threadIdx.x];
  __syncthreads();
  for (int r = threadIdx.y; r < 32; r += 8) At[(bx + r) * n + by + threadIdx.x] = t[threadIdx.x][r];
}

int transpose_launch(mfgp_ctx* h, const double* A, int n, double* At) {
  ARG_CHECK(h, n % 32 == 0);
  prof_begin(h, PC_MISC);
  transpose_kernel<<<dim3(n / 32, n / 32), dim3(32, 8), 0, h->stream>>>(A, n, At);
  prof_end(h, PC_MISC);
  LAUNCH_CHECK(h);
  return 0;
}

int syrk_tn_sub(mfgp_ctx* h, const double* T, long long ldt, int k, double* C, int n) {
  ARG_CHECK(h, n % LEAF == 0 && k % LEAF == 0 && ldt >= n);
  // C[i][j] -= sum_r T[r][i] * T[r][j] on the lower tiles
  dg::GemmParams p = gp(T, ldt, T, ldt, C, n, n, n, k, -1.0, 1.0);
  p.lower_only = 1;
  return launch_gemm<false, false>(h, p, PC_MISC);
}

int trmm_right_store(mfgp_ctx* h, const double* L, int n, const double* E, long long ldc, double* Z) {
  ARG_CHECK(h, n % LEAF == 0 && ldc % dg::Big16::BN == 0 && ldc < (1LL << 31));
  dg::GemmParams p = gp(L, n, E, ldc, Z, ldc, n, (int)ldc, n, 1.0, 0.0);
  p.ke_row = 1;
  return launch_gemm<true, false>(h, p, PC_MISC);
}

int trmm_sumsq(mfgp_ctx* h, const double* W, int npad, const double* Ks, long long cols_pad,
               double* out_ss) {
  ARG_CHECK(h, npad % LEAF == 0 && cols_pad % dg::Big16::BN == 0);
  if (cols_pad == 0) return 0;
  // TMA operands, measured r02: 2.42 -> 2.27 ms per 75 776 x 1024 launch, bit-identical sums
  if (cols_pad < (1LL << 31)) {
    CUtensorMap tmW, tmK;
    if (make_map(&tmW, W, npad, npad, npad) && make_map(&tmK, Ks, npad, (unsigned long long)cols_pad, npad)) {
      prof_begin(h, PC_TRMM_SUMSQ);
      dg::trmm_sumsq_tma_kernel<dg::Big16><<<(unsigned)(cols_pad / dg::Big16::BN), dg::Big16::THREADS,
                                             dg::tma::SMEM_BYTES, h->stream>>>(tmW, tmK, npad, out_ss);
      prof_end(h, PC_TRMM_SUMSQ);
      LAUNCH_CHECK(h);
      return 0;
    }
  }
  prof_begin(h, PC_TRMM_SUMSQ);
  dg::trmm_sumsq_kernel<dg::Big16><<<(unsigned)(cols_pad / dg::Big16::BN), dg::Big16::THREADS,
                                     dg::Big16::SMEM_BYTES, h->stream>>>(W, npad, Ks, out_ss);
  prof_end(h, PC_TRMM_SUMSQ);
  LAUNCH_CHECK(h);
  return 0;
}


// N <= 128: one fused launch (see small_gp_kernel).  d_A, d_W are 128 x 128 (ld 128), d_alpha 128;
// d_out: [0..2] = {LML, logdet, y^T alpha}, [8..13] = the six gradient sums (want_grad).
int small_gp_launch(mfgp_ctx* h, const KParams& kp, const double* X, const double* y, int N, double diag_add,
                    double* A, double* W, double* alpha, double* d_out, int want_grad) {
  ARG_CHECK(h, N >= 1 && N <= LEAF);
  const size_t smem = SMALL_SMEM_FIXED + (size_t)kp.D * LEAF * sizeof(double);
  CUDA_TRY(h, cudaMemsetAsync(h->d_info, 0, 4 * sizeof(int), h->stream));
  prof_begin(h, PC_LEAF);
  small_gp_kernel<<<1, 256, smem, h->stream>>>(kp, X, y, N, diag_add, A, W, alpha, d_out, h->d_info, want_grad);
  prof_end(h, PC_LEAF);
  LAUNCH_CHECK(h);
  return 0;
}

int small_gp_configure(mfgp_ctx* h) {
  CUDA_TRY(h, cudaFuncSetAttribute(small_gp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   SMALL_SMEM_FIXED + MFGP_MAX_D * LEAF * (int)sizeof(double)));
  return 0;
}


// ---- batched-theta objective (see small_lml_batch_kernel) ----------------------------------------------
template <int NB>
static int small_batch_run(mfgp_ctx* h, const SmallBatch& sb, int B, int D, int d, const double* X, const double* y,
                           int N, double* d_out, int* d_info, int want_grad) {
  const size_t smem = (size_t)small_batch_smem_doubles<NB>(D) * sizeof(double);
  prof_begin(h, PC_LEAF);
  small_lml_batch_kernel<NB><<<B, 256, smem, h->stream>>>(sb, D, d, X, y, N, h->d_exp_tbl, d_out, d_info, want_grad);
  prof_end(h, PC_LEAF);
  LAUNCH_CHECK(h);
  return 0;
}

int small_batch_max() { return SMALL_BATCH_MAX; }

// kps: B <= SMALL_BATCH_MAX parameter sets; diag_add[b] = noise + 1e-8 + jitter.  d_out: (B, 16) doubles,
// [0..2] = {LML, logdet, y^T alpha}, [8..13] = the six gradient sums; d_info: (B) first bad pivot or 0.
int small_lml_batch_launch(mfgp_ctx* h, const KParams* kps, const double* diag_add, int B, const double* X,
                           const double* y, int N, double* d_out, int* d_info, int want_grad) {
  ARG_CHECK(h, N >= 1 && N <= LEAF && B >= 1 && B <= SMALL_BATCH_MAX);
  SmallBatch sb;
  memset(&sb, 0, sizeof(sb));
  for (int b = 0; b < B; b++) {
    sb.th[b].uz = kps[b].uz; sb.th[b].ux = kps[b].ux; sb.th[b].u3 = kps[b].u3;
    sb.th[b].lc12 = kps[b].lc12; sb.th[b].ls3 = kps[b].ls3; sb.th[b].s3 = kps[b].s3;
    sb.th[b].diag_add = diag_add[b];
  }
  const int D = kps[0].D, d = kps[0].d;
  switch ((N + LT - 1) / LT) {
    case 1: return small_batch_run<1>(h, sb, B, D, d, X, y, N, d_out, d_info, want_grad);
    case 2: return small_batch_run<2>(h, sb, B, D, d, X, y, N, d_out, d_info, want_grad);
    case 3: return small_batch_run<3>(h, sb, B, D, d, X, y, N, d_out, d_info, want_grad);
    case 4: return small_batch_run<4>(h, sb, B, D, d, X, y, N, d_out, d_info, want_grad);
    case 5: return small_batch_run<5>(h, sb, B, D, d, X, y, N, d_out, d_info, want_grad);
    case 6: return small_batch_run<6>(h, sb, B, D, d, X, y, N, d_out, d_info, want_grad);
    case 7: return small_batch_run<7>(h, sb, B, D, d, X, y, N, d_out, d_info, want_grad);
    default: return small_batch_run<8>(h, sb, B, D, d, X, y, N, d_out, d_info, want_grad);
  }
}

template <int NB>
static int small_batch_cfg(mfgp_ctx* h) {
  CUDA_TRY(h, cudaFuncSetAttribute(small_lml_batch_kernel<NB>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   small_batch_smem_doubles<NB>(MFGP_MAX_D) * (int)sizeof(double)));
  return 0;
}

int small_batch_configure(mfgp_ctx* h) {
  int rc = 0;
  rc |= small_batch_cfg<1>(h); rc |= small_batch_cfg<2>(h); rc |= small_batch_cfg<3>(h); rc |= small_batch_cfg<4>(h);
  rc |= small_batch_cfg<5>(h); rc |= small_batch_cfg<6>(h); rc |= small_batch_cfg<7>(h); rc |= small_batch_cfg<8>(h);
  return rc ? -100 : 0;
}

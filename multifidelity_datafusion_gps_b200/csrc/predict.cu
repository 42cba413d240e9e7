// K6 prediction, K7 Monte-Carlo propagation, K8 acquisition argmax, and the O(N^2) solve kernels.
//
// K6 replaces GP.predict -> Posterior._raw_predict (reference src/MFDataFusion.py:156,
// src/abstractMFGP.py:104): the cross-covariance block is generated on the fly in column chunks
// (never an N x M matrix in HBM beyond one chunk), the mean is reduced while it is generated, and
// the variance comes from tmp = W Kx as a DMMA GEMM with a fused column sum-of-squares epilogue.
#include "common.cuh"
#include "fastmath.cuh"

namespace {

__device__ __forceinline__ double kernel_eval(const KParams& kp, const double* __restrict__ q,
                                              const double* __restrict__ xk) {
  double rx = 0.0, rz = 0.0;
  for (int dd = 0; dd < kp.d; dd++) {
    double t = q[dd] - xk[dd];
    rx = fma(t, t, rx);
  }
  for (int dd = kp.d; dd < kp.D; dd++) {
    double t = q[dd] - xk[dd];
    rz = fma(t, t, rz);
  }
  double v = kp.c12 * exp(fma(kp.az, rz, kp.ax * rx));
  if (kp.s3 != 0.0) v = fma(kp.s3, exp(kp.a3 * rx), v);
  return v;
}

// One warp per query column c: Ks[c][k] = K(q_c, X_k) for k < N (0 on the pad), mean[c] = Ks[c].alpha
__global__ void __launch_bounds__(256)
    cross_gen_kernel(KParams kp, const double* __restrict__ X, int N, int npad,
                     const double* __restrict__ alpha, const double* __restrict__ Xq,
                     long long ncols, long long cols_pad, double* __restrict__ Ks,
                     double* __restrict__ mean) {
  const int lane = threadIdx.x & 31;
  const long long c = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (c >= cols_pad) return;
  double* row = Ks ? Ks + c * npad : nullptr;
  if (c >= ncols) {
    if (row)
      for (int k = lane; k < npad; k += 32) row[k] = 0.0;
    return;
  }
  double q[MFGP_MAX_D];
  for (int dd = 0; dd < kp.D; dd++) q[dd] = Xq[c * kp.D + dd];
  double acc = 0.0;
  for (int k = lane; k < npad; k += 32) {
    double v = 0.0;
    if (k < N) {
      v = kernel_eval(kp, q, X + (long)k * kp.D);
      acc = fma(v, alpha[k], acc);
    }
    if (row) row[k] = v;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0 && mean) mean[c] = acc;
}

// Same contract, input width known at compile time: the query row lives in registers and the
// distance loops are unrolled (the generic kernel spends most of its issue slots on local-memory
// traffic and loop control: 183 instructions per element in ncu).
template <int DT>
__global__ void __launch_bounds__(256)
    cross_gen_fixed_kernel(KParams kp, const double* __restrict__ X, int N, int npad,
                           const double* __restrict__ alpha, const double* __restrict__ Xq,
                           long long ncols, long long cols_pad, double* __restrict__ Ks,
                           double* __restrict__ mean) {
  __shared__ double stbl_all[fm::EXP_TBL_DOUBLES];
  fm::load_exp_table(stbl_all, kp.exp_tbl);
  const unsigned tbl = fm::lane_table(stbl_all);
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const long long c = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (c >= cols_pad) return;
  double* row = Ks ? Ks + c * npad : nullptr;
  if (c >= ncols) {
    if (row)
      for (int k = lane; k < npad; k += 32) row[k] = 0.0;
    return;
  }
  double q[DT];
#pragma unroll
  for (int dd = 0; dd < DT; dd++) q[dd] = Xq[c * DT + dd];
  const int d = kp.d;
  const bool has3 = kp.s3 != 0.0;
  double acc = 0.0;
  for (int k = lane; k < npad; k += 32) {
    double v = 0.0;
    if (k < N) {
      const double* xk = X + (long)k * DT;
      double rx = 0.0, rz = 0.0;
#pragma unroll
      for (int dd = 0; dd < DT; dd++) {
        const double t = q[dd] - xk[dd];
        if (dd < d) rx = fma(t, t, rx);
        else rz = fma(t, t, rz);
      }
      v = fm::exp2s(fma(kp.uz, rz, fma(kp.ux, rx, kp.lc12)), tbl);
      if (has3) v += fm::exp2s(fma(kp.u3, rx, kp.ls3), tbl);
      acc = fma(v, alpha[k], acc);
    }
    if (row) row[k] = v;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0 && mean) mean[c] = acc;
}

// floor = 1e-15 for GPy's reported variance; -inf leaves the latent variance unclipped (batch acquisition)
__global__ void finish_var_kernel(const double* ss, long long n, double kdiag, double noise_add,
                                  double floor, double* var) {   // may run in place (ss == var)
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double v = kdiag - ss[i];
  v = v < floor ? floor : v;   // GPy posterior.py: np.clip(var, 1e-15, inf)
  var[i] = v + noise_add;
}

// locations x_i + o_e * tau, row (i*E + e)
__global__ void build_locs_kernel(const double* __restrict__ X, long long rows, int d,
                                  const double* __restrict__ offs, int E, double tau,
                                  double* __restrict__ out) {
  long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long total = rows * E * d;
  if (idx >= total) return;
  int dd = (int)(idx % d);
  long long re = idx / d;
  int e = (int)(re % E);
  long long i = re / E;
  out[idx] = X[i * d + dd] + offs[e * d + dd] * tau;
}

// Xaug[i] = [x_i, vals[i*E + 0..E-1]]
__global__ void concat_aug_kernel(const double* __restrict__ X, const double* __restrict__ vals,
                                  long long rows, int d, int E, double* __restrict__ out) {
  long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int D = d + E;
  if (idx >= rows * D) return;
  long long i = idx / D;
  int c = (int)(idx - i * D);
  out[idx] = c < d ? X[i * d + c] : vals[i * E + (c - d)];
}

// ---- Philox4x32-10 + Box-Muller: one N(0,1) per 64-bit counter --------------------------------
__device__ __forceinline__ void philox4x32_10(unsigned long long ctr, unsigned long long key,
                                              unsigned (&out)[4]) {
  unsigned c0 = (unsigned)ctr, c1 = (unsigned)(ctr >> 32), c2 = 0u, c3 = 0u;
  unsigned k0 = (unsigned)key, k1 = (unsigned)(key >> 32);
#pragma unroll
  for (int r = 0; r < 10; r++) {
    unsigned hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    unsigned hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    unsigned n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

__device__ __forceinline__ double philox_normal(unsigned long long ctr, unsigned long long seed) {
  unsigned r[4];
  philox4x32_10(ctr, seed, r);
  // two 53-bit-ish uniforms in (0,1)
  const double u1 = ((double)(((unsigned long long)r[0] << 21) ^ (r[1] >> 11)) + 0.5) * (1.0 / 9007199254740992.0);
  const double u2 = ((double)(((unsigned long long)r[2] << 21) ^ (r[3] >> 11)) + 0.5) * (1.0 / 9007199254740992.0);
  return sqrt(-2.0 * log(u1)) * cospi(2.0 * u2);
}

__global__ void fill_normal_kernel(unsigned long long seed, long long first, long long count,
                                   double* __restrict__ out) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < count) out[i] = philox_normal((unsigned long long)(first + i), seed);
}

// rows [x_m, mu_l[m] + sd_l[m]*eps] for columns c = (m - m_lo)*S + s of the current chunk
__global__ void build_mc_rows_kernel(const double* __restrict__ Xtest, const double* __restrict__ mu_l,
                                     const double* __restrict__ sd_l, const double* __restrict__ eps,
                                     unsigned long long seed, long long m_global0, long long m_lo,
                                     long long ncols, int S, int d, double* __restrict__ out) {
  long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= ncols) return;
  const long long m = m_lo + c / S;
  const int s = (int)(c % S);
  const double e = eps ? eps[m * S + s]
                       : philox_normal((unsigned long long)((m_global0 + m) * S + s), seed);
  double* row = out + c * (d + 1);
  for (int dd = 0; dd < d; dd++) row[dd] = Xtest[m * d + dd];
  row[d] = fma(sd_l[m], e, mu_l[m]);
}

// K7 generator: one CTA per test point m, all S samples of it.  Only k1(z_s, Z_k) depends on the
// sample, so the x-dependent factors are computed once per (m, k) into shared memory
//   su[k] = ux |x_m - X_k|^2 + lc12,  sv[k] = exp2s(u3 |x_m - X_k|^2 + ls3),  sz[k] = Z_k,  sa[k] = alpha_k
// (exp2s units, see KParams) and every (sample, k) element then costs ONE exponential:
//   Ks[(m,s)][k] = exp2s(uz (z_s - Z_k)^2 + su[k]) + sv[k],   mu[(m,s)] = sum_k Ks alpha_k.
// Columns are written with 16-byte stores; the per-sample mean is reduced in a fixed order.
// Shared memory per CTA decides how many test points an SM works on at once (the kernel is bound by HBM
// write latency, ncu r01: dram 43 %, 2 CTAs / SM): 512 staged k values (4 arrays x 4 KB) and sample arrays
// sized by S leave room for four CTAs per SM at S = 100 (50 KB each) instead of two (80 KB).
constexpr int MC_KCHUNK = 512;    // k values staged per pass (static smem)
constexpr int MC_MAXS = 1024;
#ifndef MFGP_MC_SB
#define MFGP_MC_SB 2
#endif
constexpr int MC_SB = MFGP_MC_SB;  // samples sharing one pass over the staged chunk

__global__ void __launch_bounds__(256)
    cross_gen_mc_kernel(KParams kp, const double* __restrict__ X, int N, int npad,
                        const double* __restrict__ alpha, const double* __restrict__ Xtest,
                        const double* __restrict__ mu_l, const double* __restrict__ sd_l,
                        const double* __restrict__ eps, unsigned long long seed, long long m_global0,
                        long long m_lo, int S, double* __restrict__ Ks, double* __restrict__ mu_c,
                        const double* __restrict__ zcol, long long z_off, long long ldz) {
  extern __shared__ __align__(16) double stbl_all[];   // exp table (32 KB) | zs[S rounded up] | macc[S rounded up]
  __shared__ __align__(16) double su[MC_KCHUNK], sv[MC_KCHUNK], sz[MC_KCHUNK], sa[MC_KCHUNK];
  double* zs = stbl_all + fm::EXP_TBL_DOUBLES;
  double* macc = zs + ((S + 31) & ~31);
  fm::load_exp_table(stbl_all, kp.exp_tbl);
  const unsigned tbl = fm::lane_table(stbl_all);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const long long m = m_lo + blockIdx.x;
  const int d = kp.d;               // D = d + 1
  double xm[MFGP_MAX_D];
  for (int dd = 0; dd < d; dd++) xm[dd] = Xtest[m * d + dd];
  const double mul = mu_l ? mu_l[m] : 0.0, sdl = sd_l ? sd_l[m] : 1.0;
  const double uz = kp.uz;
  // all S low-fidelity samples of this point up front, one thread each (Philox + Box-Muller costs a few
  // hundred instructions: left to lane 0 of the sample's warp it stalled the other 31 lanes).  With zcol the
  // samples were drawn by the caller (deeper levels of a chain, joint sampling across test points):
  // z_s = mul + zcol[(z_off + point) * ldz + s]
  for (int s = tid; s < S; s += 256) {
    macc[s] = 0.0;
    if (zcol) {
      zs[s] = mul + zcol[(z_off + blockIdx.x) * ldz + s];
    } else {
      const double e = eps ? eps[m * S + s] : philox_normal((unsigned long long)((m_global0 + m) * S + s), seed);
      zs[s] = fma(sdl, e, mul);
    }
  }
  for (int k0 = 0; k0 < npad; k0 += MC_KCHUNK) {
    const int klen = min(MC_KCHUNK, npad - k0);
    __syncthreads();
    for (int kk = tid; kk < klen; kk += 256) {
      const int k = k0 + kk;
      if (k < N) {
        const double* xk = X + (long)k * (d + 1);
        double rx = 0.0;
        for (int dd = 0; dd < d; dd++) {
          const double t = xm[dd] - xk[dd];
          rx = fma(t, t, rx);
        }
        su[kk] = fma(kp.ux, rx, kp.lc12);
        sv[kk] = kp.s3 != 0.0 ? fm::exp2s(fma(kp.u3, rx, kp.ls3), tbl) : 0.0;
        sz[kk] = xk[d];
        sa[kk] = alpha[k];
      } else {   // pad: the element is forced to exactly 0 below
        su[kk] = 0.0;
        sv[kk] = 0.0;
        sz[kk] = 0.0;
        sa[kk] = 0.0;
      }
    }
    __syncthreads();
    // MC_SB samples per pass over the staged chunk: the four shared-memory operands of an element pair are loaded
    // once for all of them (ncu r02: the kernel was bound by shared-memory wavefronts -- short-scoreboard stalls,
    // LSU 58 % busy -- not by the FP64 pipe or HBM); per sample the arithmetic and its order are unchanged
    for (int s0 = warp * MC_SB; s0 < S; s0 += 8 * MC_SB) {
      double z[MC_SB], acc[MC_SB];
      double* row[MC_SB];
      bool live[MC_SB];
#pragma unroll
      for (int q = 0; q < MC_SB; q++) {
        live[q] = s0 + q < S;
        z[q] = live[q] ? zs[s0 + q] : 0.0;
        acc[q] = 0.0;
        row[q] = Ks + ((long long)blockIdx.x * S + (live[q] ? s0 + q : s0)) * npad + k0;
      }
      const int kval = min(klen, N - k0);        // training points in this chunk (the rest is pad)
      const int kfull = kval & ~1;
      for (int kk = 2 * lane; kk < kfull; kk += 64) {
        const double2 u = *reinterpret_cast<const double2*>(su + kk);
        const double2 v = *reinterpret_cast<const double2*>(sv + kk);
        const double2 zz = *reinterpret_cast<const double2*>(sz + kk);
        const double2 a = *reinterpret_cast<const double2*>(sa + kk);
#pragma unroll
        for (int q = 0; q < MC_SB; q++) {
          if (!live[q]) continue;
          const double t0 = z[q] - zz.x, t1 = z[q] - zz.y;
          double2 o;
          o.x = fm::exp2s(fma(uz * t0, t0, u.x), tbl) + v.x;
          o.y = fm::exp2s(fma(uz * t1, t1, u.y), tbl) + v.y;
          *reinterpret_cast<double2*>(row[q] + kk) = o;
          acc[q] = fma(o.x, a.x, acc[q]);
          acc[q] = fma(o.y, a.y, acc[q]);
        }
      }
      // ragged end: at most one training point, then the zero pad up to the 128-multiple
      for (int kk = kfull + 2 * lane; kk < klen; kk += 64) {
#pragma unroll
        for (int q = 0; q < MC_SB; q++) {
          if (!live[q]) continue;
          double2 o = make_double2(0.0, 0.0);
          if (kk < kval) {
            const double t0 = z[q] - sz[kk];
            o.x = fm::exp2s(fma(uz * t0, t0, su[kk]), tbl) + sv[kk];
            acc[q] = fma(o.x, sa[kk], acc[q]);
          }
          *reinterpret_cast<double2*>(row[q] + kk) = o;
        }
      }
#pragma unroll
      for (int q = 0; q < MC_SB; q++) {
        double r = acc[q];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) r += __shfl_xor_sync(0xffffffffu, r, o);
        if (lane == 0 && live[q]) macc[s0 + q] += r;   // one warp is the only writer of macc[s]
      }
    }
  }
  __syncthreads();
  for (int s = tid; s < S; s += 256) mu_c[(long long)blockIdx.x * S + s] = macc[s];
}


// ---- K7 for small upper levels (N <= 64): generator AND contraction in one kernel, nothing N-wide in HBM ----
// The reference's own high-fidelity levels hold 5-30 points (src/gpc/mfgp_gpc.py:10,18-20).  Through the
// general path a (point, sample) column of such a level costs a 128-wide row of Ks written to HBM and read
// back, and a 128 x 128 triangular product: at N = 30 that is (128/30)^2 = 18 times the algorithmic flops.
// Here ONE WARP owns a test point: the x-dependent factors of its S columns go to the warp's slice of shared
// memory once (as in cross_gen_mc_kernel), the columns are taken eight at a time as the n dimension of
// DMMA.8x8x4, the lane that owns B[k = 4 kk + t][n = g] COMPUTES that cross-covariance element (one exp2s) in
// the register the tensor instruction reads, and the NP x NP leading block of W = L^-1 (NP = 16, 32 or 64) sits in
// registers as A fragments for the whole kernel (6 / 20 / 72 doubles per lane; only blocks with k <= row).
// Per column: N exponentials and NP^2/2 multiply-adds, no shared-memory traffic in the product, no barrier.
// All reductions in fixed order; a column's result does not depend on how points are split over launches.
__device__ __forceinline__ void dmma884p(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
               : "+d"(c0), "+d"(c1)
               : "d"(a), "d"(b));
}

constexpr int MCS_WARPS = 8;

template <int NP>
__global__ void __launch_bounds__(MCS_WARPS * 32, NP <= 32 ? 2 : 1)
    mc_small_kernel(KParams kp, const double* __restrict__ X, int N, int ldw, const double* __restrict__ W,
                    const double* __restrict__ alpha, const double* __restrict__ Xtest,
                    const double* __restrict__ mu_l, const double* __restrict__ sd_l,
                    const double* __restrict__ eps, unsigned long long seed, long long m_global0, long long m_lo,
                    long long npts, int S, double* __restrict__ mu_c, double* __restrict__ ss_out,
                    const double* __restrict__ zcol, long long z_off, long long ldz) {
  constexpr int RB = NP / 8, KS = NP / 4;                // row blocks, k steps
  extern __shared__ __align__(16) double sm_mcs[];       // tbl[256] | sz[NP] | sa[NP] | sX[d][NP] | per warp: su[NP], sv[NP]
  const int d = kp.d;                                    // D = d + 1
  double* stbl = sm_mcs;
  double* sz = stbl + 256;
  double* sa = sz + NP;
  double* sX = sa + NP;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = lane >> 2, t = lane & 3;
  double* su = sX + d * NP + warp * 2 * NP;
  double* sv = su + NP;
  stbl[tid] = kp.exp_tbl[tid];
  for (int idx = tid; idx < NP * (d + 1); idx += MCS_WARPS * 32) {
    const int j = idx / (d + 1), dd = idx - j * (d + 1);
    const double v = j < N ? X[idx] : 0.0;
    if (dd < d) sX[dd * NP + j] = v;
    else sz[j] = v;
  }
  if (tid < NP) sa[tid] = tid < N ? alpha[tid] : 0.0;
  // A fragments: wf[r][kk] = W[8 r + g][4 kk + t] for the blocks that touch the lower triangle (kk <= 2 r + 1)
  double wf[RB][KS];
#pragma unroll
  for (int r = 0; r < RB; r++)
#pragma unroll
    for (int kk = 0; kk < KS; kk++)
      if (kk <= 2 * r + 1) wf[r][kk] = W[(long)(8 * r + g) * ldw + 4 * kk + t];
  __syncthreads();
  const unsigned tbl = (unsigned)__cvta_generic_to_shared(stbl);
  const double uz = kp.uz;
  const bool has3 = kp.s3 != 0.0;
  for (long long pl = (long long)blockIdx.x * MCS_WARPS + warp; pl < npts; pl += (long long)gridDim.x * MCS_WARPS) {
    const long long m = m_lo + pl;
    // x-dependent factors of this point, one training point per lane
    __syncwarp();
#pragma unroll
    for (int j0 = 0; j0 < NP; j0 += 32) {
      const int j = j0 + lane;
      if (NP < 32 && j >= NP) break;
      double rx = 0.0;
      for (int dd = 0; dd < d; dd++) {
        const double q = Xtest[m * d + dd] - sX[dd * NP + j];
        rx = fma(q, q, rx);
      }
      su[j] = fma(kp.ux, rx, kp.lc12);
      sv[j] = has3 ? fm::exp2s_flat(fma(kp.u3, rx, kp.ls3), tbl) : 0.0;
    }
    __syncwarp();
    const double mul = mu_l ? mu_l[m] : 0.0, sdl = sd_l ? sd_l[m] : 1.0;
    for (int s0 = 0; s0 < S; s0 += 32) {
      // the samples of 32 columns, one per lane (same draws as cross_gen_mc_kernel)
      double zl = 0.0;
      if (s0 + lane < S) {
        const int sidx = s0 + lane;
        if (zcol) {
          zl = mul + zcol[(z_off + pl) * ldz + sidx];
        } else {
          const double e = eps ? eps[m * S + sidx]
                               : philox_normal((unsigned long long)((m_global0 + m) * S + sidx), seed);
          zl = fma(sdl, e, mul);
        }
      }
      const int ngrp = min(4, (S - s0 + 7) >> 3);
      for (int grp = 0; grp < ngrp; grp++) {
        const double zc = __shfl_sync(0xffffffffu, zl, 8 * grp + g);     // sample of column g of this group
        double D0[RB], D1[RB];
#pragma unroll
        for (int r = 0; r < RB; r++) D0[r] = D1[r] = 0.0;
        double macc = 0.0;
#pragma unroll
        for (int kk = 0; kk < KS; kk++) {
          const int j = 4 * kk + t;
          const double q = zc - sz[j];
          double b = fm::exp2s_flat(fma(uz * q, q, su[j]), tbl) + sv[j];
          if (j >= N) b = 0.0;                                           // identity pad: exactly zero
          macc = fma(b, sa[j], macc);
#pragma unroll
          for (int r = kk / 2; r < RB; r++) dmma884p(D0[r], D1[r], wf[r][kk], b);
        }
        // column sums of squares: rows 8 r + g of columns 2 t, 2 t + 1; then over g
        double q0 = 0.0, q1 = 0.0;
#pragma unroll
        for (int r = 0; r < RB; r++) {
          q0 = fma(D0[r], D0[r], q0);
          q1 = fma(D1[r], D1[r], q1);
        }
#pragma unroll
        for (int o = 4; o < 32; o <<= 1) {
          q0 += __shfl_xor_sync(0xffffffffu, q0, o);
          q1 += __shfl_xor_sync(0xffffffffu, q1, o);
        }
        macc += __shfl_xor_sync(0xffffffffu, macc, 1);
        macc += __shfl_xor_sync(0xffffffffu, macc, 2);
        const long long c0 = pl * S + s0 + 8 * grp;
        const int left = S - s0 - 8 * grp;                               // valid columns in this group
        if (g == 0) {
          if (2 * t < left) ss_out[c0 + 2 * t] = q0;
          if (2 * t + 1 < left) ss_out[c0 + 2 * t + 1] = q1;
        }
        if (t == 0 && g < left) mu_c[c0 + g] = macc;
      }
    }
  }
}

// ---- K7 with delays: joint low-fidelity posterior at the E augmented locations of a test point ----
// G[p][a,b] = sum_i T[i][p*E+a] * T[i][p*E+b]  (packed lower triangle, a >= b); eight threads per point
// (row groups), rows of T read coalesced (adjacent points are adjacent columns), fixed summation order.
constexpr int GG_PTS = 16, GG_RG = 8;   // points per CTA x row groups: 128 threads
template <int E>
__global__ void __launch_bounds__(GG_PTS * GG_RG)
    group_gram_kernel(const double* __restrict__ T, int npad, long long ldt, long long npts,
                      double* __restrict__ G) {
  // thread (rg, pl): point p = 16*blockIdx + pl, rows i = rg, rg+8, ...; threads of one row group read
  // adjacent columns (coalesced); the 8 partial Grams of a point are added in row-group order
  constexpr int NP = E * (E + 1) / 2;
  __shared__ double part[GG_RG][GG_PTS][NP];
  const int pl = threadIdx.x % GG_PTS, rg = threadIdx.x / GG_PTS;
  const long long p = (long long)blockIdx.x * GG_PTS + pl;
  double acc[NP];
#pragma unroll
  for (int q = 0; q < NP; q++) acc[q] = 0.0;
  if (p < npts) {
    const double* col = T + p * E;
#pragma unroll 4
    for (int i = rg; i < npad; i += GG_RG) {
      double v[E];
#pragma unroll
      for (int e = 0; e < E; e++) v[e] = col[(long long)i * ldt + e];
      int q = 0;
#pragma unroll
      for (int a = 0; a < E; a++)
#pragma unroll
        for (int b = 0; b <= a; b++, q++) acc[q] = fma(v[a], v[b], acc[q]);
    }
  }
#pragma unroll
  for (int q = 0; q < NP; q++) part[rg][pl][q] = acc[q];
  __syncthreads();
  if (rg == 0 && p < npts) {
#pragma unroll
    for (int q = 0; q < NP; q++) {
      double v = part[0][pl][q];
#pragma unroll
      for (int r = 1; r < GG_RG; r++) v += part[r][pl][q];
      G[p * NP + q] = v;
    }
  }
}

// cov = kab - G (diagonal clipped at 1e-15 like GPy's predictive variance, then + diag_add);
// Lc[p] = chol(cov) (E x E, row-major lower).  A non-positive pivot records the point (1-based) in
// info[1] (lowest index wins) and is replaced by 1e-300 so that the kernel finishes.
template <int E>
__global__ void __launch_bounds__(128)
    joint_chol_kernel(const double* __restrict__ G, const double* __restrict__ kab, long long npts,
                      double diag_add, long long p_global0, double* __restrict__ Lc, int* __restrict__ info) {
  const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= npts) return;
  constexpr int NP = E * (E + 1) / 2;
  double c[E][E];
  int q = 0;
#pragma unroll
  for (int a = 0; a < E; a++)
#pragma unroll
    for (int b = 0; b <= a; b++, q++) {
      double v = kab[a * E + b] - G[p * NP + q];
      if (a == b) v = (v < 1e-15 ? 1e-15 : v) + diag_add;
      c[a][b] = v;
    }
  bool bad = false;
#pragma unroll
  for (int j = 0; j < E; j++) {
    double dj = c[j][j];
#pragma unroll
    for (int k = 0; k < j; k++) dj = fma(-c[j][k], c[j][k], dj);
    if (!(dj > 0.0)) { bad = true; dj = 1e-300; }
    const double lj = sqrt(dj);
    c[j][j] = lj;
#pragma unroll
    for (int i = j + 1; i < E; i++) {
      double v = c[i][j];
#pragma unroll
      for (int k = 0; k < j; k++) v = fma(-c[i][k], c[j][k], v);
      c[i][j] = v / lj;
    }
  }
  if (bad) {
    const long long idx = p_global0 + p + 1;
    atomicMin(reinterpret_cast<unsigned*>(info + 1), (unsigned)(idx > 0x7fffffffLL ? 0x7fffffffLL : idx));
  }
#pragma unroll
  for (int a = 0; a < E; a++)
#pragma unroll
    for (int b = 0; b < E; b++) Lc[(p * E + a) * E + b] = b <= a ? c[a][b] : 0.0;
}

// rows [x_m, mu_l[m] + Lc[m] eps] for columns c = (m - m_lo)*S + s of the current chunk;
// eps: (M, S, E) supplied, or Philox counter ((m_global0 + m)*S + s)*E + e
__global__ void build_mc_rows_joint_kernel(const double* __restrict__ Xtest, const double* __restrict__ mu_l,
                                           const double* __restrict__ Lc, const double* __restrict__ eps,
                                           unsigned long long seed, long long m_global0, long long m_lo,
                                           long long ncols, int S, int d, int E,
                                           double* __restrict__ out) {
  const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= ncols) return;
  const long long pl = c / S;               // point within the chunk (mu_l / Lc are chunk-local)
  const long long m = m_lo + pl;            // point within the call
  const int s = (int)(c - pl * S);
  double e[MFGP_MAX_E];
  for (int b = 0; b < E; b++)
    e[b] = eps ? eps[(m * S + s) * E + b]
               : philox_normal((unsigned long long)(((m_global0 + m) * S + s) * E + b), seed);
  double* row = out + c * (d + E);
  for (int dd = 0; dd < d; dd++) row[dd] = Xtest[m * d + dd];
  for (int a = 0; a < E; a++) {
    double z = mu_l[pl * E + a];
    for (int b = 0; b <= a; b++) z = fma(Lc[(pl * E + a) * E + b], e[b], z);
    row[d + a] = z;
  }
}

__global__ void zero_rows_kernel(double* __restrict__ p, long long n) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = 0.0;
}

__global__ void sqrt_kernel(double* __restrict__ v, long long n) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) v[i] = sqrt(v[i]);
}

// mean_m = mean_s mu;  var_m = mean_s v + population variance of mu (two-pass, fixed order)
__global__ void mc_aggregate_kernel(const double* __restrict__ mu_c, const double* __restrict__ v_c,
                                    long long npts, int S, double* __restrict__ mean,
                                    double* __restrict__ var) {
  long long m = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= npts) return;
  const double* mu = mu_c + m * S;
  const double* vv = v_c + m * S;
  double sm = 0.0, sv = 0.0;
  for (int s = 0; s < S; s++) {
    sm += mu[s];
    sv += vv[s];
  }
  const double mbar = sm / S;
  double dev = 0.0;
  for (int s = 0; s < S; s++) {
    double t = mu[s] - mbar;
    dev = fma(t, t, dev);
  }
  mean[m] = mbar;
  var[m] = sv / S + dev / S;
}

// z[c] = mu_c[c] + sqrt(v_c[c]) * eps for the columns c = (m - m_lo) * S + s of the current chunk: the sample
// one level of a NARGP chain hands to the next (eps supplied as (M, S), or Philox counter (m_global0 + m) S + s)
__global__ void sample_cols_kernel(const double* __restrict__ mu_c, const double* __restrict__ v_c,
                                   const double* __restrict__ eps, unsigned long long key, long long m_global0,
                                   long long m_lo, long long ncols, int S, double* __restrict__ z) {
  const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= ncols) return;
  const long long m = m_lo + c / S;
  const int s = (int)(c % S);
  const double e = eps ? eps[m * S + s] : philox_normal((unsigned long long)((m_global0 + m) * S + s), key);
  z[c] = fma(sqrt(v_c[c]), e, mu_c[c]);
}

// E[j][s] (ld = ldE, zero padded to rows x ldE) from supplied normals (M, S) or Philox counter j * S + s
__global__ void fill_normal_padded_kernel(const double* __restrict__ eps, unsigned long long seed, long long M,
                                          int S, long long rows, long long ldE, double* __restrict__ E) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= rows * ldE) return;
  const long long j = idx / ldE;
  const int s = (int)(idx - j * ldE);
  double v = 0.0;
  if (j < M && s < S) v = eps ? eps[j * S + s] : philox_normal((unsigned long long)(j * S + s), seed);
  E[idx] = v;
}

// path[s] += sum_m w[m_lo + m] * mu_c[m * S + s] over the points of one chunk; one block per sample path,
// fixed-order reduction, chunks arrive in stream order: deterministic
__global__ void __launch_bounds__(256)
    path_wsum_kernel(const double* __restrict__ mu_c, const double* __restrict__ w, long long m_lo,
                     long long npts, int S, double* __restrict__ path) {
  __shared__ double sv[256];
  const int s = blockIdx.x;
  double acc = 0.0;
  for (long long m = threadIdx.x; m < npts; m += 256) acc = fma(w ? w[m_lo + m] : 1.0, mu_c[m * S + s], acc);
  sv[threadIdx.x] = acc;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) sv[threadIdx.x] += sv[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) path[s] += sv[0];
}

// ---- latency path: a handful of query rows, one CTA each, results straight into mapped host memory ----------
// The reference's default acquisition is a sequential DIRECT search of up to 20 000 single-point predicts
// (src/adaptation_maximizers/scipydirect_wrapper.py:22-26).  Through mfgp_predict every one of them costs an
// upload, three launches and two downloads (~130 us); here it is one or two launches and ONE synchronisation:
// the query row is read from, and (mean, variance) written to, pinned host memory mapped into the device.
constexpr int PS_MAXN = 2048;     // training points (kx lives in shared memory)

__device__ __forceinline__ double small_kernel_value(const KParams& kp, const double* __restrict__ q,
                                                     const double* __restrict__ xk, unsigned tbl) {
  double rx = 0.0, rz = 0.0;
  for (int dd = 0; dd < kp.D; dd++) {
    const double t = q[dd] - xk[dd];
    if (dd < kp.d) rx = fma(t, t, rx);
    else rz = fma(t, t, rz);
  }
  double v = fm::exp2s_flat(fma(kp.uz, rz, fma(kp.ux, rx, kp.lc12)), tbl);
  if (kp.s3 != 0.0) v += fm::exp2s_flat(fma(kp.u3, rx, kp.ls3), tbl);
  return v;
}

// Block-wide pieces shared by the latency kernels and the point service (256 threads; every thread must call).
// mu_l(loc) = sum_k K_l(loc, Xl_k) alpha_k, fixed-order block reduction; the result is returned to every thread.
__device__ __forceinline__ double ps_lf_mean(const KParams& kl, const double* __restrict__ Xl, int Nl,
                                             const double* __restrict__ alpha_l, const double* loc, unsigned tbl,
                                             double* red /* [256] shared */) {
  const int tid = threadIdx.x;
  double acc = 0.0;
  for (int k = tid; k < Nl; k += 256) acc = fma(small_kernel_value(kl, loc, Xl + (long)k * kl.D, tbl), alpha_l[k], acc);
  red[tid] = acc;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (tid < o) red[tid] += red[tid + o];
    __syncthreads();
  }
  const double v = red[0];
  __syncthreads();
  return v;
}

// (mean, var) of one query row q: kx in shared memory, mean by a fixed-order block reduction, then tmp = W kx with
// one warp per row of W (coalesced), sum of squares in a fixed order.  Valid in thread 0 on return.
__device__ __forceinline__ void ps_predict_row(const KParams& kp, const double* __restrict__ X, int N, int npad,
                                               const double* __restrict__ alpha, const double* __restrict__ W,
                                               const double* q, double noise_add, unsigned tbl, double* kx,
                                               double* red, double* wss, double& mean, double& var) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  double acc = 0.0;
  for (int k = tid; k < N; k += 256) {
    const double v = small_kernel_value(kp, q, X + (long)k * kp.D, tbl);
    kx[k] = v;
    acc = fma(v, alpha[k], acc);
  }
  red[tid] = acc;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (tid < o) red[tid] += red[tid + o];
    __syncthreads();
  }
  double ss = 0.0;
  for (int i = warp; i < N; i += 8) {
    const double* row = W + (long)i * npad;
    double t = 0.0;
    for (int k = lane; k <= i; k += 32) t = fma(row[k], kx[k], t);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
    ss = fma(t, t, ss);
  }
  if (lane == 0) wss[warp] = ss;
  __syncthreads();
  mean = 0.0;
  var = 0.0;
  if (tid == 0) {
    double sum = 0.0;
    for (int w = 0; w < 8; w++) sum += wss[w];
    double v = kp.kdiag - sum;
    v = v < 1e-15 ? 1e-15 : v;   // GPy posterior.py: np.clip(var, 1e-15, inf)
    mean = red[0];
    var = v + noise_add;
  }
  __syncthreads();
}

// Xaug[m] = [x_m, mu_l(x_m + o_0 tau), ...]: one CTA per (row, location); fixed-order block reduction
__global__ void __launch_bounds__(256)
    augment_small_kernel(KParams kl, const double* __restrict__ Xl, int Nl, const double* __restrict__ alpha_l,
                         const double* __restrict__ Xq, int d, const double* __restrict__ offs, int E,
                         double tau, double* __restrict__ Xaug) {
  __shared__ double stbl[256];
  __shared__ double red[256];
  __shared__ double loc[MFGP_MAX_D];
  const int m = blockIdx.x / E, e = blockIdx.x - m * E, tid = threadIdx.x;
  stbl[tid] = kl.exp_tbl[tid];
  if (tid < d) loc[tid] = Xq[m * d + tid] + offs[e * d + tid] * tau;
  __syncthreads();
  const unsigned tbl = (unsigned)__cvta_generic_to_shared(stbl);
  const double mu = ps_lf_mean(kl, Xl, Nl, alpha_l, loc, tbl, red);
  double* row = Xaug + (long)m * (d + E);
  if (tid == 0) row[d + e] = mu;
  if (e == 0 && tid < d) row[tid] = Xq[m * d + tid];
}

// (mean, var) of one query row per CTA
__global__ void __launch_bounds__(256)
    predict_small_kernel(KParams kp, const double* __restrict__ X, int N, int npad,
                         const double* __restrict__ alpha, const double* __restrict__ W,
                         const double* __restrict__ Xq, double noise_add, double* __restrict__ out /* (M, 2) */) {
  __shared__ double stbl[256];
  __shared__ double kx[PS_MAXN];
  __shared__ double red[256];
  __shared__ double wss[8];
  const int tid = threadIdx.x;
  const double* q = Xq + (long)blockIdx.x * kp.D;
  stbl[tid] = kp.exp_tbl[tid];
  __syncthreads();
  const unsigned tbl = (unsigned)__cvta_generic_to_shared(stbl);
  double mean, var;
  ps_predict_row(kp, X, N, npad, alpha, W, q, noise_add, tbl, kx, red, wss, mean, var);
  if (tid == 0) {
    out[2 * blockIdx.x] = mean;
    out[2 * blockIdx.x + 1] = var;
  }
}

// ---- point service: single-row predicts answered by a RESIDENT single-CTA kernel through mapped host memory ----
// The reference's default acquisition (scipydirect DIRECT, src/adaptation_maximizers/scipydirect_wrapper.py:22-26)
// asks for up to 20 000 single-point predicts ONE AFTER THE OTHER; each answer decides the next question, so they
// cannot be batched.  Per question the launch + synchronise path costs ~30 us of driver latency for ~3 us of
// arithmetic.  Here one CTA stays resident for the duration of a search: the host writes the query row and a
// sequence number into mapped pinned memory, thread 0 polls that number over PCIe, the CTA evaluates the row with
// the very device functions of the latency kernels (bit-identical results) and writes (mean, variance) and the
// acknowledged sequence number back.  No launch, no stream synchronisation per question.  The kernel leaves on a
// stop flag or after `idle_ns` without a question (a crashed host cannot pin the SM); the host relaunches it when
// it finds it gone.  It occupies ONE SM and runs on its own non-blocking stream.
__device__ __forceinline__ unsigned long long ps_globaltimer() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

__global__ void __launch_bounds__(256)
    point_service_kernel(PointServiceArgs a, PointServiceCtl* ctl) {
  __shared__ double stbl[256];
  __shared__ double kx[PS_MAXN];
  __shared__ double red[256];
  __shared__ double wss[8];
  __shared__ double q[MFGP_MAX_D + MFGP_MAX_E];
  __shared__ double loc[MFGP_MAX_D];
  __shared__ unsigned long long s_seq;
  __shared__ int s_go;
  const int tid = threadIdx.x;
  stbl[tid] = a.kh.exp_tbl[tid];
  __syncthreads();
  const unsigned tbl = (unsigned)__cvta_generic_to_shared(stbl);
  unsigned long long last = a.start_seq;
  const int width = a.has_lf ? a.d : a.kh.D;
  for (;;) {
    if (tid == 0) {
      const unsigned long long t0 = ps_globaltimer();
      int go = 0;
      unsigned long long seq = last;
      for (unsigned spin = 0;; spin++) {
        seq = ctl->req_seq;                     // one PCIe read per poll
        if (seq != last) { go = 1; break; }
        if ((spin & 15u) == 15u) {
          if (ctl->stop) break;
          if (ps_globaltimer() - t0 > a.idle_ns) break;
        }
      }
      s_go = go;
      s_seq = seq;
    }
    __syncthreads();
    if (!s_go) break;
    if (tid < width) q[tid] = ctl->x[tid];
    __syncthreads();
    if (a.has_lf) {
      for (int e = 0; e < a.E; e++) {
        if (tid < a.d) loc[tid] = q[tid] + a.offs[e * a.d + tid] * a.tau;
        __syncthreads();
        const double mu = ps_lf_mean(a.kl, a.Xl, a.Nl, a.alpha_l, loc, tbl, red);
        if (tid == 0) q[a.d + e] = mu;
        __syncthreads();
      }
    }
    double mean, var;
    ps_predict_row(a.kh, a.Xh, a.Nh, a.npad_h, a.alpha_h, a.Wh, q, a.noise_add, tbl, kx, red, wss, mean, var);
    if (tid == 0) {
      ctl->out[0] = mean;
      ctl->out[1] = var;
      __threadfence_system();
      ctl->ack_seq = s_seq;
    }
    last = s_seq;
    __syncthreads();
  }
  if (tid == 0) {
    __threadfence_system();
    ctl->alive = 0;
  }
}

// ---- deterministic reductions -----------------------------------------------------------------
constexpr int RED_BLOCKS = 1024;

__global__ void __launch_bounds__(256)
    argmax_stage1_kernel(const double* __restrict__ v, long long n, double* __restrict__ pval,
                         long long* __restrict__ pidx) {
  __shared__ double sv[256];
  __shared__ long long si[256];
  double best = -INFINITY;
  long long bi = 0x7fffffffffffffffLL;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
       i += (long long)gridDim.x * blockDim.x) {
    double x = v[i];
    if (x > best) {   // strictly greater: the lowest index wins (indices ascend per thread)
      best = x;
      bi = i;
    }
  }
  sv[threadIdx.x] = best;
  si[threadIdx.x] = bi;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) {
      double x = sv[threadIdx.x + o];
      long long xi = si[threadIdx.x + o];
      if (x > sv[threadIdx.x] || (x == sv[threadIdx.x] && xi < si[threadIdx.x])) {
        sv[threadIdx.x] = x;
        si[threadIdx.x] = xi;
      }
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    pval[blockIdx.x] = sv[0];
    pidx[blockIdx.x] = si[0];
  }
}

__global__ void argmax_stage2_kernel(const double* __restrict__ pval, const long long* __restrict__ pidx,
                                     int nb, double* __restrict__ out_val, long long* __restrict__ out_idx) {
  __shared__ double sv[256];
  __shared__ long long si[256];
  double best = -INFINITY;
  long long bi = 0x7fffffffffffffffLL;
  for (int b = threadIdx.x; b < nb; b += blockDim.x) {
    double x = pval[b];
    long long xi = pidx[b];
    if (x > best || (x == best && xi < bi)) {
      best = x;
      bi = xi;
    }
  }
  sv[threadIdx.x] = best;
  si[threadIdx.x] = bi;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) {
      double x = sv[threadIdx.x + o];
      long long xi = si[threadIdx.x + o];
      if (x > sv[threadIdx.x] || (x == sv[threadIdx.x] && xi < si[threadIdx.x])) {
        sv[threadIdx.x] = x;
        si[threadIdx.x] = xi;
      }
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    out_val[0] = sv[0];
    out_idx[0] = si[0];
  }
}

// ---- K8b greedy batch acquisition: pivoted partial Cholesky of the posterior covariance over the candidates ----
// At fixed theta the posterior covariance kappa(c, a) = k(c, a) - k_c^T K_y^-1 k_a does not depend on the targets,
// so the q points that q sequential "arg-max, then append" steps pick are known in advance.  With
// s^2 = noise + 1e-8 + jitter (the diagonal of a bordered update) and v_0(c) = k(c, c) - |W k_c|^2 (unclipped),
// step i conditions on pivot p_i with augmented row a_i:
//   u_i = K_y^-1 k(X, a_i),   g_i(c) = sum_k K(c, X_k) u_i[k],   rho_i = sqrt(v_i(p_i) + s^2),
//   R[i][c] = (k(c, a_i) - g_i(c) - sum_{l<i} R[l][c] R[l][p_i]) / rho_i,   v_{i+1}(c) = v_i(c) - R[i][c]^2.
// k(c, a_i) - g_i(c) comes from ONE mean-mode pass of the cross-covariance generator over X' = [X; a_i] with the
// coefficients [-u_i; 1] (acq_coef_kernel): no C x N block is stored.  Reported and compared values are GPy's
// max(v, 1e-15) + noise, lowest index on ties, so the first pick is exactly mfgp_argmax over mfgp_predict's variance.

// coef[k] = -u[k] (k < N), 1 (k == N), 0 on the pad up to npad1
__global__ void acq_coef_kernel(const double* u, int N, int npad1, double* coef) {   // may run in place
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k < npad1) coef[k] = k < N ? -u[k] : (k == N ? 1.0 : 0.0);
}

// Per candidate (grid-stride): with kg, r = (kg[c] - sum_{l<i} R[l][c] rp[l]) / rho in a fixed order, R[i][c] = r,
// v[c] -= r^2; without kg, v is read as it is (the first pick).  Then stage 1 of the arg-max over
// max(v, 1e-15) + noise_add with argmax_stage1_kernel's tie rule; argmax_stage2_kernel finishes it.
// R is (q, C) row-major: the reads of one l are coalesced over the candidates.
__global__ void __launch_bounds__(256)
    acq_update_kernel(const double* __restrict__ kg, double* __restrict__ R, long long C, int i,
                      const double* __restrict__ rp, double rho, double* __restrict__ v, double noise_add,
                      double* __restrict__ pval, long long* __restrict__ pidx) {
  __shared__ double srp[MFGP_ACQ_MAX_Q];
  __shared__ double sv[256];
  __shared__ long long si[256];
  if (kg)
    for (int l = threadIdx.x; l < i; l += blockDim.x) srp[l] = rp[l];
  __syncthreads();
  double best = -INFINITY;
  long long bi = 0x7fffffffffffffffLL;
  for (long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x; c < C;
       c += (long long)gridDim.x * blockDim.x) {
    double x = v[c];
    if (kg) {
      double t = kg[c];
      for (int l = 0; l < i; l++) t = fma(-R[(long long)l * C + c], srp[l], t);
      const double r = t / rho;
      R[(long long)i * C + c] = r;
      x = fma(-r, r, x);
      v[c] = x;
    }
    const double rep = (x < 1e-15 ? 1e-15 : x) + noise_add;   // what finish_var_kernel reports
    if (rep > best) {   // strictly greater: the lowest index wins (indices ascend per thread)
      best = rep;
      bi = c;
    }
  }
  sv[threadIdx.x] = best;
  si[threadIdx.x] = bi;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) {
      double x = sv[threadIdx.x + o];
      long long xi = si[threadIdx.x + o];
      if (x > sv[threadIdx.x] || (x == sv[threadIdx.x] && xi < si[threadIdx.x])) {
        sv[threadIdx.x] = x;
        si[threadIdx.x] = xi;
      }
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    pval[blockIdx.x] = sv[0];
    pidx[blockIdx.x] = si[0];
  }
}

// The winner's record for the host (out: mapped pinned memory): out[0] = reported variance, out[1] = local index
// (int64 bits), out[2..] = [v(p) unclipped, a = cands[p] (D values), R[0..nr)[p], zeros up to q entries].
__global__ void acq_gather_kernel(const double* __restrict__ best_val, const long long* __restrict__ best_idx,
                                  const double* __restrict__ v, const double* __restrict__ cands, int D,
                                  const double* __restrict__ R, long long C, int nr, int q, double* __restrict__ out) {
  const long long p = best_idx[0];
  const bool ok = p >= 0 && p < C;   // no candidate with a comparable variance (all NaN): the host reports it
  double* rec = out + 2;
  if (threadIdx.x == 0) {
    out[0] = best_val[0];
    out[1] = __longlong_as_double(ok ? p : -1LL);
    rec[0] = ok ? v[p] : NAN;
  }
  for (int k = threadIdx.x; k < D; k += blockDim.x) rec[1 + k] = ok ? cands[p * D + k] : NAN;
  for (int l = threadIdx.x; l < q; l += blockDim.x) rec[1 + D + l] = ok && l < nr ? R[(long long)l * C + p] : 0.0;
}

// sum_i w[i]*x[i], two deterministic stages
__global__ void __launch_bounds__(256)
    wdot_stage1_kernel(const double* __restrict__ w, const double* __restrict__ x, long long n,
                       double* __restrict__ partials) {
  __shared__ double sv[256];
  double acc = 0.0;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
       i += (long long)gridDim.x * blockDim.x)
    acc = fma(w ? w[i] : 1.0, x[i], acc);
  sv[threadIdx.x] = acc;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) sv[threadIdx.x] += sv[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) partials[blockIdx.x] = sv[0];
}

__global__ void sum_stage2_kernel(const double* __restrict__ partials, int nb, double* __restrict__ out) {
  __shared__ double sv[256];
  double acc = 0.0;
  for (int b = threadIdx.x; b < nb; b += blockDim.x) acc += partials[b];
  sv[threadIdx.x] = acc;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) sv[threadIdx.x] += sv[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) out[0] = sv[0];
}

// ---- O(N^2) solves with the explicit inverse factor W = L^-1 ----------------------------------
// v[i] = sum_{k<=i} W[i][k] y[k]     (one warp per row)
__global__ void __launch_bounds__(256)
    trmv_lower_kernel(const double* __restrict__ W, int npad, const double* __restrict__ y, int N,
                      double* __restrict__ v) {
  const int i = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (i >= npad) return;
  const double* row = W + (long)i * npad;
  const int kend = min(i + 1, N);
  double acc = 0.0;
  for (int k = lane; k < kend; k += 32) acc = fma(row[k], y[k], acc);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0) v[i] = acc;
}

// alpha[k] = sum_{i>=k} W[i][k] v[i]; a block owns 32 columns, 8 row lanes, fixed-order reduction
__global__ void __launch_bounds__(256)
    trmv_lower_t_kernel(const double* __restrict__ W, int npad, const double* __restrict__ v,
                        double* __restrict__ alpha) {
  __shared__ double red[8][33];
  const int cx = threadIdx.x & 31, ry = threadIdx.x >> 5;
  const int k0 = blockIdx.x * 32;
  const int k = k0 + cx;
  double a0 = 0.0, a1 = 0.0;
  int i = k0 + ry;
  for (; i + 8 < npad; i += 16) {
    a0 = fma(W[(long)i * npad + k], v[i], a0);
    a1 = fma(W[(long)(i + 8) * npad + k], v[i + 8], a1);
  }
  if (i < npad) a0 = fma(W[(long)i * npad + k], v[i], a0);
  red[ry][cx] = a0 + a1;
  __syncthreads();
  if (ry == 0) {
    double s = 0.0;
#pragma unroll
    for (int r = 0; r < 8; r++) s += red[r][cx];
    alpha[k] = s;
  }
}

// out[0] = LML, out[1] = logdet, out[2] = y^T alpha     (single block)
__global__ void __launch_bounds__(256)
    lml_kernel(const double* __restrict__ L, int npad, int N, const double* __restrict__ y,
               const double* __restrict__ alpha, double* __restrict__ out) {
  __shared__ double s0[256], s1[256];
  double ld = 0.0, ya = 0.0;
  for (int i = threadIdx.x; i < N; i += 256) {
    ld += log(L[(long)i * npad + i]);
    ya = fma(y[i], alpha[i], ya);
  }
  s0[threadIdx.x] = ld;
  s1[threadIdx.x] = ya;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) {
      s0[threadIdx.x] += s0[threadIdx.x + o];
      s1[threadIdx.x] += s1[threadIdx.x + o];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    const double logdet = 2.0 * s0[0];
    out[1] = logdet;
    out[2] = s1[0];
    out[0] = 0.5 * (-(double)N * 1.8378770664093453 - logdet - s1[0]);
  }
}


// Bordered Cholesky update (one appended training point, fixed theta):
//   l = W k (done), t = W^T l (done);  s = K(a,a) + diag_add - |l|^2;  L[N] = [l, sqrt(s)];
//   W[N] = [-t / sqrt(s), 1 / sqrt(s)].   Single block; the sum runs in a fixed order.
__global__ void __launch_bounds__(256)
    append_finish_kernel(const double* __restrict__ l, const double* __restrict__ t, int N, int npad,
                         double kaa, double* __restrict__ A, double* __restrict__ W, int write_L,
                         int* __restrict__ info, double* __restrict__ out /* [0] = l_nn, [1] = s */) {
  __shared__ double sv[256];
  __shared__ double s_lnn;
  double acc = 0.0;
  for (int i = threadIdx.x; i < N; i += 256) acc = fma(l[i], l[i], acc);
  sv[threadIdx.x] = acc;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) sv[threadIdx.x] += sv[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    double s = kaa - sv[0];
    if (!(s > 0.0)) {
      info[0] = N + 1;
      s = 1.0;
    }
    s_lnn = sqrt(s);
    out[0] = s_lnn;
    out[1] = s;
  }
  __syncthreads();
  const double lnn = s_lnn, rinv = 1.0 / lnn;
  double* Arow = A + (long)N * npad;
  double* Wrow = W + (long)N * npad;
  for (int j = threadIdx.x; j < npad; j += 256) {
    if (j < N) {
      if (write_L) Arow[j] = l[j];
      Wrow[j] = -t[j] * rinv;
    } else if (j == N) {
      if (write_L) Arow[j] = lnn;
      Wrow[j] = rinv;
    } else {
      if (write_L) Arow[j] = 0.0;
      Wrow[j] = 0.0;
    }
  }
}

inline unsigned nblk(long long n, int b) { return (unsigned)((n + b - 1) / b); }

}  // namespace

// ---- host launchers ----------------------------------------------------------------------------
// ldl: row stride of L for the diagonal L[i * ldl + i] of the log-determinant (npad for the factor itself; 0 when
// L points at a packed copy of the diagonal)
int solve_alpha_launch(mfgp_ctx* h, const double* L, const double* W, int npad, int N,
                       const double* y, double* v_tmp, double* alpha, double* d_out3, int ldl) {
  trmv_lower_kernel<<<nblk(npad, 8), 256, 0, h->stream>>>(W, npad, y, N, v_tmp);
  LAUNCH_CHECK(h);
  trmv_lower_t_kernel<<<npad / 32, 256, 0, h->stream>>>(W, npad, v_tmp, alpha);
  LAUNCH_CHECK(h);
  lml_kernel<<<1, 256, 0, h->stream>>>(L, ldl, N, y, alpha, d_out3);
  LAUNCH_CHECK(h);
  return 0;
}


int kinv_apply_launch(mfgp_ctx* h, const double* W, int npad, int N, const double* k, double* l_tmp, double* u);

// l = W k and t = W^T l for the bordered update, then the finishing kernel
int append_point_launch(mfgp_ctx* h, const double* k, int N, int npad, double kaa, double* A, double* W,
                        int write_L, double* l_tmp, double* t_tmp, double* d_out2) {
  int rc = kinv_apply_launch(h, W, npad, N, k, l_tmp, t_tmp);
  if (rc) return rc;
  append_finish_kernel<<<1, 256, 0, h->stream>>>(l_tmp, t_tmp, N, npad, kaa, A, W, write_L, h->d_info, d_out2);
  LAUNCH_CHECK(h);
  return 0;
}

int cross_gen_launch(mfgp_ctx* h, const KParams& kp, const double* X, int N, int npad,
                     const double* alpha, const double* Xq, long long ncols, long long cols_pad,
                     double* Ks, double* mean) {
  if (cols_pad <= 0) return 0;
  const unsigned grid = nblk(cols_pad, 8);
  prof_begin(h, PC_CROSSGEN);
  if (cross_tile_launch(h, kp, X, N, npad, alpha, Xq, ncols, cols_pad, Ks, mean)) {   // large batches: tiled kernel
    prof_end(h, PC_CROSSGEN);
    LAUNCH_CHECK(h);
    return 0;
  }
#define MFGP_XGEN(DT)                                                                              \
  case DT:                                                                                         \
    cross_gen_fixed_kernel<DT><<<grid, 256, 0, h->stream>>>(kp, X, N, npad, alpha, Xq, ncols,      \
                                                            cols_pad, Ks, mean);                   \
    break;
  switch (kp.D) {
    MFGP_XGEN(1) MFGP_XGEN(2) MFGP_XGEN(3) MFGP_XGEN(4) MFGP_XGEN(5) MFGP_XGEN(6) MFGP_XGEN(7)
    MFGP_XGEN(8) MFGP_XGEN(9) MFGP_XGEN(10) MFGP_XGEN(11) MFGP_XGEN(12) MFGP_XGEN(13)
    default:
      cross_gen_kernel<<<grid, 256, 0, h->stream>>>(kp, X, N, npad, alpha, Xq, ncols, cols_pad, Ks,
                                                    mean);
  }
#undef MFGP_XGEN
  prof_end(h, PC_CROSSGEN);
  LAUNCH_CHECK(h);
  return 0;
}

// K7 generator for npts test points x S samples starting at point m_lo; zero-fills the pad columns
int cross_gen_mc_launch(mfgp_ctx* h, const KParams& kp, const double* X, int N, int npad,
                        const double* alpha, const double* Xtest, const double* mu_l,
                        const double* sd_l, const double* eps, unsigned long long seed,
                        long long m_global0, long long m_lo, long long npts, int S,
                        long long cols_pad, double* Ks, double* mu_c, const double* zcol, long long z_off,
                        long long ldz) {
  if (npts <= 0) return 0;
  ARG_CHECK(h, S <= MC_MAXS);
  prof_begin(h, PC_CROSSGEN);
  cross_gen_mc_kernel<<<(unsigned)npts, 256, fm::EXP_TBL_BYTES + 2 * ((S + 31) & ~31) * sizeof(double), h->stream>>>(
      kp, X, N, npad, alpha, Xtest, mu_l, sd_l, eps, seed, m_global0, m_lo, S, Ks, mu_c, zcol, z_off, ldz);
  prof_end(h, PC_CROSSGEN);
  LAUNCH_CHECK(h);
  const long long tail = (cols_pad - npts * S) * npad;
  if (tail > 0) {
    zero_rows_kernel<<<nblk(tail, 256), 256, 0, h->stream>>>(Ks + npts * S * npad, tail);
    LAUNCH_CHECK(h);
  }
  return 0;
}

int mc_small_applies(int N) { return N <= 64; }

// Fused generator + contraction for an upper level with N <= 64 (see mc_small_kernel).  Writes mu_c and the raw
// column sums of squares of the npts * S columns; returns 0 without launching (and *took = 0) when the level does
// not qualify.
int mc_small_launch(mfgp_ctx* h, const KParams& kp, const double* X, int N, int npad, const double* W,
                    const double* alpha, const double* Xtest, const double* mu_l, const double* sd_l,
                    const double* eps, unsigned long long seed, long long m_global0, long long m_lo,
                    long long npts, int S, double* mu_c, double* ss, const double* zcol, long long z_off,
                    long long ldz, int* took) {
  *took = 0;
  if (!mc_small_applies(N) || npts <= 0) return 0;
  const int NP = N <= 16 ? 16 : (N <= 32 ? 32 : 64);
  const size_t smem = (size_t)(256 + 2 * NP + kp.d * NP + MCS_WARPS * 2 * NP) * sizeof(double);
  const long long want = (npts + MCS_WARPS - 1) / MCS_WARPS;
  // exactly the resident CTAs: a warp walks over its share of the points, so the CTA's set-up (exp table, training
  // inputs, W fragments) is paid once per launch
  const long long cap = (long long)MFGP_NUM_SMS * (NP <= 32 ? 2 : 1);
  const unsigned grid = (unsigned)(want < cap ? want : cap);
  prof_begin(h, PC_TRMM_SUMSQ);
  if (NP == 16)
    mc_small_kernel<16><<<grid, MCS_WARPS * 32, smem, h->stream>>>(kp, X, N, npad, W, alpha, Xtest, mu_l, sd_l, eps, seed,
                                                                  m_global0, m_lo, npts, S, mu_c, ss, zcol, z_off, ldz);
  else if (NP == 32)
    mc_small_kernel<32><<<grid, MCS_WARPS * 32, smem, h->stream>>>(kp, X, N, npad, W, alpha, Xtest, mu_l, sd_l, eps, seed,
                                                                  m_global0, m_lo, npts, S, mu_c, ss, zcol, z_off, ldz);
  else
    mc_small_kernel<64><<<grid, MCS_WARPS * 32, smem, h->stream>>>(kp, X, N, npad, W, alpha, Xtest, mu_l, sd_l, eps, seed,
                                                                  m_global0, m_lo, npts, S, mu_c, ss, zcol, z_off, ldz);
  prof_end(h, PC_TRMM_SUMSQ);
  LAUNCH_CHECK(h);
  *took = 1;
  return 0;
}

int mc_max_samples() { return MC_MAXS; }

int predict_configure(mfgp_ctx* h) {
  CUDA_TRY(h, cudaFuncSetAttribute(cross_gen_mc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   fm::EXP_TBL_BYTES + 2 * MC_MAXS * (int)sizeof(double)));
  return 0;
}

int finish_var_launch(mfgp_ctx* h, const double* ss, long long n, double kdiag, double noise_add,
                      double* var, bool latent) {
  if (n <= 0) return 0;
  finish_var_kernel<<<nblk(n, 256), 256, 0, h->stream>>>(ss, n, kdiag, noise_add, latent ? -INFINITY : 1e-15, var);
  LAUNCH_CHECK(h);
  return 0;
}

int build_locs_launch(mfgp_ctx* h, const double* X, long long rows, int d, const double* d_offs,
                      int E, double tau, double* out) {
  long long total = rows * E * d;
  if (total <= 0) return 0;
  build_locs_kernel<<<nblk(total, 256), 256, 0, h->stream>>>(X, rows, d, d_offs, E, tau, out);
  LAUNCH_CHECK(h);
  return 0;
}

int concat_aug_launch(mfgp_ctx* h, const double* X, const double* vals, long long rows, int d, int E,
                      double* out) {
  long long total = rows * (d + E);
  if (total <= 0) return 0;
  concat_aug_kernel<<<nblk(total, 256), 256, 0, h->stream>>>(X, vals, rows, d, E, out);
  LAUNCH_CHECK(h);
  return 0;
}

int fill_normal_launch(mfgp_ctx* h, unsigned long long seed, long long first, long long count,
                       double* out) {
  if (count <= 0) return 0;
  fill_normal_kernel<<<nblk(count, 256), 256, 0, h->stream>>>(seed, first, count, out);
  LAUNCH_CHECK(h);
  return 0;
}

int build_mc_rows_launch(mfgp_ctx* h, const double* Xtest, const double* mu_l, const double* sd_l,
                         const double* eps, unsigned long long seed, long long m_global0,
                         long long m_lo, long long ncols, int S, int d, double* out) {
  if (ncols <= 0) return 0;
  build_mc_rows_kernel<<<nblk(ncols, 256), 256, 0, h->stream>>>(Xtest, mu_l, sd_l, eps, seed,
                                                                m_global0, m_lo, ncols, S, d, out);
  LAUNCH_CHECK(h);
  return 0;
}


int group_gram_launch(mfgp_ctx* h, const double* T, int npad, long long ldt, long long npts, int E, double* G) {
  if (npts <= 0) return 0;
#define MFGP_GG(E_)                                                                          \
  case E_:                                                                                   \
    group_gram_kernel<E_><<<nblk(npts, GG_PTS), GG_PTS * GG_RG, 0, h->stream>>>(T, npad, ldt, npts, G); \
    break;
  switch (E) {
    MFGP_GG(1) MFGP_GG(2) MFGP_GG(3) MFGP_GG(4) MFGP_GG(5) MFGP_GG(6) MFGP_GG(7) MFGP_GG(8)
    default:
      snprintf(h->err, sizeof(h->err), "joint low-fidelity sampling supports E <= 8 (got %d)", E);
      return -1;
  }
#undef MFGP_GG
  LAUNCH_CHECK(h);
  return 0;
}

int joint_chol_launch(mfgp_ctx* h, const double* G, const double* d_kab, long long npts, int E,
                      double diag_add, long long p_global0, double* Lc) {
  if (npts <= 0) return 0;
#define MFGP_JC(E_)                                                                                     \
  case E_:                                                                                              \
    joint_chol_kernel<E_><<<nblk(npts, 128), 128, 0, h->stream>>>(G, d_kab, npts, diag_add, p_global0, \
                                                                 Lc, h->d_info);                        \
    break;
  switch (E) {
    MFGP_JC(1) MFGP_JC(2) MFGP_JC(3) MFGP_JC(4) MFGP_JC(5) MFGP_JC(6) MFGP_JC(7) MFGP_JC(8)
    default:
      return -1;
  }
#undef MFGP_JC
  LAUNCH_CHECK(h);
  return 0;
}

int build_mc_rows_joint_launch(mfgp_ctx* h, const double* Xtest, const double* mu_l, const double* Lc,
                               const double* eps, unsigned long long seed, long long m_global0,
                               long long m_lo, long long ncols, int S, int d, int E, double* out) {
  if (ncols <= 0) return 0;
  build_mc_rows_joint_kernel<<<nblk(ncols, 256), 256, 0, h->stream>>>(Xtest, mu_l, Lc, eps, seed, m_global0,
                                                                      m_lo, ncols, S, d, E, out);
  LAUNCH_CHECK(h);
  return 0;
}

int sqrt_launch(mfgp_ctx* h, double* v, long long n) {
  if (n <= 0) return 0;
  sqrt_kernel<<<nblk(n, 256), 256, 0, h->stream>>>(v, n);
  LAUNCH_CHECK(h);
  return 0;
}

int mc_aggregate_launch(mfgp_ctx* h, const double* mu_c, const double* v_c, long long npts, int S,
                        double* mean, double* var) {
  if (npts <= 0) return 0;
  mc_aggregate_kernel<<<nblk(npts, 128), 128, 0, h->stream>>>(mu_c, v_c, npts, S, mean, var);
  LAUNCH_CHECK(h);
  return 0;
}

int argmax_launch(mfgp_ctx* h, const double* v, long long n, double* d_val, long long* d_idx) {
  int nb = (int)((n + 255) / 256);
  if (nb > RED_BLOCKS) nb = RED_BLOCKS;
  if (nb < 1) nb = 1;
  double* pval = h->d_partials;
  long long* pidx = reinterpret_cast<long long*>(h->d_partials + RED_BLOCKS);
  argmax_stage1_kernel<<<nb, 256, 0, h->stream>>>(v, n, pval, pidx);
  LAUNCH_CHECK(h);
  argmax_stage2_kernel<<<1, 256, 0, h->stream>>>(pval, pidx, nb, d_val, d_idx);
  LAUNCH_CHECK(h);
  return 0;
}

int acq_partials_doubles() { return 2 * RED_BLOCKS; }

// u = K_y^-1 k = W^T (W k) for one column k (zero on the pad); l_tmp, u: npad doubles
int kinv_apply_launch(mfgp_ctx* h, const double* W, int npad, int N, const double* k, double* l_tmp, double* u) {
  trmv_lower_kernel<<<nblk(npad, 8), 256, 0, h->stream>>>(W, npad, k, N, l_tmp);
  LAUNCH_CHECK(h);
  trmv_lower_t_kernel<<<npad / 32, 256, 0, h->stream>>>(W, npad, l_tmp, u);
  LAUNCH_CHECK(h);
  return 0;
}

int acq_coef_launch(mfgp_ctx* h, const double* u, int N, int npad1, double* coef) {
  acq_coef_kernel<<<nblk(npad1, 256), 256, 0, h->stream>>>(u, N, npad1, coef);
  LAUNCH_CHECK(h);
  return 0;
}

// kg == nullptr: arg-max of the first pick only.  partials: acq_partials_doubles(); best: [value, index bits]
int acq_update_launch(mfgp_ctx* h, const double* kg, double* R, long long C, int i, const double* rp, double rho,
                      double* v, double noise_add, double* partials, double* best) {
  int nb = (int)((C + 255) / 256);
  if (nb > RED_BLOCKS) nb = RED_BLOCKS;
  if (nb < 1) nb = 1;
  long long* pidx = reinterpret_cast<long long*>(partials + RED_BLOCKS);
  prof_begin(h, PC_ARGMAX);
  acq_update_kernel<<<nb, 256, 0, h->stream>>>(kg, R, C, i, rp, rho, v, noise_add, partials, pidx);
  prof_end(h, PC_ARGMAX);
  LAUNCH_CHECK(h);
  argmax_stage2_kernel<<<1, 256, 0, h->stream>>>(partials, pidx, nb, best, reinterpret_cast<long long*>(best + 1));
  LAUNCH_CHECK(h);
  return 0;
}

int acq_gather_launch(mfgp_ctx* h, const double* best, const double* v, const double* cands, int D,
                      const double* R, long long C, int nr, int q, double* out) {
  acq_gather_kernel<<<1, 128, 0, h->stream>>>(best, reinterpret_cast<const long long*>(best + 1), v, cands, D, R, C,
                                               nr, q, out);
  LAUNCH_CHECK(h);
  return 0;
}

int wdot_launch(mfgp_ctx* h, const double* w, const double* x, long long n, double* d_out) {
  int nb = (int)((n + 255) / 256);
  if (nb > RED_BLOCKS) nb = RED_BLOCKS;
  if (nb < 1) nb = 1;
  wdot_stage1_kernel<<<nb, 256, 0, h->stream>>>(w, x, n, h->d_partials);
  LAUNCH_CHECK(h);
  sum_stage2_kernel<<<1, 256, 0, h->stream>>>(h->d_partials, nb, d_out);
  LAUNCH_CHECK(h);
  return 0;
}

int sample_cols_launch(mfgp_ctx* h, const double* mu_c, const double* v_c, const double* eps,
                       unsigned long long key, long long m_global0, long long m_lo, long long ncols, int S,
                       double* z) {
  if (ncols <= 0) return 0;
  sample_cols_kernel<<<nblk(ncols, 256), 256, 0, h->stream>>>(mu_c, v_c, eps, key, m_global0, m_lo, ncols, S, z);
  LAUNCH_CHECK(h);
  return 0;
}

int fill_normal_padded_launch(mfgp_ctx* h, const double* eps, unsigned long long seed, long long M, int S,
                              long long rows, long long ldE, double* E) {
  if (rows * ldE <= 0) return 0;
  fill_normal_padded_kernel<<<nblk(rows * ldE, 256), 256, 0, h->stream>>>(eps, seed, M, S, rows, ldE, E);
  LAUNCH_CHECK(h);
  return 0;
}

int path_wsum_launch(mfgp_ctx* h, const double* mu_c, const double* w, long long m_lo, long long npts, int S,
                     double* path) {
  if (npts <= 0 || S <= 0) return 0;
  path_wsum_kernel<<<S, 256, 0, h->stream>>>(mu_c, w, m_lo, npts, S, path);
  LAUNCH_CHECK(h);
  return 0;
}

int point_service_launch(mfgp_ctx* h, const PointServiceArgs& a, PointServiceCtl* d_ctl, cudaStream_t stream) {
  point_service_kernel<<<1, 256, 0, stream>>>(a, d_ctl);
  LAUNCH_CHECK(h);
  return 0;
}

int predict_small_max_n() { return PS_MAXN; }

// lf may be null (Xq already augmented, width kp.D); else Xq holds plain inputs (width d) and Xaug_tmp
// receives the augmented rows.  All pointers device-accessible (mapped host memory included).
int predict_small_launch(mfgp_ctx* h, const KParams& kh, const mfgp_level_t* hf, const KParams* kl,
                         const mfgp_level_t* lf, const double* Xq, int M, const double* d_offs, int E, double tau,
                         double* Xaug_tmp, double noise_add, double* out) {
  const int npad = mfgp_padded_n(hf->N);
  const double* rows = Xq;
  if (lf) {
    augment_small_kernel<<<M * E, 256, 0, h->stream>>>(*kl, lf->d_X, lf->N, lf->d_alpha, Xq, lf->D, d_offs, E, tau,
                                                       Xaug_tmp);
    LAUNCH_CHECK(h);
    rows = Xaug_tmp;
  }
  predict_small_kernel<<<M, 256, 0, h->stream>>>(kh, hf->d_X, hf->N, npad, hf->d_alpha, hf->d_W, rows, noise_add, out);
  LAUNCH_CHECK(h);
  return 0;
}

// K1 covariance assembly and K5 gradient reduction.
//
// K1 replaces kern.K(X) for the reference's two kernels (src/abstractMFGP.py:59-60 and :62-80:
// RBF(z)*RBF(x) + RBF(x)) plus GPy's diag.add(Ky, noise + 1e-8): one fused pass, no N x N
// temporaries (GPy materialises three distance matrices and ~6 elementwise temporaries).
// The product k1*k2 is folded into a single exponential, so a composite element costs two exps.
// HBM-bound by contract (8 bytes written per element, inputs (N x D) stay in shared memory), but on
// B200 the FP64 pipe is the tighter bound: 2D + 3 + 2*8 + 1 FP64 instructions per composite element
// (30 at D = 5 -> 0.22 ms at N = 16384 with the pipe saturated, against 0.16 ms of HBM time for the
// lower triangle).  DMMA is no way out: it shares the FP64 units (tools/pipe_probe.cu: DFMA and DMMA
// streams serialise) and has the same FMA rate, so distances as a k-padded DMMA product cost as much
// as the direct form (tried in r01: 0.40 ms, tensor 31 % + fp64 34 %).  What keeps the kernel close:
//   - fastmath.cuh's exp2s (8 FP64 + 5 integer instructions + one table lookup, variances folded
//     into the exponent),
//   - input width D and the number of trailing z columns E as template parameters (distance loops
//     fully unrolled, all shared-memory reads of a sub-block issued up front),
//   - persistent CTAs (the 32 KB exp table is loaded once per CTA) that prefetch the NEXT tile's
//     input rows with cp.async while the current tile is computed,
//   - a thread mapping whose 16-byte shared reads and global stores are contiguous per half-warp
//     (minimum LDS wavefronts; every STG covers whole 32-byte sectors: the store pattern alone
//     sustains 5.3 TB/s),
//   - 2 x 4 elements per thread and sub-block at 2 CTAs per SM (119 registers, the eight exponentials
//     of a thread interleaved by the scheduler).
// Measured (tools/exp_probe.cu): exp2s sustains 25 cycles per warp against the 16-cycle FP64 bound --
// the table LDS.64 costs ~4 cycles of issue, the clamp ~2 -- which is what holds K1 at ~0.36 ms.
//
// K5 replaces GPy's update_gradients_full chain (stationary.py / prod.py / add.py) for
// dL_dK = 0.5 (alpha alpha^T - K^-1): one streaming pass over K^-1's lower triangle that
// recomputes the kernel factors from X on the fly and produces six sums
//   S0 = sum G K12, S1 = sum G K12 rz2, S2 = sum G K12 rx2, S3 = sum G K3, S4 = sum G K3 rx2, S5 = tr G
// in a fixed order (persistent blocks, fixed tile->block map, two-stage reduction).
#include "common.cuh"
#include "fastmath.cuh"

namespace {

constexpr int BT = 128;          // CTA tile edge
#ifndef MFGP_ASM_RI      // tuning overrides (tools/build_variants.sh); the defaults are the measured best
#define MFGP_ASM_RI 2
#endif
#ifndef MFGP_ASM_CTAS
#define MFGP_ASM_CTAS 2
#endif
constexpr int RI = MFGP_ASM_RI;  // rows per thread and sub-block
// sub-block: SBR rows x SBC columns; thread (ty,tx) owns rows ty+16i and the column pairs
// {2tx, 2tx+1} and {32+2tx, 33+2tx}: a half-warp's 16-byte accesses are then contiguous (256 B), so
// shared-memory reads take the minimum number of wavefronts and every global store / load
// instruction covers whole 32-byte sectors
constexpr int SBR = 16 * RI;
constexpr int SBC = 64;
constexpr int NSB = (BT / SBR) * (BT / SBC);
constexpr int CTAS_PER_SM = MFGP_ASM_CTAS;
constexpr int MAX_DT = 8;        // widths with a specialised kernel

__device__ __forceinline__ int col_of(int tx, int j) { return (j >> 1) * 32 + 2 * tx + (j & 1); }

__device__ __forceinline__ void tile_from_linear(int tt, int& ti, int& tj) {
  ti = (int)((sqrt(8.0 * tt + 1.0) - 1.0) * 0.5);
  while ((long)(ti + 1) * (ti + 2) / 2 <= tt) ti++;
  while ((long)ti * (ti + 1) / 2 > tt) ti--;
  tj = tt - ti * (ti + 1) / 2;
}

__device__ __forceinline__ void cp_async8_zfill(double* sdst, const double* gsrc, bool valid) {
  const unsigned s = (unsigned)__cvta_generic_to_shared(sdst);
  const int n = valid ? 8 : 0;   // src-size 0: nothing is read, the destination is zero-filled
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;\n" ::"r"(s), "l"(gsrc), "r"(n));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int K>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(K)); }

// sX[dd][r] = X[row0 + r][dd] for r < BT (0 beyond N), asynchronously.  The tile's rows are one
// contiguous run of BT*D doubles of X, so the global side is perfectly coalesced; the transposition
// to dd-major (a row of threads then reads consecutive shared-memory words) happens in the copy.
template <int DT>
__device__ __forceinline__ void prefetch_rows(double* sX, const double* __restrict__ X, int N, int Drt,
                                              int row0) {
  const int D = DT > 0 ? DT : Drt;
  const double* base = X + (long)row0 * D;
  for (int i = threadIdx.x; i < BT * D; i += blockDim.x) {
    const int r = i / D, dd = i - r * D;
    const bool ok = row0 + r < N;
    cp_async8_zfill(sX + dd * BT + r, ok ? base + i : X, ok);
  }
}

// Squared distances of the thread's RI x 4 sub-block.  DT > 0: width and split known at compile
// time (x = first DT-E columns, z = the last E); DT == 0: runtime D and d.
template <int DT, int E>
__device__ __forceinline__ void sub_block_dist(const double* sXi, const double* sXj, int Drt, int drt,
                                               int tx, int ty, double (&rx)[RI][4], double (&rz)[RI][4]) {
#pragma unroll
  for (int i = 0; i < RI; i++)
#pragma unroll
    for (int j = 0; j < 4; j++) rx[i][j] = rz[i][j] = 0.0;
  if (DT > 0) {
#pragma unroll
    for (int dd = 0; dd < DT; dd++) {
      double xi[RI], xj[4];
#pragma unroll
      for (int i = 0; i < RI; i++) xi[i] = sXi[dd * BT + ty + 16 * i];             // broadcast within a half-warp
      const double2 p0 = *reinterpret_cast<const double2*>(sXj + dd * BT + 2 * tx);   // 16 lanes x 16 B contiguous
      const double2 p1 = *reinterpret_cast<const double2*>(sXj + dd * BT + 32 + 2 * tx);
      xj[0] = p0.x; xj[1] = p0.y; xj[2] = p1.x; xj[3] = p1.y;
#pragma unroll
      for (int i = 0; i < RI; i++)
#pragma unroll
        for (int j = 0; j < 4; j++) {
          const double t = xi[i] - xj[j];
          if (dd < DT - E) rx[i][j] = fma(t, t, rx[i][j]);
          else rz[i][j] = fma(t, t, rz[i][j]);
        }
    }
  } else {
    for (int dd = 0; dd < Drt; dd++) {
      double xi[RI], xj[4];
#pragma unroll
      for (int i = 0; i < RI; i++) xi[i] = sXi[dd * BT + ty + 16 * i];
      const double2 p0 = *reinterpret_cast<const double2*>(sXj + dd * BT + 2 * tx);
      const double2 p1 = *reinterpret_cast<const double2*>(sXj + dd * BT + 32 + 2 * tx);
      xj[0] = p0.x; xj[1] = p0.y; xj[2] = p1.x; xj[3] = p1.y;
      if (dd < drt) {
#pragma unroll
        for (int i = 0; i < RI; i++)
#pragma unroll
          for (int j = 0; j < 4; j++) {
            const double t = xi[i] - xj[j];
            rx[i][j] = fma(t, t, rx[i][j]);
          }
      } else {
#pragma unroll
        for (int i = 0; i < RI; i++)
#pragma unroll
          for (int j = 0; j < 4; j++) {
            const double t = xi[i] - xj[j];
            rz[i][j] = fma(t, t, rz[i][j]);
          }
      }
    }
  }
}

// element value from the two squared distances (exp2s form, see KParams)
template <int DT, int E>
struct KEval {
  double uz, ux, lc12, u3, ls3;
  bool has3;
  unsigned tbl;
  __device__ __forceinline__ KEval(const KParams& kp, unsigned tbl_)
      : uz(kp.uz), ux(kp.ux), lc12(kp.lc12), u3(kp.u3), ls3(kp.ls3), has3(kp.s3 != 0.0), tbl(tbl_) {}
  __device__ __forceinline__ double k12(double rx, double rz) const {
    if (DT > 0 && E == 0) return fm::exp2s(fma(ux, rx, lc12), tbl);   // no z columns: rz == 0
    return fm::exp2s(fma(uz, rz, fma(ux, rx, lc12)), tbl);
  }
  __device__ __forceinline__ double k3(double rx) const { return fm::exp2s(fma(u3, rx, ls3), tbl); }
};

template <bool VEC, int DT, int E>
__global__ void __launch_bounds__(256, CTAS_PER_SM)
    assemble_kernel(KParams kp, const double* __restrict__ X, int N, double diag_add,
                    double* __restrict__ K, long ldk, int lower_only, int tiles, int nrows, int ntiles) {
  extern __shared__ __align__(16) double dsm[];   // exp table | 2 x (sXi[D][BT] | sXj[D][BT])
  const int D = DT > 0 ? DT : kp.D, d = DT > 0 ? DT - E : kp.d;
  double* sX = dsm + fm::EXP_TBL_DOUBLES;
  const int panel = 2 * D * BT;
  fm::load_exp_table(dsm, kp.exp_tbl);
  const KEval<DT, E> ke(kp, fm::lane_table(dsm));
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  auto tile_rc = [&](int tile, int& ti, int& tj) {
    if (lower_only) {
      tile_from_linear(tile, ti, tj);
    } else {
      ti = tile / tiles;
      tj = tile % tiles;
    }
  };
  auto prefetch = [&](int tile, int buf) {
    int ti, tj;
    tile_rc(tile, ti, tj);
    prefetch_rows<DT>(sX + buf * panel, X, N, D, ti * BT);
    prefetch_rows<DT>(sX + buf * panel + D * BT, X, N, D, tj * BT);
  };
  int buf = 0;
  if ((int)blockIdx.x < ntiles) prefetch(blockIdx.x, 0);
  cp_async_commit();
  // persistent, static round-robin over the tiles; the next tile's rows land while this one is computed
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, buf ^= 1) {
    if (tile + (int)gridDim.x < ntiles) prefetch(tile + gridDim.x, buf ^ 1);
    cp_async_commit();
    cp_async_wait<1>();
    __syncthreads();
    int ti, tj;
    tile_rc(tile, ti, tj);
    const double* sXi = sX + buf * panel;
    const double* sXj = sXi + D * BT;
#pragma unroll 1
    for (int sb = 0; sb < NSB; sb++) {
      const int si = sb >> 1, sj = sb & 1;
      const int row0 = ti * BT + si * SBR, col0 = tj * BT + sj * SBC;
      if (row0 >= nrows || col0 >= nrows) continue;
      if (lower_only && col0 >= row0 + SBR) continue;   // sub-block strictly above the diagonal
      double rx[RI][4], rz[RI][4];
      sub_block_dist<DT, E>(sXi + si * SBR, sXj + sj * SBC, D, d, tx, ty, rx, rz);
      const bool on_diag = col0 < row0 + SBR && row0 < col0 + SBC;   // the diagonal crosses this sub-block
      if (row0 + SBR <= N && col0 + SBC <= N && !on_diag) {
        // Interior sub-block (almost all of them): straight-line code, no per-element predicates
        double v[RI][4];
#pragma unroll
        for (int i = 0; i < RI; i++)
#pragma unroll
          for (int j = 0; j < 4; j++) v[i][j] = ke.k12(rx[i][j], rz[i][j]);
        if (ke.has3) {
#pragma unroll
          for (int i = 0; i < RI; i++)
#pragma unroll
            for (int j = 0; j < 4; j++) v[i][j] += ke.k3(rx[i][j]);
        }
#pragma unroll
        for (int i = 0; i < RI; i++) {
          double* dst = K + (long)(row0 + ty + 16 * i) * ldk + col0 + 2 * tx;
          if (VEC) {
            *reinterpret_cast<double2*>(dst) = make_double2(v[i][0], v[i][1]);
            *reinterpret_cast<double2*>(dst + 32) = make_double2(v[i][2], v[i][3]);
          } else {
            dst[0] = v[i][0]; dst[1] = v[i][1]; dst[32] = v[i][2]; dst[33] = v[i][3];
          }
        }
        continue;
      }
#pragma unroll
      for (int i = 0; i < RI; i++) {
        const int r = row0 + ty + 16 * i;
        if (r >= nrows) continue;
        double v[4];
#pragma unroll
        for (int j = 0; j < 4; j++) {
          const int c = col0 + col_of(tx, j);
          double val;
          if (r < N && c < N) {
            val = ke.k12(rx[i][j], rz[i][j]);
            if (ke.has3) val += ke.k3(rx[i][j]);
            if (r == c) val += diag_add;
          } else {
            val = (r == c) ? 1.0 : 0.0;   // identity pad block
          }
          v[j] = val;
        }
        double* dst = K + (long)r * ldk + col0;
        if (VEC) {
          // nrows is a multiple of 64 here (padded buffer): no column guard needed
          *reinterpret_cast<double2*>(dst + 2 * tx) = make_double2(v[0], v[1]);
          *reinterpret_cast<double2*>(dst + 32 + 2 * tx) = make_double2(v[2], v[3]);
        } else {
#pragma unroll
          for (int j = 0; j < 4; j++)
            if (col0 + col_of(tx, j) < nrows) dst[col_of(tx, j)] = v[j];
        }
      }
    }
    __syncthreads();   // all readers done with this buffer before the next iteration refills it
  }
  cp_async_wait<0>();
}


constexpr int GR_BLOCKS = MFGP_NUM_SMS * CTAS_PER_SM;   // persistent; fixed tile -> block map

template <int DT, int E>
__global__ void __launch_bounds__(256, CTAS_PER_SM)
    grad_reduce_kernel(KParams kp, const double* __restrict__ X, int N,
                       const double* __restrict__ Kinv, long ld, const double* __restrict__ alpha,
                       int ntiles_lin, double* __restrict__ partials) {
  extern __shared__ __align__(16) double dsm[];   // exp table | 2 x (sXi[D][BT] | sXj[D][BT] | ai[BT] | aj[BT])
  __shared__ double red[8][6];
  const int D = DT > 0 ? DT : kp.D, d = DT > 0 ? DT - E : kp.d;
  double* sX = dsm + fm::EXP_TBL_DOUBLES;
  const int panel = 2 * (D + 1) * BT;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  fm::load_exp_table(dsm, kp.exp_tbl);
  const KEval<DT, E> ke(kp, fm::lane_table(dsm));
  const bool has3 = ke.has3;
  auto prefetch = [&](int tt, int buf) {
    int ti, tj;
    tile_from_linear(tt, ti, tj);
    double* p = sX + buf * panel;
    prefetch_rows<DT>(p, X, N, D, ti * BT);
    prefetch_rows<DT>(p + D * BT, X, N, D, tj * BT);
    const int r = (threadIdx.x < BT ? ti : tj) * BT + (threadIdx.x & (BT - 1));
    cp_async8_zfill(p + 2 * D * BT + threadIdx.x, r < N ? alpha + r : alpha, r < N);
  };
  double S[6] = {0, 0, 0, 0, 0, 0};
  int buf = 0;
  if ((int)blockIdx.x < ntiles_lin) prefetch(blockIdx.x, 0);
  cp_async_commit();
  for (int tt = blockIdx.x; tt < ntiles_lin; tt += gridDim.x, buf ^= 1) {
    if (tt + (int)gridDim.x < ntiles_lin) prefetch(tt + gridDim.x, buf ^ 1);
    cp_async_commit();
    cp_async_wait<1>();
    __syncthreads();
    int ti, tj;
    tile_from_linear(tt, ti, tj);
    const double* sXi_t = sX + buf * panel;
    const double* sXj_t = sXi_t + D * BT;
    const double* sAi_t = sXi_t + 2 * D * BT;
    const double* sAj_t = sAi_t + BT;
#pragma unroll 1
    for (int sb = 0; sb < NSB; sb++) {
      const int si = sb >> 1, sj = sb & 1;
      const int row0 = ti * BT + si * SBR, col0 = tj * BT + sj * SBC;
      if (row0 >= N || col0 >= row0 + SBR) continue;   // beyond the data / strictly above the diagonal
      const double* sAi = sAi_t + si * SBR;
      const double* sAj = sAj_t + sj * SBC;
      // issue the K^-1 loads first so that they overlap the distance computation
      double kin[RI][4];
#pragma unroll
      for (int i = 0; i < RI; i++) {
        const int r = row0 + ty + 16 * i;
        if (r < N) {
          const double* src = Kinv + (long)r * ld + col0 + 2 * tx;
          const double2 q0 = *reinterpret_cast<const double2*>(src);
          const double2 q1 = *reinterpret_cast<const double2*>(src + 32);
          kin[i][0] = q0.x; kin[i][1] = q0.y; kin[i][2] = q1.x; kin[i][3] = q1.y;
        } else {
          kin[i][0] = kin[i][1] = kin[i][2] = kin[i][3] = 0.0;
        }
      }
      double rx[RI][4], rz[RI][4];
      sub_block_dist<DT, E>(sXi_t + si * SBR, sXj_t + sj * SBC, D, d, tx, ty, rx, rz);
      const double2 a0 = *reinterpret_cast<const double2*>(sAj + 2 * tx);
      const double2 a1 = *reinterpret_cast<const double2*>(sAj + 32 + 2 * tx);
      const double aj[4] = {a0.x, a0.y, a1.x, a1.y};
      if (col0 + SBC <= row0 && row0 + SBR <= N) {
        // interior sub-block strictly below the diagonal: every element counts twice (weight 1)
#pragma unroll
        for (int i = 0; i < RI; i++) {
          const double ai = sAi[ty + 16 * i];
#pragma unroll
          for (int j = 0; j < 4; j++) {
            const double G = fma(ai, aj[j], -kin[i][j]);
            const double gk = G * ke.k12(rx[i][j], rz[i][j]);
            S[0] += gk;
            if (!(DT > 0 && E == 0)) S[1] = fma(gk, rz[i][j], S[1]);
            S[2] = fma(gk, rx[i][j], S[2]);
            if (has3) {
              const double g3 = G * ke.k3(rx[i][j]);
              S[3] += g3;
              S[4] = fma(g3, rx[i][j], S[4]);
            }
          }
        }
        continue;
      }
#pragma unroll
      for (int i = 0; i < RI; i++) {
        const int r = row0 + ty + 16 * i;
        if (r >= N) continue;
        const double ai = sAi[ty + 16 * i];
#pragma unroll
        for (int j = 0; j < 4; j++) {
          const int c = col0 + col_of(tx, j);
          if (c > r || c >= N) continue;
          const double w = (c == r) ? 0.5 : 1.0;   // G = 0.5(aa^T - Kinv); off-diagonal counted twice
          const double G = w * fma(ai, aj[j], -kin[i][j]);
          const double gk = G * ke.k12(rx[i][j], rz[i][j]);
          S[0] += gk;
          S[1] = fma(gk, rz[i][j], S[1]);
          S[2] = fma(gk, rx[i][j], S[2]);
          if (has3) {
            const double g3 = G * ke.k3(rx[i][j]);
            S[3] += g3;
            S[4] = fma(g3, rx[i][j], S[4]);
          }
          if (c == r) S[5] += G;
        }
      }
    }
    __syncthreads();
  }
  cp_async_wait<0>();
  // block reduction in a fixed order
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int q = 0; q < 6; q++) {
    double v = S[q];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0) red[warp][q] = v;
  }
  __syncthreads();
  if (threadIdx.x < 6) {
    double v = 0.0;
    for (int w = 0; w < 8; w++) v += red[w][threadIdx.x];
    partials[blockIdx.x * 8 + threadIdx.x] = v;
  }
}

__global__ void reduce_partials_kernel(const double* __restrict__ partials, int nblocks,
                                       double* __restrict__ out8) {
  // 6 warps, one quantity each; lanes stride over blocks, then a shuffle tree: fixed order
  const int q = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (q >= 6) return;
  double v = 0.0;
  for (int b = lane; b < nblocks; b += 32) v += partials[b * 8 + q];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  if (lane == 0) out8[q] = v;
}

// ---- dispatch on (input width, trailing z columns) -----------------------------------------------
// RBF kind: az == ax, so every column is treated as an x column (E = 0).  Composite: E = D - d.
// Specialised for D <= 8 with E in {0, 1} (plain GP levels, NARGP, GPDF) and for the composite kernel
// with two backward delays in 1-D and 2-D (GPDFC: d = 1, E = 3 and d = 2, E = 5, tests/test_mfgp_adapt_2d.py:27);
// everything else (D > 8, other composite splits) takes the runtime-width kernel.
struct Shape {
  int DT, E;
};
Shape shape_of(const KParams& kp) {
  const int E = kp.kind == MFGP_KIND_RBF ? 0 : kp.D - kp.d;
  if (kp.D <= MAX_DT && E <= 1) return {kp.D, E};
  if ((kp.D == 4 && E == 3) || (kp.D == 7 && E == 5)) return {kp.D, E};
  return {0, 0};
}


// ---- K6a, tiled: cross-covariance block Ks[c][k] = K(q_c, X_k) and mean[c] = sum_k Ks[c][k] alpha_k -------
// Same machinery as K1 (compile-time widths, exp2s, sector-complete thread mapping, cp.async
// double-buffering), on a rectangular problem: a CTA owns 128 query rows and walks the training points
// in tiles of 128, so the mean accumulates in registers and is reduced once, in a fixed order.  Replaces
// the one-warp-per-query kernel (4 global loads per element, ~5 % of the FP64 pipe) for large batches.
template <int DT, int E>
__global__ void __launch_bounds__(256, CTAS_PER_SM)
    cross_tile_kernel(KParams kp, const double* __restrict__ X, int N, int npad,
                      const double* __restrict__ alpha, const double* __restrict__ Xq, long ncols,
                      double* __restrict__ Ks, double* __restrict__ mean) {
  extern __shared__ __align__(16) double dsm[];   // exp table | sXq[D][BT] | 2 x (sXk[D][BT] | alpha[BT])
  constexpr int D = DT;
  double* sXq = dsm + fm::EXP_TBL_DOUBLES;
  double* sK = sXq + D * BT;
  constexpr int kpanel = (D + 1) * BT;
  fm::load_exp_table(dsm, kp.exp_tbl);
  const KEval<DT, E> ke(kp, fm::lane_table(dsm));
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const long c0 = (long)blockIdx.x * BT;
  const int ktiles = npad / BT;
  // query rows of this CTA (zero beyond ncols): the cp.async helper takes an int row count
  {
    const long left = ncols - c0;
    prefetch_rows<DT>(sXq, Xq + c0 * D, left > BT ? BT : (left > 0 ? (int)left : 0), D, 0);
  }
  auto prefetch_k = [&](int kt, int buf) {
    double* p = sK + buf * kpanel;
    prefetch_rows<DT>(p, X, N, D, kt * BT);
    if (threadIdx.x < BT) {
      const int r = kt * BT + threadIdx.x;
      cp_async8_zfill(p + D * BT + threadIdx.x, r < N ? alpha + r : alpha, r < N);
    }
  };
  prefetch_k(0, 0);
  cp_async_commit();
  double macc[BT / SBR][RI];
#pragma unroll
  for (int q = 0; q < BT / SBR; q++)
#pragma unroll
    for (int i = 0; i < RI; i++) macc[q][i] = 0.0;
  int buf = 0;
  for (int kt = 0; kt < ktiles; kt++, buf ^= 1) {
    if (kt + 1 < ktiles) prefetch_k(kt + 1, buf ^ 1);
    cp_async_commit();
    cp_async_wait<1>();
    __syncthreads();
    const double* sXk = sK + buf * kpanel;
    const double* sAk = sXk + D * BT;
    const int kbase = kt * BT;
#pragma unroll
    for (int si = 0; si < BT / SBR; si++) {
      const long row0 = c0 + si * SBR;
#pragma unroll 1
      for (int sj = 0; sj < BT / SBC; sj++) {
        const int col0 = kbase + sj * SBC;
        double rx[RI][4], rz[RI][4];
        sub_block_dist<DT, E>(sXq + si * SBR, sXk + sj * SBC, D, D - E, tx, ty, rx, rz);
        double v[RI][4];
#pragma unroll
        for (int i = 0; i < RI; i++)
#pragma unroll
          for (int j = 0; j < 4; j++) v[i][j] = ke.k12(rx[i][j], rz[i][j]);
        if (ke.has3) {
#pragma unroll
          for (int i = 0; i < RI; i++)
#pragma unroll
            for (int j = 0; j < 4; j++) v[i][j] += ke.k3(rx[i][j]);
        }
        if (col0 + SBC > N || row0 + SBR > ncols) {   // ragged edge: pad entries are exactly zero
#pragma unroll
          for (int i = 0; i < RI; i++)
#pragma unroll
            for (int j = 0; j < 4; j++)
              if (row0 + ty + 16 * i >= ncols || col0 + col_of(tx, j) >= N) v[i][j] = 0.0;
        }
        const double2 a0 = *reinterpret_cast<const double2*>(sAk + sj * SBC + 2 * tx);
        const double2 a1 = *reinterpret_cast<const double2*>(sAk + sj * SBC + 32 + 2 * tx);
#pragma unroll
        for (int i = 0; i < RI; i++) {
          macc[si][i] = fma(v[i][0], a0.x, macc[si][i]);
          macc[si][i] = fma(v[i][1], a0.y, macc[si][i]);
          macc[si][i] = fma(v[i][2], a1.x, macc[si][i]);
          macc[si][i] = fma(v[i][3], a1.y, macc[si][i]);
          if (Ks) {
            double* dst = Ks + (row0 + ty + 16 * i) * (long)npad + col0 + 2 * tx;
            *reinterpret_cast<double2*>(dst) = make_double2(v[i][0], v[i][1]);
            *reinterpret_cast<double2*>(dst + 32) = make_double2(v[i][2], v[i][3]);
          }
        }
      }
    }
    __syncthreads();
  }
  cp_async_wait<0>();
  if (mean) {
    // reduce over the 16 tx lanes of a half-warp (fixed shuffle tree), one value per query row
#pragma unroll
    for (int si = 0; si < BT / SBR; si++)
#pragma unroll
      for (int i = 0; i < RI; i++) {
        double m = macc[si][i];
#pragma unroll
        for (int o = 8; o > 0; o >>= 1) m += __shfl_xor_sync(0xffffffffu, m, o);
        const long c = c0 + si * SBR + ty + 16 * i;
        if (tx == 0 && c < ncols) mean[c] = m;
      }
  }
}

constexpr size_t cross_smem(int D) {
  return fm::EXP_TBL_BYTES + ((size_t)D * BT + 2 * (size_t)(D + 1) * BT) * sizeof(double);
}

// ---- K6d: predictive gradients of one level -------------------------------------------------------------------
//   dmean[c][j] = 2 sum_k alpha_k (q_cj - X_kj) w_kj,   dvar[c][j] = -4 sum_k u_kc (q_cj - X_kj) w_kj
//   w = ax k12 + a3 k3 for an x column, az k12 for a z column (u_c = K_y^-1 k_c, rows of Ut = Ks K_y^-1);
// by-products mean[c] = sum_k alpha_k k and quad[c] = sum_k u_kc k (the variance is kdiag - quad).
// A CTA owns 128 queries and walks the training points in double-buffered stages of GK (cp.async: their rows,
// alpha, and the matching 128 x GK block of Ut, whose rows are contiguous in global memory).  Thread t serves
// query t/2 and the stage's points k = 2m + t%2; the two partial sums of a query meet in one shuffle at the end, so
// every sum runs in a fixed order that depends on nothing but N.  DT = 0 (runtime width) accumulates the gradient
// columns [j0, j0 + GJ) per launch.
constexpr int GK = 16;           // training points per stage
constexpr int GU_LD = GK + 2;    // Ut stage row stride: a half-warp's reads (8 queries x 2 points) hit 16 bank pairs
constexpr int GJ = 8;            // gradient columns per launch of the runtime-width kernel

template <int DT, int E>
__global__ void __launch_bounds__(256, 2)
    cross_grad_kernel(KParams kp, const double* __restrict__ X, int N, const double* __restrict__ alpha,
                      const double* __restrict__ Ut, long ldu, const double* __restrict__ Xq, long ncols, int j0,
                      double* __restrict__ dmean, double* __restrict__ dvar, double* __restrict__ mean,
                      double* __restrict__ quad) {
  extern __shared__ __align__(16) double dsm[];   // exp table | sXq[D][BT] | 2 x (sXk[D][GK] | alpha[GK] | sU[BT][GU_LD])
  const int D = DT > 0 ? DT : kp.D, d = DT > 0 ? DT - E : kp.d;
  constexpr int NJ = DT > 0 ? DT : GJ;
  double* sXq = dsm + fm::EXP_TBL_DOUBLES;
  double* sSt = sXq + D * BT;
  const int stage = D * GK + GK + BT * GU_LD;
  fm::load_exp_table(dsm, kp.exp_tbl);
  const KEval<DT, E> ke(kp, fm::lane_table(dsm));
  const bool has3 = ke.has3, want_u = Ut != nullptr;
  const double ax = kp.ax, az = kp.az, a3 = kp.a3;
  const long c0 = (long)blockIdx.x * BT;
  const int cl = threadIdx.x >> 1, h = threadIdx.x & 1;
  {
    const long left = ncols - c0;
    prefetch_rows<DT>(sXq, Xq + c0 * D, left > BT ? BT : (int)left, D, 0);
  }
  auto prefetch = [&](int s, int buf) {
    double* p = sSt + buf * stage;
    const int k0 = s * GK;
    for (int i = threadIdx.x; i < GK * D; i += blockDim.x) {   // rows k0.. are one contiguous run of X
      const int r = i / D, dd = i - r * D;
      const bool ok = k0 + r < N;
      cp_async8_zfill(p + dd * GK + r, ok ? X + (long)k0 * D + i : X, ok);
    }
    if (threadIdx.x < GK) {
      const bool ok = k0 + (int)threadIdx.x < N;
      cp_async8_zfill(p + D * GK + threadIdx.x, ok ? alpha + k0 + threadIdx.x : alpha, ok);
    }
    if (want_u) {
      double* su = p + D * GK + GK;
      for (int i = threadIdx.x; i < BT * GK; i += blockDim.x) {
        const int r = i / GK, kk = i - r * GK;
        const bool ok = c0 + r < ncols && k0 + kk < N;
        cp_async8_zfill(su + r * GU_LD + kk, ok ? Ut + (c0 + r) * ldu + k0 + kk : Ut, ok);
      }
    }
  };
  const int nst = (N + GK - 1) / GK;
  prefetch(0, 0);
  cp_async_commit();
  double gm[NJ], gv[NJ], q[DT > 0 ? DT : 1];
#pragma unroll
  for (int j = 0; j < NJ; j++) gm[j] = gv[j] = 0.0;
  double am = 0.0, aq = 0.0;
  int buf = 0;
  for (int s = 0; s < nst; s++, buf ^= 1) {
    if (s + 1 < nst) prefetch(s + 1, buf ^ 1);
    cp_async_commit();
    cp_async_wait<1>();
    __syncthreads();
    if (DT > 0 && s == 0) {
#pragma unroll
      for (int dd = 0; dd < (DT > 0 ? DT : 1); dd++) q[dd] = sXq[dd * BT + cl];
    }
    const double* sXk = sSt + buf * stage;
    const double* sA = sXk + D * GK;
    const double* sU = sA + GK;
#pragma unroll 2
    for (int m = 0; m < GK / 2; m++) {
      const int k = 2 * m + h;
      double t[NJ];
      double rx = 0.0, rz = 0.0;
      if (DT > 0) {
#pragma unroll
        for (int dd = 0; dd < NJ; dd++) {
          t[dd] = q[dd] - sXk[dd * GK + k];
          if (dd < DT - E) rx = fma(t[dd], t[dd], rx);
          else rz = fma(t[dd], t[dd], rz);
        }
      } else {
        for (int dd = 0; dd < D; dd++) {
          const double tt = sXq[dd * BT + cl] - sXk[dd * GK + k];
          if (dd < d) rx = fma(tt, tt, rx);
          else rz = fma(tt, tt, rz);
        }
#pragma unroll
        for (int jj = 0; jj < NJ; jj++) {
          const int j = j0 + jj;
          t[jj] = j < D ? sXq[j * BT + cl] - sXk[j * GK + k] : 0.0;
        }
      }
      const double k12 = ke.k12(rx, rz);
      const double k3 = has3 ? ke.k3(rx) : 0.0;
      const double kv = k12 + k3;
      const double gx = has3 ? fma(ax, k12, a3 * k3) : ax * k12, gz = az * k12;
      const double a = sA[k];
      am = fma(a, kv, am);
      const double wax = a * gx, waz = a * gz;
#pragma unroll
      for (int jj = 0; jj < NJ; jj++) {
        const bool xcol = DT > 0 ? jj < DT - E : j0 + jj < d;
        gm[jj] = fma(t[jj], xcol ? wax : waz, gm[jj]);
      }
      if (want_u) {
        const double u = sU[cl * GU_LD + k];
        aq = fma(u, kv, aq);
        const double wux = u * gx, wuz = u * gz;
#pragma unroll
        for (int jj = 0; jj < NJ; jj++) {
          const bool xcol = DT > 0 ? jj < DT - E : j0 + jj < d;
          gv[jj] = fma(t[jj], xcol ? wux : wuz, gv[jj]);
        }
      }
    }
    __syncthreads();   // all readers done with this buffer before the next iteration refills it
  }
  cp_async_wait<0>();
  // the two halves of a query sit in adjacent lanes: one shuffle, the same sum in both
#pragma unroll
  for (int jj = 0; jj < NJ; jj++) {
    gm[jj] += __shfl_xor_sync(0xffffffffu, gm[jj], 1);
    gv[jj] += __shfl_xor_sync(0xffffffffu, gv[jj], 1);
  }
  am += __shfl_xor_sync(0xffffffffu, am, 1);
  aq += __shfl_xor_sync(0xffffffffu, aq, 1);
  const long c = c0 + cl;
  if (h != 0 || c >= ncols) return;
#pragma unroll
  for (int jj = 0; jj < NJ; jj++) {
    const int j = (DT > 0 ? 0 : j0) + jj;
    if (DT == 0 && j >= D) break;
    dmean[c * D + j] = 2.0 * gm[jj];
    if (dvar) dvar[c * D + j] = -4.0 * gv[jj];
  }
  if (DT > 0 || j0 == 0) {
    if (mean) mean[c] = am;
    if (quad) quad[c] = aq;
  }
}

constexpr size_t xgrad_smem(int D) {
  return fm::EXP_TBL_BYTES + ((size_t)D * BT + 2 * ((size_t)D * GK + GK + (size_t)BT * GU_LD)) * sizeof(double);
}

// ---- K8c: integrated-variance (ALC) reduction ------------------------------------------------------------------
//   alc[c] = sum_r w_r (k(c, r) - G[c][r])^2 / (kdiag - sum_i Tt[c][i]^2 + s2),  -inf where the denominator is <= 0
// with G = Tt_C Tt_R^T (the latent posterior covariance is k - G).  The layout is cross_grad_kernel's: a CTA owns
// 128 candidates and walks the reference rows in double-buffered stages of GK (cp.async: their rows, weights, and
// the matching 128 x GK block of G).  Thread t serves candidate t/2 and the stage's references r = 2m + t%2; the two
// partial sums meet in one shuffle, and the squared norm of the Tt row is summed the same way, so every value runs
// in a fixed order that depends on nothing but R and npad.  w == nullptr: every weight is w_def.
template <int DT, int E>
__global__ void __launch_bounds__(256, 2)
    alc_reduce_kernel(KParams kp, const double* __restrict__ Xr, long R, const double* __restrict__ w, double w_def,
                      const double* __restrict__ G, long ldg, const double* __restrict__ Tt, int npad,
                      const double* __restrict__ Xc, long ncols, double s2, double* __restrict__ alc) {
  extern __shared__ __align__(16) double dsm[];   // exp table | sXc[D][BT] | 2 x (sXr[D][GK] | w[GK] | sG[BT][GU_LD])
  const int D = DT > 0 ? DT : kp.D, d = DT > 0 ? DT - E : kp.d;
  double* sXc = dsm + fm::EXP_TBL_DOUBLES;
  double* sSt = sXc + D * BT;
  const int stage = D * GK + GK + BT * GU_LD;
  fm::load_exp_table(dsm, kp.exp_tbl);
  const KEval<DT, E> ke(kp, fm::lane_table(dsm));
  const long c0 = (long)blockIdx.x * BT;
  const int cl = threadIdx.x >> 1, h = threadIdx.x & 1;
  {
    const long left = ncols - c0;
    prefetch_rows<DT>(sXc, Xc + c0 * D, left > BT ? BT : (int)left, D, 0);
  }
  auto prefetch = [&](long s, int buf) {
    double* p = sSt + buf * stage;
    const long r0 = s * GK;
    for (int i = threadIdx.x; i < GK * D; i += blockDim.x) {   // rows r0.. are one contiguous run of Xr
      const int r = i / D, dd = i - r * D;
      const bool ok = r0 + r < R;
      cp_async8_zfill(p + dd * GK + r, ok ? Xr + r0 * D + i : Xr, ok);
    }
    if (threadIdx.x < GK) {
      const bool ok = r0 + (long)threadIdx.x < R;
      if (w) cp_async8_zfill(p + D * GK + threadIdx.x, ok ? w + r0 + threadIdx.x : w, ok);
      else p[D * GK + threadIdx.x] = ok ? w_def : 0.0;
    }
    double* sg = p + D * GK + GK;
    for (int i = threadIdx.x; i < BT * GK; i += blockDim.x) {
      const int r = i / GK, kk = i - r * GK;
      const bool ok = c0 + r < ncols && r0 + kk < R;
      cp_async8_zfill(sg + r * GU_LD + kk, ok ? G + (c0 + r) * ldg + r0 + kk : G, ok);
    }
  };
  const long nst = (R + GK - 1) / GK;
  prefetch(0, 0);
  cp_async_commit();
  // |W k_c|^2 from the candidate's Tt row while the first stage lands: thread h takes the pairs 4m + 2h, 4m + 2h + 1
  double sq = 0.0;
  {
    const long c = c0 + cl < ncols ? c0 + cl : c0;
    const double2* row = reinterpret_cast<const double2*>(Tt + c * (long)npad);
    for (int m = 0; m < npad / 4; m++) {
      const double2 t = row[2 * m + h];
      sq = fma(t.x, t.x, sq);
      sq = fma(t.y, t.y, sq);
    }
  }
  double q[DT > 0 ? DT : 1];
  double acc = 0.0;
  int buf = 0;
  for (long s = 0; s < nst; s++, buf ^= 1) {
    if (s + 1 < nst) prefetch(s + 1, buf ^ 1);
    cp_async_commit();
    cp_async_wait<1>();
    __syncthreads();
    if (DT > 0 && s == 0) {
#pragma unroll
      for (int dd = 0; dd < (DT > 0 ? DT : 1); dd++) q[dd] = sXc[dd * BT + cl];
    }
    const double* sXr = sSt + buf * stage;
    const double* sW = sXr + D * GK;
    const double* sG = sW + GK;
#pragma unroll 2
    for (int m = 0; m < GK / 2; m++) {
      const int k = 2 * m + h;
      double rx = 0.0, rz = 0.0;
      if (DT > 0) {
#pragma unroll
        for (int dd = 0; dd < (DT > 0 ? DT : 1); dd++) {
          const double t = q[dd] - sXr[dd * GK + k];
          if (dd < DT - E) rx = fma(t, t, rx);
          else rz = fma(t, t, rz);
        }
      } else {
        for (int dd = 0; dd < D; dd++) {
          const double t = sXc[dd * BT + cl] - sXr[dd * GK + k];
          if (dd < d) rx = fma(t, t, rx);
          else rz = fma(t, t, rz);
        }
      }
      double kv = ke.k12(rx, rz);
      if (ke.has3) kv += ke.k3(rx);
      const double g = kv - sG[cl * GU_LD + k];
      acc = fma(sW[k] * g, g, acc);
    }
    __syncthreads();   // all readers done with this buffer before the next iteration refills it
  }
  cp_async_wait<0>();
  acc += __shfl_xor_sync(0xffffffffu, acc, 1);
  sq += __shfl_xor_sync(0xffffffffu, sq, 1);
  const long c = c0 + cl;
  if (h != 0 || c >= ncols) return;
  const double den = (kp.kdiag - sq) + s2;
  alc[c] = den > 0.0 ? acc / den : -INFINITY;
}

constexpr size_t alc_smem(int D) { return xgrad_smem(D); }

constexpr size_t asm_smem(int D) { return fm::EXP_TBL_BYTES + (size_t)2 * 2 * D * BT * sizeof(double); }
constexpr size_t grad_smem(int D) { return fm::EXP_TBL_BYTES + (size_t)2 * 2 * (D + 1) * BT * sizeof(double); }

#define MFGP_SHAPES(M)                                                                       \
  M(1, 0) M(2, 0) M(3, 0) M(4, 0) M(5, 0) M(6, 0) M(7, 0) M(8, 0)                            \
  M(2, 1) M(3, 1) M(4, 1) M(5, 1) M(6, 1) M(7, 1) M(8, 1) M(4, 3) M(7, 5)

}  // namespace

int assemble_configure(mfgp_ctx* h) {
  // exp table + double-buffered row panels: 160 KB at the maximum input width (runtime-width kernels)
  const int smem_max = (int)asm_smem(MFGP_MAX_D), gmax = (int)grad_smem(MFGP_MAX_D);
  CUDA_TRY(h, cudaFuncSetAttribute(assemble_kernel<true, 0, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max));
  CUDA_TRY(h, cudaFuncSetAttribute(assemble_kernel<false, 0, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max));
  CUDA_TRY(h, cudaFuncSetAttribute(grad_reduce_kernel<0, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, gmax));
  CUDA_TRY(h, cudaFuncSetAttribute(cross_grad_kernel<0, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   (int)xgrad_smem(MFGP_MAX_D)));
  CUDA_TRY(h, cudaFuncSetAttribute(alc_reduce_kernel<0, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   (int)alc_smem(MFGP_MAX_D)));
#define MFGP_CFG(DT, E)                                                                                   \
  CUDA_TRY(h, cudaFuncSetAttribute(assemble_kernel<true, DT, E>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                   (int)asm_smem(DT)));                                                   \
  CUDA_TRY(h, cudaFuncSetAttribute(grad_reduce_kernel<DT, E>, cudaFuncAttributeMaxDynamicSharedMemorySize,    \
                                   (int)grad_smem(DT)));                                                  \
  CUDA_TRY(h, cudaFuncSetAttribute(cross_tile_kernel<DT, E>, cudaFuncAttributeMaxDynamicSharedMemorySize,     \
                                   (int)cross_smem(DT)));                                                 \
  CUDA_TRY(h, cudaFuncSetAttribute(cross_grad_kernel<DT, E>, cudaFuncAttributeMaxDynamicSharedMemorySize,     \
                                   (int)xgrad_smem(DT)));                                                 \
  CUDA_TRY(h, cudaFuncSetAttribute(alc_reduce_kernel<DT, E>, cudaFuncAttributeMaxDynamicSharedMemorySize,     \
                                   (int)alc_smem(DT)));
  MFGP_SHAPES(MFGP_CFG)
#undef MFGP_CFG
  return 0;
}

int assemble_launch(mfgp_ctx* h, const KParams& kp, const double* X, int N, double diag_add,
                    double* K, long long ldk, int uplo, int npad_identity) {
  const int nrows = npad_identity > 0 ? npad_identity : N;
  const int tiles = (nrows + BT - 1) / BT;
  const int lower = uplo == MFGP_UPLO_LOWER;
  const int ntiles = lower ? tiles * (tiles + 1) / 2 : tiles * tiles;
  const int grid = ntiles < CTAS_PER_SM * MFGP_NUM_SMS ? ntiles : CTAS_PER_SM * MFGP_NUM_SMS;
  const bool vec = (nrows % SBC == 0) && (ldk % 2 == 0) && ((uintptr_t)K % 16 == 0);
  const Shape sh = vec ? shape_of(kp) : Shape{0, 0};
  const size_t smem = asm_smem(kp.D);
  prof_begin(h, PC_ASSEMBLE);
  bool done = false;
#define MFGP_RUN(DT_, E_)                                                                          \
  if (!done && sh.DT == DT_ && sh.E == E_) {                                                       \
    assemble_kernel<true, DT_, E_><<<grid, 256, smem, h->stream>>>(kp, X, N, diag_add, K, ldk, lower, \
                                                                   tiles, nrows, ntiles);          \
    done = true;                                                                                   \
  }
  MFGP_SHAPES(MFGP_RUN)
#undef MFGP_RUN
  if (!done) {
    if (vec)
      assemble_kernel<true, 0, 0><<<grid, 256, smem, h->stream>>>(kp, X, N, diag_add, K, ldk, lower, tiles,
                                                                  nrows, ntiles);
    else
      assemble_kernel<false, 0, 0><<<grid, 256, smem, h->stream>>>(kp, X, N, diag_add, K, ldk, lower, tiles,
                                                                   nrows, ntiles);
  }
  prof_end(h, PC_ASSEMBLE);
  LAUNCH_CHECK(h);
  return 0;
}

int grad_reduce_launch(mfgp_ctx* h, const KParams& kp, const double* X, int N, const double* Kinv,
                       long long ld, const double* alpha, double* d_out8) {
  const int tiles = (N + BT - 1) / BT;
  const int nlin = tiles * (tiles + 1) / 2;
  const int grid = nlin < GR_BLOCKS ? nlin : GR_BLOCKS;
  const Shape sh = shape_of(kp);
  const size_t smem = grad_smem(kp.D);
  prof_begin(h, PC_GRAD);
  bool done = false;
#define MFGP_RUN(DT_, E_)                                                                             \
  if (!done && sh.DT == DT_ && sh.E == E_) {                                                          \
    grad_reduce_kernel<DT_, E_><<<grid, 256, smem, h->stream>>>(kp, X, N, Kinv, ld, alpha, nlin,      \
                                                               h->d_partials);                        \
    done = true;                                                                                      \
  }
  MFGP_SHAPES(MFGP_RUN)
#undef MFGP_RUN
  if (!done) grad_reduce_kernel<0, 0><<<grid, 256, smem, h->stream>>>(kp, X, N, Kinv, ld, alpha, nlin, h->d_partials);
  prof_end(h, PC_GRAD);
  LAUNCH_CHECK(h);
  reduce_partials_kernel<<<1, 192, 0, h->stream>>>(h->d_partials, grid, d_out8);
  LAUNCH_CHECK(h);
  return 0;
}


// Tiled cross-covariance generator for the specialised shapes; returns 1 if it took the launch, 0 if the
// caller should use the one-warp-per-query kernels (small batches, wide or unusual inputs).
int cross_tile_launch(mfgp_ctx* h, const KParams& kp, const double* X, int N, int npad, const double* alpha,
                      const double* Xq, long long ncols, long long cols_pad, double* Ks, double* mean) {
  const Shape sh = shape_of(kp);
  if (sh.DT == 0 || (Ks && cols_pad % BT != 0)) return 0;
  // The two generators produce bit-identical ELEMENTS but reduce the mean in different orders, so which
  // one computes a mean must not depend on the batch size (predictions are bit-invariant to chunking
  // and sharding): with a mean this kernel always runs; small element-only batches take the light one.
  if (!mean && ncols < 16 * BT) return 0;
  // with an output block the pad rows up to cols_pad are zero-filled; mean-only needs the real rows only
  const unsigned grid = (unsigned)(Ks ? cols_pad / BT : (ncols + BT - 1) / BT);
  bool done = false;
#define MFGP_RUN(DT_, E_)                                                                              \
  if (!done && sh.DT == DT_ && sh.E == E_) {                                                           \
    cross_tile_kernel<DT_, E_><<<grid, 256, cross_smem(DT_), h->stream>>>(kp, X, N, npad, alpha, Xq,   \
                                                                         (long)ncols, Ks, mean);       \
    done = true;                                                                                       \
  }
  MFGP_SHAPES(MFGP_RUN)
#undef MFGP_RUN
  return done ? 1 : 0;
}

// K6d launcher: gradients of the queries Xq[0, ncols) (see cross_grad_kernel).  Ut == nullptr: mean mode (dvar and
// quad are not written).  Specialised shapes take one launch; the runtime-width kernel one per GJ gradient columns.
int cross_grad_launch(mfgp_ctx* h, const KParams& kp, const double* X, int N, const double* alpha, const double* Ut,
                      long long ldu, const double* Xq, long long ncols, double* dmean, double* dvar, double* mean,
                      double* quad) {
  if (ncols <= 0) return 0;
  const Shape sh = shape_of(kp);
  const unsigned grid = (unsigned)((ncols + BT - 1) / BT);
  const size_t smem = xgrad_smem(kp.D);
  prof_begin(h, PC_CROSSGEN);
  bool done = false;
#define MFGP_RUN(DT_, E_)                                                                                     \
  if (!done && sh.DT == DT_ && sh.E == E_) {                                                                  \
    cross_grad_kernel<DT_, E_><<<grid, 256, smem, h->stream>>>(kp, X, N, alpha, Ut, (long)ldu, Xq, (long)ncols, 0, \
                                                               dmean, dvar, mean, quad);                      \
    done = true;                                                                                              \
  }
  MFGP_SHAPES(MFGP_RUN)
#undef MFGP_RUN
  if (!done)
    for (int j0 = 0; j0 < kp.D; j0 += GJ)
      cross_grad_kernel<0, 0><<<grid, 256, smem, h->stream>>>(kp, X, N, alpha, Ut, (long)ldu, Xq, (long)ncols, j0,
                                                              dmean, dvar, mean, quad);
  prof_end(h, PC_CROSSGEN);
  LAUNCH_CHECK(h);
  return 0;
}

// K8c launcher: alc of the candidates Xc[0, ncols) (see alc_reduce_kernel), timed as acquisition work (class 9).
int alc_reduce_launch(mfgp_ctx* h, const KParams& kp, const double* Xr, long long R, const double* w, double w_def,
                      const double* G, long long ldg, const double* Tt, int npad, const double* Xc, long long ncols,
                      double s2, double* alc) {
  if (ncols <= 0) return 0;
  const Shape sh = shape_of(kp);
  const unsigned grid = (unsigned)((ncols + BT - 1) / BT);
  const size_t smem = alc_smem(kp.D);
  prof_begin(h, PC_ARGMAX);
  bool done = false;
#define MFGP_RUN(DT_, E_)                                                                                      \
  if (!done && sh.DT == DT_ && sh.E == E_) {                                                                   \
    alc_reduce_kernel<DT_, E_><<<grid, 256, smem, h->stream>>>(kp, Xr, (long)R, w, w_def, G, (long)ldg, Tt, npad, \
                                                               Xc, (long)ncols, s2, alc);                      \
    done = true;                                                                                               \
  }
  MFGP_SHAPES(MFGP_RUN)
#undef MFGP_RUN
  if (!done)
    alc_reduce_kernel<0, 0><<<grid, 256, smem, h->stream>>>(kp, Xr, (long)R, w, w_def, G, (long)ldg, Tt, npad, Xc,
                                                            (long)ncols, s2, alc);
  prof_end(h, PC_ARGMAX);
  LAUNCH_CHECK(h);
  return 0;
}

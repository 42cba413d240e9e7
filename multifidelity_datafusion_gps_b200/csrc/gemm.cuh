// FP64 tensor-pipe GEMM core for sm_100a.
//
// tcgen05/UMMA has no FP64 kind, and every mma.sync f64 shape (m8n8k4, m16n8k4/8/16) lowers to
// DMMA.8x8x4 on sm_100a (checked with cuobjdump), so the FP64 tensor path on B200 is the warp-level
// DMMA.8x8x4 fed from shared memory.  The core is a BMxBNx32 CTA tile with a 3-stage cp.async
// (LDGSTS) pipeline (measured against 16-deep / 4 stages: fewer barriers per flop, deeper prefetch:
// +1.5 % on every GEMM) and conflict-free padded shared-memory layouts; instantiations:
//   Big16 128x128, 16 warps of 32x32 -- throughput shape (1 CTA / SM, 216 KB smem)
//   Small  64x64,  4 warps of 32x32  -- latency shape for the narrow GEMMs on the critical path of the
//                                       recursive factorisation (4x the CTAs, 2 CTAs / SM)
//
//   C[m][n] (+)= alpha * sum_k A(m,k) * B(n,k)
//
// Operand layouts (template flags):
//   A_KC = true : A(m,k) = A[m*lda + k]   (k contiguous)     false: A(m,k) = A[k*lda + m]
//   B_KC = true : B(n,k) = B[n*ldb + k]   (k contiguous)     false: B(n,k) = B[k*ldb + n]
// All extents are multiples of 128 (the factor buffers are padded, see common.cuh), all leading
// dimensions are even and all base pointers 16-byte aligned, so there is no edge handling.
#pragma once
#include <cuda.h>
#include "common.cuh"

namespace dg {

#ifndef MFGP_BK          // tuning overrides (tools/build_variants.sh)
#define MFGP_BK 32
#endif
#ifndef MFGP_STAGES
#define MFGP_STAGES 3
#endif
constexpr int BK = MFGP_BK, STAGES = MFGP_STAGES;
constexpr int KC_STRIDE = BK + 4;   // [rows][BK] tile: row stride 36 doubles (== 4 mod 16 -> no LDS conflicts)

template <int BM_, int BN_, int WGM_, int WGN_>
struct TileCfg {
  static constexpr int BM = BM_, BN = BN_, WGM = WGM_, WGN = WGN_;
  static constexpr int THREADS = 32 * WGM * WGN;
  static constexpr int WTM = BM / WGM, WTN = BN / WGN;   // warp tile
  static constexpr int MT = WTM / 8, NT = WTN / 8;       // 8x8 DMMA tiles per warp
  static constexpr int A_MC_STRIDE = BM + 4;             // [BK][rows] tile: stride == 4 mod 16
  static constexpr int B_MC_STRIDE = BN + 4;
  static constexpr int A_STAGE = (BM * KC_STRIDE > BK * A_MC_STRIDE) ? BM * KC_STRIDE : BK * A_MC_STRIDE;
  static constexpr int B_STAGE = (BN * KC_STRIDE > BK * B_MC_STRIDE) ? BN * KC_STRIDE : BK * B_MC_STRIDE;
  static constexpr int STAGE_DOUBLES = A_STAGE + B_STAGE;
  static constexpr int SMEM_BYTES = STAGES * STAGE_DOUBLES * 8;
};
using Big16 = TileCfg<128, 128, 4, 4>;   // 221184 B smem, 16 warps of 32x32 (4 warps per scheduler)
using Small = TileCfg<64, 64, 2, 2>;     // 110592 B smem
using Row32 = TileCfg<32, 128, 1, 4>;    // 138240 B smem: owns all 128 columns of its 32 rows (in-place TRSM leaf)

__device__ __forceinline__ void cp_async16(double* smem_dst, const double* gsrc) {
  unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gsrc));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;\n" ::"n"(N));
}

__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
               : "+d"(c0), "+d"(c1)
               : "d"(a), "d"(b));
}

// one BK-deep slab of an operand: ROWS x BK doubles = ROWS*BK/2 16-byte chunks
template <bool KC, int ROWS, int THREADS>
__device__ __forceinline__ void load_operand(double* sdst, const double* g, long ld, int r0, int k0,
                                             int tid) {
  constexpr int CPR = BK / 2;                       // chunks per k-contiguous row
  constexpr int PER_THREAD = ROWS * CPR / THREADS;
  static_assert(ROWS * CPR % THREADS == 0, "slab must divide evenly over the threads");
  constexpr int MC_STRIDE = ROWS + 4;
  if (KC) {
#pragma unroll
    for (int i = 0; i < PER_THREAD; i++) {
      int c = tid + i * THREADS;
      int r = c / CPR, kc = c % CPR;
      cp_async16(sdst + r * KC_STRIDE + kc * 2, g + (long)(r0 + r) * ld + k0 + kc * 2);
    }
  } else {
#pragma unroll
    for (int i = 0; i < PER_THREAD; i++) {
      int c = tid + i * THREADS;
      int kr = c / (ROWS / 2), mc = c % (ROWS / 2);
      cp_async16(sdst + kr * MC_STRIDE + mc * 2, g + (long)(k0 + kr) * ld + r0 + mc * 2);
    }
  }
}

// acc[i][j][e]: m-tile i (8 rows each), n-tile j (8 cols each); lane holds row g, cols 2t+e.
template <class T, bool A_KC, bool B_KC>
__device__ __forceinline__ void mainloop(double (&acc)[T::MT][T::NT][2], const double* A, long lda,
                                         const double* B, long ldb, int row0, int col0, int k_begin,
                                         int k_end, double* smem) {
  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  const int g = lane >> 2, t = lane & 3;
  const int wm0 = (warp / T::WGN) * T::WTM, wn0 = (warp % T::WGN) * T::WTN;
  const int nk = (k_end - k_begin) / BK;

#pragma unroll
  for (int s = 0; s < STAGES - 1; s++) {
    if (s < nk) {
      double* sa = smem + s * T::STAGE_DOUBLES;
      load_operand<A_KC, T::BM, T::THREADS>(sa, A, lda, row0, k_begin + s * BK, tid);
      load_operand<B_KC, T::BN, T::THREADS>(sa + T::A_STAGE, B, ldb, col0, k_begin + s * BK, tid);
    }
    cp_async_commit();
  }

  for (int kt = 0; kt < nk; kt++) {
    cp_async_wait<STAGES - 2>();
    __syncthreads();
    const double* sa = smem + (kt % STAGES) * T::STAGE_DOUBLES;
    const double* sb = sa + T::A_STAGE;
#pragma unroll
    for (int kk = 0; kk < BK / 4; kk++) {
      double a[T::MT], b[T::NT];
#pragma unroll
      for (int i = 0; i < T::MT; i++)
        a[i] = A_KC ? sa[(wm0 + 8 * i + g) * KC_STRIDE + kk * 4 + t]
                    : sa[(kk * 4 + t) * T::A_MC_STRIDE + wm0 + 8 * i + g];
#pragma unroll
      for (int j = 0; j < T::NT; j++)
        b[j] = B_KC ? sb[(wn0 + 8 * j + g) * KC_STRIDE + kk * 4 + t]
                    : sb[(kk * 4 + t) * T::B_MC_STRIDE + wn0 + 8 * j + g];
#pragma unroll
      for (int i = 0; i < T::MT; i++)
#pragma unroll
        for (int j = 0; j < T::NT; j++) dmma884(acc[i][j][0], acc[i][j][1], a[i], b[j]);
      if (kk == 0) {
        // refill the stage freed by the previous k tile only now: the first DMMAs are already
        // queued, so the tensor pipe does not drain while the copies are being issued
        int nxt = kt + STAGES - 1;
        if (nxt < nk) {
          double* sn = smem + (nxt % STAGES) * T::STAGE_DOUBLES;
          load_operand<A_KC, T::BM, T::THREADS>(sn, A, lda, row0, k_begin + nxt * BK, tid);
          load_operand<B_KC, T::BN, T::THREADS>(sn + T::A_STAGE, B, ldb, col0, k_begin + nxt * BK, tid);
        }
        cp_async_commit();
      }
    }
  }
  cp_async_wait<0>();
  __syncthreads();
}

struct GemmParams {
  const double* A;
  long lda;
  const double* B;
  long ldb;
  double* C;
  long ldc;
  int M, N, K;                         // extents (multiples of 128)
  double alpha, beta;
  int lower_only;                      // enumerate only tiles with ti >= tj (M == N)
  int kb_row, kb_col, ke_row;          // triangular operands: k >= row0 / k >= col0 / k < row0+BM
  int ke_col;                          //                      k < col0+BN
  // batch of equally shaped, independent products along a diagonal (the nodes of one level of the
  // triangular-inverse recursion): node b works on A + b*stride, B + b*stride, C + b*stride
  int batch;                           // number of nodes (0 or 1: plain product)
  long batch_stride;
};

template <class T, bool A_KC, bool B_KC>
__global__ void __launch_bounds__(T::THREADS) gemm_kernel(GemmParams p) {
  extern __shared__ __align__(16) double smem[];
  int ti, tj;
  int bid = blockIdx.x;
  if (p.batch > 1) {
    const int per_node = gridDim.x / p.batch;
    const long off = (long)(bid / per_node) * p.batch_stride;
    bid %= per_node;
    p.A += off;
    p.B += off;
    p.C += off;
  }
  if (p.lower_only) {
    int tt = bid;
    ti = (int)((sqrt(8.0 * tt + 1.0) - 1.0) * 0.5);
    while ((long)(ti + 1) * (ti + 2) / 2 <= tt) ti++;
    while ((long)ti * (ti + 1) / 2 > tt) ti--;
    tj = tt - ti * (ti + 1) / 2;
  } else {
    const int tiles_n = p.N / T::BN;
    ti = bid / tiles_n;
    tj = bid % tiles_n;
  }
  const int row0 = ti * T::BM, col0 = tj * T::BN;
  int kb = 0, ke = p.K;
  // k-ranges are rounded outwards to BK; the operands hold explicit zeros there
  if (p.kb_row) kb = max(kb, row0);
  if (p.kb_col) kb = max(kb, col0);
  if (p.ke_row) ke = min(ke, row0 + T::BM);
  if (p.ke_col) ke = min(ke, col0 + T::BN);

  double acc[T::MT][T::NT][2];
#pragma unroll
  for (int i = 0; i < T::MT; i++)
#pragma unroll
    for (int j = 0; j < T::NT; j++) acc[i][j][0] = acc[i][j][1] = 0.0;

  if (ke > kb) mainloop<T, A_KC, B_KC>(acc, p.A, p.lda, p.B, p.ldb, row0, col0, kb, ke, smem);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, t = lane & 3;
  const int wm0 = (warp / T::WGN) * T::WTM, wn0 = (warp % T::WGN) * T::WTN;
#pragma unroll
  for (int i = 0; i < T::MT; i++) {
    const long r = row0 + wm0 + 8 * i + g;
#pragma unroll
    for (int j = 0; j < T::NT; j++) {
      double2* ptr = reinterpret_cast<double2*>(p.C + r * p.ldc + col0 + wn0 + 8 * j + 2 * t);
      double2 v;
      v.x = p.alpha * acc[i][j][0];
      v.y = p.alpha * acc[i][j][1];
      if (p.beta != 0.0) {
        double2 o = *ptr;
        v.x += p.beta * o.x;
        v.y += p.beta * o.y;
      }
      *ptr = v;
    }
  }
}

// tmp = W * Ks^T with fused column sum of squares; one CTA owns a 128-column tile of Ks and walks
// all row tiles of the lower-triangular W (k < row0+128), so the reduction order is fixed.
//   out_ss[c] = sum_i ( sum_{k<=i} W[i][k] * Ks[c][k] )^2
template <class T>
__global__ void __launch_bounds__(T::THREADS, 1)
    trmm_sumsq_kernel(const double* W, int npad, const double* Ks, double* out_ss) {
  extern __shared__ __align__(16) double smem[];
  __shared__ double red[T::WGM][T::BN];
  const int col0 = blockIdx.x * T::BN;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, t = lane & 3;
  const int wn0 = (warp % T::WGN) * T::WTN;
  double ss[T::NT][2];
#pragma unroll
  for (int j = 0; j < T::NT; j++) ss[j][0] = ss[j][1] = 0.0;

  // One flattened software pipeline over all (row tile, k tile) pairs: row tile ti needs the k tiles
  // 0 .. 8(ti+1)-1, the loads of the next row tile are already in flight while the current one is
  // finished, and inside the diagonal 128x128 block of W the 8-row DMMA tiles that lie entirely
  // above the diagonal (explicit zeros) are skipped -- adding 0*b is exact, so this changes no bit.
  const int tid = threadIdx.x;
  const int wm0 = (warp / T::WGN) * T::WTM;
  const int nrt = npad / T::BM;
  constexpr int KT_PER_TILE = T::BM / BK;         // 8
  const int total = KT_PER_TILE * nrt * (nrt + 1) / 2;   // sum over ti of KT_PER_TILE (ti + 1) k tiles
  int l_ti = 0, l_kt = 0;                         // loader position
  auto issue_load = [&](int stage) {
    double* sa = smem + stage * T::STAGE_DOUBLES;
    load_operand<true, T::BM, T::THREADS>(sa, W, npad, l_ti * T::BM, l_kt * BK, tid);
    load_operand<true, T::BN, T::THREADS>(sa + T::A_STAGE, Ks, npad, col0, l_kt * BK, tid);
    if (++l_kt == KT_PER_TILE * (l_ti + 1)) { l_kt = 0; ++l_ti; }
  };
#pragma unroll
  for (int s = 0; s < STAGES - 1; s++) {
    if (s < total) issue_load(s);
    cp_async_commit();
  }
  double acc[T::MT][T::NT][2];
#pragma unroll
  for (int i = 0; i < T::MT; i++)
#pragma unroll
    for (int j = 0; j < T::NT; j++) acc[i][j][0] = acc[i][j][1] = 0.0;
  int c_ti = 0, c_kt = 0;                         // consumer position
  for (int f = 0; f < total; f++) {
    cp_async_wait<STAGES - 2>();
    __syncthreads();
    const double* sa = smem + (f % STAGES) * T::STAGE_DOUBLES;
    const double* sb = sa + T::A_STAGE;
    const int krel = c_kt * BK - c_ti * T::BM;    // >= 0 inside the diagonal block
    // Inside the diagonal block only the warps whose rows straddle this k tile see zero structure: warps
    // entirely below it (wm0 >= krel + BK) hold a dense 32-deep slab and take the fully unrolled path,
    // warps entirely above it (wm0 + WTM <= krel) hold explicit zeros and have nothing to add.  Same
    // products in the same order as before: bit-identical sums.
    if (krel < 0 || wm0 >= krel + BK) {           // dense part of the row tile: no zero structure
#pragma unroll
      for (int kk = 0; kk < BK / 4; kk++) {
        double a[T::MT], b[T::NT];
#pragma unroll
        for (int i = 0; i < T::MT; i++) a[i] = sa[(wm0 + 8 * i + g) * KC_STRIDE + kk * 4 + t];
#pragma unroll
        for (int j = 0; j < T::NT; j++) b[j] = sb[(wn0 + 8 * j + g) * KC_STRIDE + kk * 4 + t];
#pragma unroll
        for (int i = 0; i < T::MT; i++)
#pragma unroll
          for (int j = 0; j < T::NT; j++) dmma884(acc[i][j][0], acc[i][j][1], a[i], b[j]);
        if (kk == 0) {                            // refill after the first DMMAs are queued
          if (f + STAGES - 1 < total) issue_load((f + STAGES - 1) % STAGES);
          cp_async_commit();
        }
      }
    } else {
      if (f + STAGES - 1 < total) issue_load((f + STAGES - 1) % STAGES);
      cp_async_commit();
      // Diagonal block.  The skipped tiles must not even be issued (a predicated-off DMMA still
      // occupies the tensor pipe), hence a warp-uniform computed entry into a fall-through chain.
      static_assert(T::MT <= 8, "fall-through chain below covers at most 8 row tiles per warp");
#pragma unroll 1
      for (int kk = 0; kk < (wm0 + T::WTM <= krel ? 0 : BK / 4); kk++) {
        const int imin = max(0, (krel + 4 * kk - wm0) >> 3);
        if (imin >= T::MT) break;                 // later kk only skip more
        double b[T::NT];
#pragma unroll
        for (int j = 0; j < T::NT; j++) b[j] = sb[(wn0 + 8 * j + g) * KC_STRIDE + kk * 4 + t];
#define MFGP_ROWTILE(i)                                                              \
  if constexpr ((i) < T::MT) {                                                       \
    const double a_ = sa[(wm0 + 8 * (i) + g) * KC_STRIDE + kk * 4 + t];              \
    _Pragma("unroll") for (int j = 0; j < T::NT; j++)                                \
        dmma884(acc[(i) < T::MT ? (i) : 0][j][0], acc[(i) < T::MT ? (i) : 0][j][1], a_, b[j]); \
  }
        switch (imin) {
          case 0: MFGP_ROWTILE(0)
          case 1: MFGP_ROWTILE(1)
          case 2: MFGP_ROWTILE(2)
          case 3: MFGP_ROWTILE(3)
          case 4: MFGP_ROWTILE(4)
          case 5: MFGP_ROWTILE(5)
          case 6: MFGP_ROWTILE(6)
          default: MFGP_ROWTILE(7)
        }
#undef MFGP_ROWTILE
      }
    }
    if (++c_kt == KT_PER_TILE * (c_ti + 1)) {     // row tile finished: fold its rows into the sums
#pragma unroll
      for (int i = 0; i < T::MT; i++)
#pragma unroll
        for (int j = 0; j < T::NT; j++) {
          ss[j][0] = fma(acc[i][j][0], acc[i][j][0], ss[j][0]);
          ss[j][1] = fma(acc[i][j][1], acc[i][j][1], ss[j][1]);
          acc[i][j][0] = acc[i][j][1] = 0.0;
        }
      c_kt = 0;
      ++c_ti;
    }
  }
  cp_async_wait<0>();
  // reduce over the 8 row groups g (lanes with equal t), then over the warp rows (fixed order)
#pragma unroll
  for (int j = 0; j < T::NT; j++)
#pragma unroll
    for (int e = 0; e < 2; e++) {
      double v = ss[j][e];
      v += __shfl_xor_sync(0xffffffffu, v, 4);
      v += __shfl_xor_sync(0xffffffffu, v, 8);
      v += __shfl_xor_sync(0xffffffffu, v, 16);
      ss[j][e] = v;
    }
  if (g == 0) {
#pragma unroll
    for (int j = 0; j < T::NT; j++) {
      red[warp / T::WGN][wn0 + 8 * j + 2 * t] = ss[j][0];
      red[warp / T::WGN][wn0 + 8 * j + 2 * t + 1] = ss[j][1];
    }
  }
  __syncthreads();
  if (threadIdx.x < T::BN) {
    double v = red[0][threadIdx.x];
#pragma unroll
    for (int r = 1; r < T::WGM; r++) v += red[r][threadIdx.x];
    out_ss[col0 + threadIdx.x] = v;
  }
}

// ---- TMA + mbarrier variant of trmm_sumsq -----------------------------------------------------------------
// Same tiles, same products in the same order (bit-identical sums), but the operand slabs are fetched by the
// TMA unit (cp.async.bulk.tensor.2d, 128-byte swizzle: conflict-free LDS without padding) and the pipeline
// is synchronised by mbarriers instead of one __syncthreads per k tile: a warp signals "done with stage s"
// (arrive on empty[s]) and moves on; nobody waits for the slowest warp of the CTA unless the ring of stages is
// exhausted.  ncu on the cp.async kernel: barrier stalls are the largest non-pipe stall (2.3 warps per issue
// against 9.4 on the math pipe), the tensor pipe idles 12 % of the time.
// One slab = 32 k values of 128 rows = two boxes of {16 doubles (128 B), 128 rows}; a stage holds four boxes
// (W k-lo, W k-hi, Ks k-lo, Ks k-hi); lane 0 of warps 0..3 issues one box each.
namespace tma {

constexpr int BOXK = 16;                          // doubles per box row: 128 bytes, the swizzle span
constexpr int BOX_BYTES = BOXK * 128 * 8;         // 16 KB
constexpr int STAGE_BYTES = 4 * BOX_BYTES;        // 64 KB
constexpr int NST = 3;
constexpr int SMEM_BYTES = NST * STAGE_BYTES + 1024;   // + slack for the 1024-byte alignment the swizzle needs

__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(unsigned bar, unsigned parity) {
  unsigned ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}\n"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(unsigned bar, unsigned parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}
__device__ __forceinline__ void load_box(unsigned dst, const void* tmap, int c_inner, int c_row, unsigned bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];\n" ::"r"(dst),
      "l"(tmap), "r"(c_inner), "r"(c_row), "r"(bar)
      : "memory");
}

}  // namespace tma

template <class T>
__global__ void __launch_bounds__(T::THREADS, 1)
    trmm_sumsq_tma_kernel(const __grid_constant__ CUtensorMap tmW, const __grid_constant__ CUtensorMap tmK,
                          int npad, double* out_ss) {
  static_assert(T::BM == 128 && T::BN == 128 && BK == 32, "box geometry below assumes 128 x 128 x 32 slabs");
  extern __shared__ unsigned char smem_raw[];
  __shared__ double red[T::WGM][T::BN];
  __shared__ __align__(8) unsigned long long bars[2 * tma::NST];
  const unsigned raw = tma::smem_u32(smem_raw);
  const unsigned base = (raw + 1023u) & ~1023u;
  const unsigned char* sbase = smem_raw + (base - raw);
  const unsigned full0 = tma::smem_u32(&bars[0]), empty0 = tma::smem_u32(&bars[tma::NST]);
  const int col0 = blockIdx.x * T::BN;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int g = lane >> 2, t = lane & 3;
  const int wm0 = (warp / T::WGN) * T::WTM, wn0 = (warp % T::WGN) * T::WTN;
  if (tid == 0) {
    for (int s = 0; s < tma::NST; s++) {
      tma::mbar_init(full0 + 8 * s, 4);                    // four box issuers
      tma::mbar_init(empty0 + 8 * s, T::THREADS / 32);     // every warp releases the stage
    }
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
  }
  __syncthreads();
  double ss[T::NT][2];
#pragma unroll
  for (int j = 0; j < T::NT; j++) ss[j][0] = ss[j][1] = 0.0;
  const int nrt = npad / T::BM;
  constexpr int KT_PER_TILE = T::BM / BK;                  // 4
  const int total = KT_PER_TILE * nrt * (nrt + 1) / 2;
  // swizzled byte offset of (row, k) inside a box: row * 128 + (((k >> 1) ^ (row & 7)) << 4) + (k & 1) * 8;
  // this lane reads rows = g (mod 8) and k = 4 q + t inside the box (q = 0..3)
  unsigned koff[4];
#pragma unroll
  for (int q = 0; q < 4; q++) koff[q] = ((((unsigned)(2 * q + (t >> 1))) ^ (unsigned)g) << 4) + (unsigned)(t & 1) * 8u;
  const unsigned rowA = (unsigned)(wm0 + g) * 128u, rowB = (unsigned)(wn0 + g) * 128u;
  const bool issuer = lane == 0 && warp < 4;
  int l_ti = 0, l_kt = 0;                                  // loader position (kept by all threads, used by issuers)
  auto issue = [&](int fl) {                               // slab fl -> stage fl % NST (issuers only do the work)
    if (issuer) {
      const int st = fl % tma::NST;
      if (fl >= tma::NST) tma::mbar_wait(empty0 + 8 * st, (unsigned)((fl / tma::NST - 1) & 1));
      const unsigned bar = full0 + 8 * st;
      tma::mbar_expect_tx(bar, tma::BOX_BYTES);
      const unsigned dst = base + st * tma::STAGE_BYTES + warp * tma::BOX_BYTES;
      const int kin = l_kt * BK + (warp & 1) * tma::BOXK;
      if (warp < 2) tma::load_box(dst, &tmW, kin, l_ti * T::BM, bar);
      else tma::load_box(dst, &tmK, kin, col0, bar);
    }
    if (++l_kt == KT_PER_TILE * (l_ti + 1)) { l_kt = 0; ++l_ti; }
  };
#pragma unroll
  for (int s = 0; s < tma::NST - 1; s++)
    if (s < total) issue(s);
  double acc[T::MT][T::NT][2];
#pragma unroll
  for (int i = 0; i < T::MT; i++)
#pragma unroll
    for (int j = 0; j < T::NT; j++) acc[i][j][0] = acc[i][j][1] = 0.0;
  int c_ti = 0, c_kt = 0;
  for (int f = 0; f < total; f++) {
    const int st = f % tma::NST;
    tma::mbar_wait(full0 + 8 * st, (unsigned)((f / tma::NST) & 1));
    const unsigned char* sa = sbase + st * tma::STAGE_BYTES;          // W boxes (k-lo, k-hi)
    const unsigned char* sb = sa + 2 * tma::BOX_BYTES;                // Ks boxes
    const int krel = c_kt * BK - c_ti * T::BM;
    if (krel < 0 || wm0 >= krel + BK) {
#pragma unroll
      for (int kk = 0; kk < BK / 4; kk++) {
        const unsigned bo = (unsigned)(kk >> 2) * tma::BOX_BYTES + koff[kk & 3];
        double a[T::MT], b[T::NT];
#pragma unroll
        for (int i = 0; i < T::MT; i++) a[i] = *reinterpret_cast<const double*>(sa + bo + rowA + i * 1024);
#pragma unroll
        for (int j = 0; j < T::NT; j++) b[j] = *reinterpret_cast<const double*>(sb + bo + rowB + j * 1024);
#pragma unroll
        for (int i = 0; i < T::MT; i++)
#pragma unroll
          for (int j = 0; j < T::NT; j++) dmma884(acc[i][j][0], acc[i][j][1], a[i], b[j]);
        if (kk == 0 && f + tma::NST - 1 < total) issue(f + tma::NST - 1);
      }
    } else {
      if (f + tma::NST - 1 < total) issue(f + tma::NST - 1);
      static_assert(T::MT <= 8, "fall-through chain below covers at most 8 row tiles per warp");
#pragma unroll 1
      for (int kk = 0; kk < (wm0 + T::WTM <= krel ? 0 : BK / 4); kk++) {
        const int imin = max(0, (krel + 4 * kk - wm0) >> 3);
        if (imin >= T::MT) break;
        // (runtime kk: the swizzled offset is recomputed instead of indexing koff[], which would spill it)
        const unsigned bo = (unsigned)(kk >> 2) * tma::BOX_BYTES +
                            ((((unsigned)(2 * (kk & 3) + (t >> 1))) ^ (unsigned)g) << 4) + (unsigned)(t & 1) * 8u;
        double b[T::NT];
#pragma unroll
        for (int j = 0; j < T::NT; j++) b[j] = *reinterpret_cast<const double*>(sb + bo + rowB + j * 1024);
#define MFGP_ROWTILE(i)                                                                      \
  if constexpr ((i) < T::MT) {                                                               \
    const double a_ = *reinterpret_cast<const double*>(sa + bo + rowA + (i) * 1024);         \
    _Pragma("unroll") for (int j = 0; j < T::NT; j++)                                        \
        dmma884(acc[(i) < T::MT ? (i) : 0][j][0], acc[(i) < T::MT ? (i) : 0][j][1], a_, b[j]); \
  }
        switch (imin) {
          case 0: MFGP_ROWTILE(0)
          case 1: MFGP_ROWTILE(1)
          case 2: MFGP_ROWTILE(2)
          case 3: MFGP_ROWTILE(3)
          case 4: MFGP_ROWTILE(4)
          case 5: MFGP_ROWTILE(5)
          case 6: MFGP_ROWTILE(6)
          default: MFGP_ROWTILE(7)
        }
#undef MFGP_ROWTILE
      }
    }
    __syncwarp();
    if (lane == 0) tma::mbar_arrive(empty0 + 8 * st);      // this warp is done reading the stage
    if (++c_kt == KT_PER_TILE * (c_ti + 1)) {
#pragma unroll
      for (int i = 0; i < T::MT; i++)
#pragma unroll
        for (int j = 0; j < T::NT; j++) {
          ss[j][0] = fma(acc[i][j][0], acc[i][j][0], ss[j][0]);
          ss[j][1] = fma(acc[i][j][1], acc[i][j][1], ss[j][1]);
          acc[i][j][0] = acc[i][j][1] = 0.0;
        }
      c_kt = 0;
      ++c_ti;
    }
  }
#pragma unroll
  for (int j = 0; j < T::NT; j++)
#pragma unroll
    for (int e = 0; e < 2; e++) {
      double v = ss[j][e];
      v += __shfl_xor_sync(0xffffffffu, v, 4);
      v += __shfl_xor_sync(0xffffffffu, v, 8);
      v += __shfl_xor_sync(0xffffffffu, v, 16);
      ss[j][e] = v;
    }
  if (g == 0) {
#pragma unroll
    for (int j = 0; j < T::NT; j++) {
      red[warp / T::WGN][wn0 + 8 * j + 2 * t] = ss[j][0];
      red[warp / T::WGN][wn0 + 8 * j + 2 * t + 1] = ss[j][1];
    }
  }
  __syncthreads();
  if (threadIdx.x < T::BN) {
    double v = red[0][threadIdx.x];
#pragma unroll
    for (int r = 1; r < T::WGM; r++) v += red[r][threadIdx.x];
    out_ss[col0 + threadIdx.x] = v;
  }
}

// ---- TMA + mbarrier variant of gemm_kernel for k-contiguous operands (NT products) -------------------------
// C[m][n] (+)= alpha * sum_k A[m][k] * B[n][k] with both operands row-major / k contiguous: every GEMM of the
// Cholesky factorisation (SYRK, TRSM updates, look-ahead), the second product of the triangular inverse and
// trmm_store.  Same tiles and accumulation order as gemm_kernel<T, true, true> (bit-identical results); the
// slabs arrive by TMA into 128-byte-swizzled boxes and the stages are handed over by mbarriers (see
// trmm_sumsq_tma_kernel).  The tensor maps describe the operand views starting at p.A / p.B; a batch node b
// adds b * batch_rows to both coordinates.
struct GemmTmaParams {
  double* C;
  long ldc;
  int M, N, K;
  double alpha, beta;
  int lower_only;
  int kb_row, kb_col, ke_row, ke_col;
  int batch;
  long c_batch_stride;     // elements between the C blocks of consecutive nodes
  int a_batch_rows, a_batch_k, b_batch_rows, b_batch_k;   // coordinate shifts per node
  // C -= A B^T (alpha = -1, beta = 1) with the accumulators STARTED at -C: the tile of C is fetched while the
  // first slabs are still in flight, and the epilogue is a plain store (no read-modify-write latency at the
  // end of every tile, where nothing is left to hide it).  Rounds like LAPACK's in-place update.
  int neg_init;
};

template <class T>
__global__ void __launch_bounds__(T::THREADS, 1)
    gemm_tma_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                    GemmTmaParams p) {
  static_assert(T::BM == 128 && T::BN == 128 && BK == 32, "box geometry assumes 128 x 128 x 32 slabs");
  extern __shared__ unsigned char smem_raw[];
  __shared__ __align__(8) unsigned long long bars[2 * tma::NST];
  const unsigned raw = tma::smem_u32(smem_raw);
  const unsigned base = (raw + 1023u) & ~1023u;
  const unsigned char* sbase = smem_raw + (base - raw);
  const unsigned full0 = tma::smem_u32(&bars[0]), empty0 = tma::smem_u32(&bars[tma::NST]);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int g = lane >> 2, t = lane & 3;
  const int wm0 = (warp / T::WGN) * T::WTM, wn0 = (warp % T::WGN) * T::WTN;
  int ti, tj, node = 0;
  int bid = blockIdx.x;
  if (p.batch > 1) {
    const int per_node = gridDim.x / p.batch;
    node = bid / per_node;
    bid %= per_node;
  }
  if (p.lower_only) {
    int tt = bid;
    ti = (int)((sqrt(8.0 * tt + 1.0) - 1.0) * 0.5);
    while ((long)(ti + 1) * (ti + 2) / 2 <= tt) ti++;
    while ((long)ti * (ti + 1) / 2 > tt) ti--;
    tj = tt - ti * (ti + 1) / 2;
  } else {
    const int tiles_n = p.N / T::BN;
    ti = bid / tiles_n;
    tj = bid % tiles_n;
  }
  const int row0 = ti * T::BM, col0 = tj * T::BN;
  int kb = 0, ke = p.K;
  if (p.kb_row) kb = max(kb, row0);
  if (p.kb_col) kb = max(kb, col0);
  if (p.ke_row) ke = min(ke, row0 + T::BM);
  if (p.ke_col) ke = min(ke, col0 + T::BN);
  const int nk = ke > kb ? (ke - kb) / BK : 0;
  if (tid == 0) {
    for (int s = 0; s < tma::NST; s++) {
      tma::mbar_init(full0 + 8 * s, 4);
      tma::mbar_init(empty0 + 8 * s, T::THREADS / 32);
    }
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
  }
  __syncthreads();
  unsigned koff[4];
#pragma unroll
  for (int q = 0; q < 4; q++) koff[q] = ((((unsigned)(2 * q + (t >> 1))) ^ (unsigned)g) << 4) + (unsigned)(t & 1) * 8u;
  const unsigned rowA = (unsigned)(wm0 + g) * 128u, rowB = (unsigned)(wn0 + g) * 128u;
  const bool issuer = lane == 0 && warp < 4;
  const int a_r = row0 + node * p.a_batch_rows, a_k = node * p.a_batch_k;
  const int b_r = col0 + node * p.b_batch_rows, b_k = node * p.b_batch_k;
  auto issue = [&](int fl) {
    if (issuer) {
      const int st = fl % tma::NST;
      if (fl >= tma::NST) tma::mbar_wait(empty0 + 8 * st, (unsigned)((fl / tma::NST - 1) & 1));
      const unsigned bar = full0 + 8 * st;
      tma::mbar_expect_tx(bar, tma::BOX_BYTES);
      const unsigned dst = base + st * tma::STAGE_BYTES + warp * tma::BOX_BYTES;
      const int kin = kb + fl * BK + (warp & 1) * tma::BOXK;
      if (warp < 2) tma::load_box(dst, &tmA, a_k + kin, a_r, bar);
      else tma::load_box(dst, &tmB, b_k + kin, b_r, bar);
    }
  };
#pragma unroll
  for (int s = 0; s < tma::NST - 1; s++)
    if (s < nk) issue(s);
  double acc[T::MT][T::NT][2];
  double* C = p.C + (long)node * p.c_batch_stride;
  if (p.neg_init) {
#pragma unroll
    for (int i = 0; i < T::MT; i++) {
      const long r = row0 + wm0 + 8 * i + g;
#pragma unroll
      for (int j = 0; j < T::NT; j++) {
        const double2 o = *reinterpret_cast<const double2*>(C + r * p.ldc + col0 + wn0 + 8 * j + 2 * t);
        acc[i][j][0] = -o.x;
        acc[i][j][1] = -o.y;
      }
    }
  } else {
#pragma unroll
    for (int i = 0; i < T::MT; i++)
#pragma unroll
      for (int j = 0; j < T::NT; j++) acc[i][j][0] = acc[i][j][1] = 0.0;
  }
  for (int f = 0; f < nk; f++) {
    const int st = f % tma::NST;
    tma::mbar_wait(full0 + 8 * st, (unsigned)((f / tma::NST) & 1));
    const unsigned char* sa = sbase + st * tma::STAGE_BYTES;
    const unsigned char* sb = sa + 2 * tma::BOX_BYTES;
#pragma unroll
    for (int kk = 0; kk < BK / 4; kk++) {
      const unsigned bo = (unsigned)(kk >> 2) * tma::BOX_BYTES + koff[kk & 3];
      double a[T::MT], b[T::NT];
#pragma unroll
      for (int i = 0; i < T::MT; i++) a[i] = *reinterpret_cast<const double*>(sa + bo + rowA + i * 1024);
#pragma unroll
      for (int j = 0; j < T::NT; j++) b[j] = *reinterpret_cast<const double*>(sb + bo + rowB + j * 1024);
#pragma unroll
      for (int i = 0; i < T::MT; i++)
#pragma unroll
        for (int j = 0; j < T::NT; j++) dmma884(acc[i][j][0], acc[i][j][1], a[i], b[j]);
      if (kk == 0 && f + tma::NST - 1 < nk) issue(f + tma::NST - 1);
    }
    __syncwarp();
    if (lane == 0) tma::mbar_arrive(empty0 + 8 * st);
  }
#pragma unroll
  for (int i = 0; i < T::MT; i++) {
    const long r = row0 + wm0 + 8 * i + g;
#pragma unroll
    for (int j = 0; j < T::NT; j++) {
      double2* ptr = reinterpret_cast<double2*>(C + r * p.ldc + col0 + wn0 + 8 * j + 2 * t);
      double2 v;
      v.x = p.alpha * acc[i][j][0];
      v.y = p.alpha * acc[i][j][1];
      if (p.neg_init) {
        v.x = -acc[i][j][0];
        v.y = -acc[i][j][1];
      } else if (p.beta != 0.0) {
        double2 o = *ptr;
        v.x += p.beta * o.x;
        v.y += p.beta * o.y;
      }
      *ptr = v;
    }
  }
}

// ---- TMA GEMM with an m-contiguous operand (TN / TT products: triangular inverse, K^-1 = W^T W) -------------
// An operand stored as X(m,k) = X[k*ld + m] is fetched as eight boxes of {16 m values (128 B), 32 k rows};
// box b holds m = 16 b .. 16 b + 15.  With the 128-byte swizzle, a DMMA step that took the four CONSECUTIVE k
// rows 4 kk .. 4 kk + 3 would put the four t-groups of a warp on the same 64 bytes of banks (4 wavefronts per
// LDS instead of 2), because consecutive rows only permute the low chunk bits.  A step therefore takes the k
// rows {b, b+1, b+4, b+5} with b = 8 (kk / 2) + 2 (kk % 2): rows b+4, b+5 flip chunk bit 2, the 32 lanes
// cover all 32 banks twice -- the minimum for 256 bytes.  Any grouping of the 32 k values of a slab into eight
// steps is a valid DMMA schedule as long as both operands use the same one; a k-contiguous partner operand
// reads the same k sets from its {16 k, 128 rows} boxes (also 2 wavefronts).  The accumulation order over k
// differs from gemm_kernel's, so results agree with it to round-off, not bit for bit.
template <class T, bool A_KC, bool B_KC>
__global__ void __launch_bounds__(T::THREADS, 1)
    gemm_tma_mc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                       GemmTmaParams p) {
  static_assert(T::BM == 128 && T::BN == 128 && BK == 32 && T::THREADS == 512, "16 warps, 128 x 128 x 32 slabs");
  static_assert(!(A_KC && B_KC), "k-contiguous pairs take gemm_tma_kernel");
  constexpr int A_BOXES = A_KC ? 2 : 8, B_BOXES = B_KC ? 2 : 8;
  constexpr int A_BOX_BYTES = A_KC ? tma::BOX_BYTES : 4096, B_BOX_BYTES = B_KC ? tma::BOX_BYTES : 4096;
  constexpr int OPND_BYTES = 2 * tma::BOX_BYTES;          // 32 KB per operand and stage, either layout
  extern __shared__ unsigned char smem_raw[];
  __shared__ __align__(8) unsigned long long bars[2 * tma::NST];
  const unsigned raw = tma::smem_u32(smem_raw);
  const unsigned base = (raw + 1023u) & ~1023u;
  const unsigned char* sbase = smem_raw + (base - raw);
  const unsigned full0 = tma::smem_u32(&bars[0]), empty0 = tma::smem_u32(&bars[tma::NST]);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int g = lane >> 2, t = lane & 3;
  const int wm0 = (warp / T::WGN) * T::WTM, wn0 = (warp % T::WGN) * T::WTN;
  int ti, tj, node = 0;
  int bid = blockIdx.x;
  if (p.batch > 1) {
    const int per_node = gridDim.x / p.batch;
    node = bid / per_node;
    bid %= per_node;
  }
  if (p.lower_only) {
    int tt = bid;
    ti = (int)((sqrt(8.0 * tt + 1.0) - 1.0) * 0.5);
    while ((long)(ti + 1) * (ti + 2) / 2 <= tt) ti++;
    while ((long)ti * (ti + 1) / 2 > tt) ti--;
    tj = tt - ti * (ti + 1) / 2;
  } else {
    const int tiles_n = p.N / T::BN;
    ti = bid / tiles_n;
    tj = bid % tiles_n;
  }
  const int row0 = ti * T::BM, col0 = tj * T::BN;
  int kb = 0, ke = p.K;
  if (p.kb_row) kb = max(kb, row0);
  if (p.kb_col) kb = max(kb, col0);
  if (p.ke_row) ke = min(ke, row0 + T::BM);
  if (p.ke_col) ke = min(ke, col0 + T::BN);
  const int nk = ke > kb ? (ke - kb) / BK : 0;
  if (tid == 0) {
    for (int s = 0; s < tma::NST; s++) {
      tma::mbar_init(full0 + 8 * s, A_BOXES + B_BOXES);
      tma::mbar_init(empty0 + 8 * s, T::THREADS / 32);
    }
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
  }
  __syncthreads();
  // k rows of step kk: k = 8 (kk >> 1) + 2 (kk & 1) + (t & 1) + 4 (t >> 1)
  const int kt = (t & 1) + 4 * (t >> 1);
  // k-contiguous operand: box kk >> 2, row r, chunk ((k & 15) >> 1) ^ (r & 7), half k & 1 = t & 1
  //   (k & 15) >> 1 = 4 ((kk >> 1) & 1) + (kk & 1) + 2 (t >> 1)
  unsigned kcoff[4];
#pragma unroll
  for (int q = 0; q < 4; q++)
    kcoff[q] = ((((unsigned)(4 * (q >> 1) + (q & 1) + 2 * (t >> 1))) ^ (unsigned)g) << 4) + (unsigned)(t & 1) * 8u;
  // m-contiguous operand: box (m >> 4), row k, chunk ((m & 15) >> 1) ^ (k & 7), half m & 1 = g & 1, with
  //   m & 15 = 8 (i & 1) + g  and  k & 7 = 2 (kk & 1) + kt
  unsigned mcoff[2][2];
#pragma unroll
  for (int io = 0; io < 2; io++)
#pragma unroll
    for (int ko = 0; ko < 2; ko++)
      mcoff[io][ko] = ((((unsigned)(4 * io + (g >> 1))) ^ (unsigned)(2 * ko + kt)) << 4) + (unsigned)(g & 1) * 8u +
                      (unsigned)kt * 128u;
  const int a_r = row0 + node * p.a_batch_rows, a_k = node * p.a_batch_k;
  const int b_r = col0 + node * p.b_batch_rows, b_k = node * p.b_batch_k;
  auto issue = [&](int fl) {
    if (lane == 0 && warp < A_BOXES + B_BOXES) {
      const int st = fl % tma::NST;
      if (fl >= tma::NST) tma::mbar_wait(empty0 + 8 * st, (unsigned)((fl / tma::NST - 1) & 1));
      const unsigned bar = full0 + 8 * st;
      const int k0 = kb + fl * BK;
      const unsigned sbase_st = base + st * tma::STAGE_BYTES;
      if (warp < A_BOXES) {
        tma::mbar_expect_tx(bar, A_BOX_BYTES);
        if (A_KC) tma::load_box(sbase_st + warp * A_BOX_BYTES, &tmA, a_k + k0 + warp * tma::BOXK, a_r, bar);
        else tma::load_box(sbase_st + warp * A_BOX_BYTES, &tmA, a_r + warp * 16, a_k + k0, bar);
      } else {
        const int w = warp - A_BOXES;
        tma::mbar_expect_tx(bar, B_BOX_BYTES);
        if (B_KC) tma::load_box(sbase_st + OPND_BYTES + w * B_BOX_BYTES, &tmB, b_k + k0 + w * tma::BOXK, b_r, bar);
        else tma::load_box(sbase_st + OPND_BYTES + w * B_BOX_BYTES, &tmB, b_r + w * 16, b_k + k0, bar);
      }
    }
  };
#pragma unroll
  for (int s = 0; s < tma::NST - 1; s++)
    if (s < nk) issue(s);
  double acc[T::MT][T::NT][2];
#pragma unroll
  for (int i = 0; i < T::MT; i++)
#pragma unroll
    for (int j = 0; j < T::NT; j++) acc[i][j][0] = acc[i][j][1] = 0.0;
  // fixed parts of the fragment addresses
  const unsigned a_fix = A_KC ? (unsigned)(wm0 + g) * 128u : (unsigned)(wm0 >> 4) * 4096u;
  const unsigned b_fix = B_KC ? (unsigned)(wn0 + g) * 128u : (unsigned)(wn0 >> 4) * 4096u;
  for (int f = 0; f < nk; f++) {
    const int st = f % tma::NST;
    tma::mbar_wait(full0 + 8 * st, (unsigned)((f / tma::NST) & 1));
    const unsigned char* sa = sbase + st * tma::STAGE_BYTES;
    const unsigned char* sb = sa + OPND_BYTES;
#pragma unroll
    for (int kk = 0; kk < BK / 4; kk++) {
      double a[T::MT], b[T::NT];
#pragma unroll
      for (int i = 0; i < T::MT; i++) {
        const unsigned off = A_KC ? (unsigned)(kk >> 2) * tma::BOX_BYTES + kcoff[kk & 3] + a_fix + i * 1024u
                                  : a_fix + (unsigned)(i >> 1) * 4096u +
                                        (unsigned)(8 * (kk >> 1) + 2 * (kk & 1)) * 128u + mcoff[i & 1][kk & 1];
        a[i] = *reinterpret_cast<const double*>(sa + off);
      }
#pragma unroll
      for (int j = 0; j < T::NT; j++) {
        const unsigned off = B_KC ? (unsigned)(kk >> 2) * tma::BOX_BYTES + kcoff[kk & 3] + b_fix + j * 1024u
                                  : b_fix + (unsigned)(j >> 1) * 4096u +
                                        (unsigned)(8 * (kk >> 1) + 2 * (kk & 1)) * 128u + mcoff[j & 1][kk & 1];
        b[j] = *reinterpret_cast<const double*>(sb + off);
      }
#pragma unroll
      for (int i = 0; i < T::MT; i++)
#pragma unroll
        for (int j = 0; j < T::NT; j++) dmma884(acc[i][j][0], acc[i][j][1], a[i], b[j]);
      if (kk == 0 && f + tma::NST - 1 < nk) issue(f + tma::NST - 1);
    }
    __syncwarp();
    if (lane == 0) tma::mbar_arrive(empty0 + 8 * st);
  }
  double* C = p.C + (long)node * p.c_batch_stride;
#pragma unroll
  for (int i = 0; i < T::MT; i++) {
    const long r = row0 + wm0 + 8 * i + g;
#pragma unroll
    for (int j = 0; j < T::NT; j++) {
      double2* ptr = reinterpret_cast<double2*>(C + r * p.ldc + col0 + wn0 + 8 * j + 2 * t);
      double2 v;
      v.x = p.alpha * acc[i][j][0];
      v.y = p.alpha * acc[i][j][1];
      if (p.beta != 0.0) {
        double2 o = *ptr;
        v.x += p.beta * o.x;
        v.y += p.beta * o.y;
      }
      *ptr = v;
    }
  }
}

}  // namespace dg

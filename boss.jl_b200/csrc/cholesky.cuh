// cholesky.cuh -- batched blocked FP64 Cholesky, triangular inverse and log-likelihood pieces.
//
// Left-looking block algorithm on 128x128 blocks, S matrices per launch (one grid.y slice each):
//   for j:  UPDATE  A_ij -= L_i,0:j L_j,0:j^T   (i >= j)      gemm core, K = 128 j      [DMMA]
//           POTRF   L_jj = chol(A_jj), Winv_jj = L_jj^-1       potrf128.cuh: 8x8 micro-tiles, DMMA, 2 CTAs / SM
//           TRSM    L_ij  = A_ij Winv_jj^T        (i >  j)      gemm core, K = 128        [DMMA]
// followed, for a posterior fit, by the full triangular inverse W = L^-1 (block recurrence, gemm core)
// and, for the log-likelihood, by a blocked forward substitution.
// Reference: AbstractGPs.posterior / logpdf(::FiniteGP) -> LinearAlgebra.cholesky (LAPACK dpotrf) as
// called from src/models/gaussian_process.jl:199-211 and :269-280.
#pragma once
#include "gemm_core.cuh"
#include "kernel_fn.cuh"
#include "tk_params.cuh"
#include "potrf128.cuh"

namespace boss {

// ---------------------------------------------------------------------------------------------
// K2: fused ARD kernel-matrix construction (lower block triangle, P-layout), per hyper-parameter sample
// ---------------------------------------------------------------------------------------------


// ---------------------------------------------------------------------------------------------
// gemm-core users
// ---------------------------------------------------------------------------------------------
struct CholGemmParams {
  double *L;             // S matrices (P-layout)
  size_t L_stride;
  double *Winv;          // S x nblk diagonal-block inverses, each a 128x128 P-layout block (8 tiles)
  size_t Winv_stride;
  int nblk, ktiles;
  int j;                 // block column (UPDATE / TRSM) or block distance delta (TRTRI)
  double *W, *WT, *TT;   // full inverse, its transpose, per-task scratch (TRTRI), one per matrix of the batch
  size_t W_stride, TT_stride;
  // in-line forward substitution of the batched log-likelihood (null = off): the diagonal-tile SYRK of block
  // column j also forms r_j = sum_{k<j} L_jk w_k from the row block it streams; potrf_tile_kernel turns it into w_j
  const double *fwd_w;   // [S][n_pad] w = L^-1 delta, blocks < j valid
  double *fwd_r;         // [S][n_pad]
  int n_pad;
};

// A_ij -= L_i,0:j * L_j,0:j^T   for i = j + blockIdx.x.  The diagonal tile (i == j) is a SYRK: only its lower
// triangle is computed (syrk_diag_pipeline, 136 of 256 micro-tiles).
__global__ void __launch_bounds__(GEMM_THREADS, 1) chol_update_kernel(CholGemmParams p) {
  const int i = p.j + blockIdx.x;
  double *Lm = p.L + (size_t)blockIdx.y * p.L_stride;
  LinearIt it{Lm + (size_t)i * p.ktiles * TILE_ELEMS, Lm + (size_t)p.j * p.ktiles * TILE_ELEMS, p.j * KT_PER_BLOCK};
  double *dst = Lm + ((size_t)i * p.ktiles + (size_t)p.j * KT_PER_BLOCK) * TILE_ELEMS;
  if (blockIdx.x == 0) {
    auto epi = [&](double(&acc)[17][2], const SyrkCoord &sc) {
      // single round trip: all loads first, then all stores
#pragma unroll
      for (int t = 0; t < 17; ++t)
#pragma unroll
        for (int e = 0; e < 2; ++e) acc[t][e] = dst[block_offset(sc.row(t), sc.col(t, e))] - acc[t][e];
#pragma unroll
      for (int t = 0; t < 17; ++t)
#pragma unroll
        for (int e = 0; e < 2; ++e) dst[block_offset(sc.row(t), sc.col(t, e))] = acc[t][e];
    };
    if (p.fwd_w) {
      // warp w owns micro-rows 2w and 2w+1 of the row block; lane T holds (row T/4, k = T%4 and 4 + T%4) of a
      // micro-tile (the DMMA fragment order), so the partial sums stay per lane until the end
      const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, c4 = lane & 3;
      const double *wv = p.fwd_w + (size_t)blockIdx.y * p.n_pad + c4;
      double r0 = 0.0, r1 = 0.0;
      syrk_diag_pipeline(it, it, epi, [&](const double *st, int g) {
        const double *a = st + (4 * w) * 64 + 2 * lane;
        const double *wk = wv + g * 16;
        const double w0 = wk[0], w1 = wk[4], w2 = wk[8], w3 = wk[12];
        const double2 a00 = lds128(a), a01 = lds128(a + 64), a10 = lds128(a + 128), a11 = lds128(a + 192);
        r0 = fma(a00.x, w0, r0);
        r0 = fma(a00.y, w1, r0);
        r0 = fma(a01.x, w2, r0);
        r0 = fma(a01.y, w3, r0);
        r1 = fma(a10.x, w0, r1);
        r1 = fma(a10.y, w1, r1);
        r1 = fma(a11.x, w2, r1);
        r1 = fma(a11.y, w3, r1);
      });
      r0 += __shfl_xor_sync(0xffffffffu, r0, 1);
      r0 += __shfl_xor_sync(0xffffffffu, r0, 2);
      r1 += __shfl_xor_sync(0xffffffffu, r1, 1);
      r1 += __shfl_xor_sync(0xffffffffu, r1, 2);
      if (c4 == 0) {
        double *rv = p.fwd_r + (size_t)blockIdx.y * p.n_pad + p.j * 128 + 16 * w + (lane >> 2);
        rv[0] = r0;
        rv[8] = r1;
      }
    } else {
      syrk_diag_pipeline(it, it, epi);
    }
  } else {
    gemm_pipeline(it, it, [&](int, double(&acc)[8][4][2], const FragCoord &fc) { rmw_sub_block(dst, acc, fc); });
  }
}

// L_ij = A_ij * Winv_jj^T       for i = j + 1 + blockIdx.x.  Winv_jj is lower triangular: k-micro-steps beyond a
// column slab are skipped (trsm_tri_pipeline).
__global__ void __launch_bounds__(GEMM_THREADS, 1) chol_trsm_kernel(CholGemmParams p) {
  const int i = p.j + 1 + blockIdx.x;
  double *Lm = p.L + (size_t)blockIdx.y * p.L_stride;
  double *blk = Lm + ((size_t)i * p.ktiles + (size_t)p.j * KT_PER_BLOCK) * TILE_ELEMS;
  const double *wi = p.Winv + (size_t)blockIdx.y * p.Winv_stride + (size_t)p.j * (TM * TM);
  LinearIt it{blk, wi, KT_PER_BLOCK};
  trsm_tri_pipeline(it, it, [&](const double(&acc)[16][2][2], const TrsmCoord &tc) {
#pragma unroll
    for (int R = 0; R < 16; ++R)
#pragma unroll
      for (int h = 0; h < 2; ++h)
#pragma unroll
        for (int e = 0; e < 2; ++e) blk[block_offset(tc.row(R), tc.col(h, e))] = acc[R][h][e];
  });
}

// Fused panel step of the left-looking factorisation (block column j >= 1, rows i > j):
//   T    = A_ij - L_i,0:j L_j,0:j^T        phase 1: the common mainloop, accumulators in registers; A_ij itself rides
//                                          through the ring as 8 tail stages (TailIt)
//   L_ij = T Winv_jj^T                     phase 2: T goes to shared memory in P-layout (it is the A operand now),
//                                          Winv_jj's live lower-triangular part is resident in shared memory
// so the tile makes one trip to HBM instead of three and the K = 128 product needs no pipeline fill of its own.
// Shared memory: [0, 160 KB) ring, reused after phase 1 as T (128 KB) + Winv k-tiles 0-1 (30 KB); k-tiles 2-7
// (42 KB live) are prefetched behind the ring while phase 1 runs.
constexpr int PANEL_WHI_OFF = GEMM_SMEM_BYTES;                        // live parts of Winv k-tiles 2..7, packed
constexpr int PANEL_WHI_BYTES = (12 + 10 + 8 + 6 + 4 + 2) * 1024;
constexpr int PANEL_SMEM_BYTES = PANEL_WHI_OFF + PANEL_WHI_BYTES;     // 207 104 B
// byte offset of the live part of k-tile g (rows >= 16 g, i.e. 16 - 2g KB) inside its home region
__host__ __device__ constexpr int panel_w_off(int g) {
  return g == 0 ? 8 * TILE_BYTES : g == 1 ? 9 * TILE_BYTES
       : PANEL_WHI_OFF + (g == 2 ? 0 : g == 3 ? 12 : g == 4 ? 22 : g == 5 ? 30 : g == 6 ? 36 : 40) * 1024;
}

__global__ void __launch_bounds__(GEMM_THREADS, 1) chol_panel_kernel(CholGemmParams p) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  const int i = p.j + 1 + blockIdx.x;
  double *Lm = p.L + (size_t)blockIdx.y * p.L_stride;
  double *dst = Lm + ((size_t)i * p.ktiles + (size_t)p.j * KT_PER_BLOCK) * TILE_ELEMS;
  // the last 8 ring stages carry A_ij itself: the accumulators leave the mainloop as T = A_ij - L_i,0:j L_j,0:j^T
  TailIt it{Lm + (size_t)i * p.ktiles * TILE_ELEMS, Lm + (size_t)p.j * p.ktiles * TILE_ELEMS, dst,
            (p.j + 1) * KT_PER_BLOCK};
  const unsigned char *wi = reinterpret_cast<const unsigned char *>(p.Winv + (size_t)blockIdx.y * p.Winv_stride +
                                                                    (size_t)p.j * (TM * TM));
  uint64_t *wbar = reinterpret_cast<uint64_t *>(smem_raw + GEMM_RING_BYTES + GEMM_SCRATCH_BYTES) + 2 * GEMM_STAGES;
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  if (tid == 32 || tid == 33) {   // not warp 0: it initialises the ring's barriers at the same time
    mbar_init(smem_u32(&wbar[tid - 32]), 1);
    mbar_fence_init();
  }
  // requested after the first ring stages: anything queued ahead of stage 0 delays the first DMMA
  auto prefetch_whi = [&]() {
    if (tid == 0) {
      mbar_arrive_expect_tx(smem_u32(&wbar[0]), PANEL_WHI_BYTES);
#pragma unroll
      for (int g = 2; g < 8; ++g)
        bulk_g2s(smem_u32(smem_raw + panel_w_off(g)), wi + (size_t)g * TILE_BYTES + g * 2048, TILE_BYTES - g * 2048,
                 smem_u32(&wbar[0]));
    }
  };
  gemm_pipeline<true>(it, it, [&](int, double(&acc)[8][4][2], const FragCoord &fc) {
    __syncthreads();   // every warp has consumed its last ring stage
    if (tid == 0) {
      mbar_arrive_expect_tx(smem_u32(&wbar[1]), 2 * TILE_BYTES - 2048);
      bulk_g2s(smem_u32(smem_raw + panel_w_off(0)), wi, TILE_BYTES, smem_u32(&wbar[1]));
      bulk_g2s(smem_u32(smem_raw + panel_w_off(1)), wi + TILE_BYTES + 2048, TILE_BYTES - 2048, smem_u32(&wbar[1]));
    }
    double *Ts = reinterpret_cast<double *>(smem_raw);   // acc = T
#pragma unroll
    for (int fm = 0; fm < 8; ++fm)
#pragma unroll
      for (int fn = 0; fn < 4; ++fn)
        p_store_cfrag(Ts, 8 * fc.wm + fm, 4 * fc.wn + fn, lane, acc[fm][fn][0], acc[fm][fn][1]);
    __syncthreads();
    mbar_wait(smem_u32(&wbar[0]), 0);

    // phase 2: warps tile the output 4 x 2.  Warp w owns row slabs 4 (w & 3) .. + 3 and the eight column slabs of
    // group cg = w >> 2: {4 cg + i} and {15 - 4 cg - i}, i < 4 (68 live k-steps in either group).  A warp then reads
    // a quarter of T and half of Winv instead of all of T (shared-memory traffic 1.1 MB -> 0.5 MB per tile).  The
    // k-tiles are consumed from 7 down to 0: tiles 2-7 have been resident since phase 1, so the two tiles requested
    // a moment ago (0 and 1) arrive while the others are being multiplied.
    const int rg = w & 3, cg = w >> 2;
    double o[4][8][2];
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
      for (int m = 0; m < 8; ++m) o[r][m][0] = o[r][m][1] = 0.0;
#pragma unroll
    for (int g = 7; g >= 0; --g) {
      if (g == 1) mbar_wait(smem_u32(&wbar[1]), 0);
      const double *As = Ts + g * TILE_ELEMS + (8 * rg) * 64 + 2 * lane;
      // virtual base of k-tile g: its live part starts at row 16 g = byte 2048 g of the tile
      const double *Bs = reinterpret_cast<const double *>(smem_raw + panel_w_off(g) - g * 2048) + 2 * lane;
#pragma unroll
      for (int mc = 0; mc < 2; ++mc) {
        const int kk = 2 * g + mc;   // k micro-step 0..15; column slab c is live iff kk <= c
        double2 a[4];
#pragma unroll
        for (int r = 0; r < 4; ++r) a[r] = lds128(As + (r * 2 + mc) * 64);
#pragma unroll
        for (int half = 0; half < 2; ++half) {   // half 0: slabs 4 cg + i (ascending), half 1: 15 - 4 cg - i (descending)
          const int cfirst = half ? 15 - 4 * cg : 4 * cg, cstep = half ? -1 : 1;
          const int cmin = half ? cfirst - 3 : cfirst;
          if (kk <= cmin) {            // all four slabs live: 16 independent accumulator pairs
            double2 bq[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) bq[i] = lds128(Bs + ((cfirst + cstep * i) * 2 + mc) * 64);
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
              for (int r = 0; r < 4; ++r) dmma884(o[r][4 * half + i][0], o[r][4 * half + i][1], a[r].x, bq[i].x);
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
              for (int r = 0; r < 4; ++r) dmma884(o[r][4 * half + i][0], o[r][4 * half + i][1], a[r].y, bq[i].y);
          } else if (kk <= cmin + 3) { // the staircase: some of the four
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const int c = cfirst + cstep * i;
              if (kk <= c) {
                const double2 bb = lds128(Bs + (c * 2 + mc) * 64);
#pragma unroll
                for (int r = 0; r < 4; ++r) dmma884(o[r][4 * half + i][0], o[r][4 * half + i][1], a[r].x, bb.x);
#pragma unroll
                for (int r = 0; r < 4; ++r) dmma884(o[r][4 * half + i][0], o[r][4 * half + i][1], a[r].y, bb.y);
              }
            }
          }
        }
      }
    }
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
      for (int m = 0; m < 8; ++m) {
        const int c = m < 4 ? 4 * cg + m : 15 - 4 * cg - (m - 4);
        p_store_cfrag(dst, 4 * rg + r, c, lane, o[r][m][0], o[r][m][1]);
      }
  }, prefetch_whi);
}

// ---- right-looking variants for small batches (a single posterior fit): every step exposes all tiles of the
// trailing matrix as independent K = 128 products instead of a few CTAs with a long k-range ----
// A_ik -= L_ij L_kj^T for j < k <= i  (after block column j has been solved)
__global__ void __launch_bounds__(GEMM_THREADS, 1) chol_update_rl_kernel(CholGemmParams p) {
  int t = blockIdx.x, ii = 0;
  while (t >= ii + 1) {
    t -= ii + 1;
    ++ii;
  }
  const int i = p.j + 1 + ii, k = p.j + 1 + t;
  double *Lm = p.L + (size_t)blockIdx.y * p.L_stride;
  LinearIt it{Lm + ((size_t)i * p.ktiles + (size_t)p.j * KT_PER_BLOCK) * TILE_ELEMS,
              Lm + ((size_t)k * p.ktiles + (size_t)p.j * KT_PER_BLOCK) * TILE_ELEMS, KT_PER_BLOCK};
  double *dst = Lm + ((size_t)i * p.ktiles + (size_t)k * KT_PER_BLOCK) * TILE_ELEMS;
  if (i == k) {
    syrk_diag_pipeline(it, it, [&](double(&acc)[17][2], const SyrkCoord &sc) {
#pragma unroll
      for (int q = 0; q < 17; ++q)
#pragma unroll
        for (int e = 0; e < 2; ++e) acc[q][e] = dst[block_offset(sc.row(q), sc.col(q, e))] - acc[q][e];
#pragma unroll
      for (int q = 0; q < 17; ++q)
#pragma unroll
        for (int e = 0; e < 2; ++e) dst[block_offset(sc.row(q), sc.col(q, e))] = acc[q][e];
    });
  } else {
    gemm_pipeline(it, it, [&](int, double(&acc)[8][4][2], const FragCoord &fc) { rmw_sub_block(dst, acc, fc); });
  }
}

// Triangular inverse, right-looking step k = p.j:  T_ij^T += W_kj^T L_ik^T for i > k >= j, accumulated in the
// (still unused) block WT(j, i);  blockIdx.x enumerates (i - k - 1, j)
__global__ void __launch_bounds__(GEMM_THREADS, 1) trtri_acc_rl_kernel(CholGemmParams p) {
  const int k = p.j, jb = blockIdx.x % (k + 1), i = k + 1 + blockIdx.x / (k + 1);
  const double *Lm = p.L + (size_t)blockIdx.y * p.L_stride;
  double *WTm = p.WT + (size_t)blockIdx.y * p.W_stride;
  LinearIt it{WTm + ((size_t)jb * p.ktiles + (size_t)k * KT_PER_BLOCK) * TILE_ELEMS,
              Lm + ((size_t)i * p.ktiles + (size_t)k * KT_PER_BLOCK) * TILE_ELEMS, KT_PER_BLOCK};
  double *dst = WTm + ((size_t)jb * p.ktiles + (size_t)i * KT_PER_BLOCK) * TILE_ELEMS;
  gemm_pipeline(it, it, [&](int, double(&acc)[8][4][2], const FragCoord &fc) {
#pragma unroll
    for (int fm = 0; fm < 8; ++fm)
#pragma unroll
      for (int fn = 0; fn < 4; ++fn)
#pragma unroll
        for (int e = 0; e < 2; ++e) acc[fm][fn][e] += dst[block_offset(fc.row(fm), fc.col(fn, e))];
#pragma unroll
    for (int fm = 0; fm < 8; ++fm)
#pragma unroll
      for (int fn = 0; fn < 4; ++fn)
#pragma unroll
        for (int e = 0; e < 2; ++e) dst[block_offset(fc.row(fm), fc.col(fn, e))] = acc[fm][fn][e];
  });
}
//   W_ij = -Winv_ii T_ij for row i = p.j, j = blockIdx.x < i, T_ij^T read from WT(j, i) and overwritten by W_ij^T
__global__ void __launch_bounds__(GEMM_THREADS, 1) trtri_row_rl_kernel(CholGemmParams p) {
  const int i = p.j, jb = blockIdx.x;
  double *WTm = p.WT + (size_t)blockIdx.y * p.W_stride;
  double *dWT = WTm + ((size_t)jb * p.ktiles + (size_t)i * KT_PER_BLOCK) * TILE_ELEMS;
  LinearIt it{p.Winv + (size_t)blockIdx.y * p.Winv_stride + (size_t)i * (TM * TM), dWT, KT_PER_BLOCK};
  double *dW = p.W + (size_t)blockIdx.y * p.W_stride + ((size_t)i * p.ktiles + (size_t)jb * KT_PER_BLOCK) * TILE_ELEMS;
  gemm_pipeline(it, it, [&](int, const double(&acc)[8][4][2], const FragCoord &fc) {
    store_block(dW, false, -1.0, nullptr, acc, fc);
    store_block(dWT, true, -1.0, nullptr, acc, fc);
  });
}

// Fused step of the (left-looking, batched) triangular inverse, block distance delta = p.j, i = blockIdx.x + delta:
//   T_ij = sum_{k=j}^{i-1} L_ik W_kj          phase 1: the common mainloop
//   W_ij = -Winv_ii T_ij                      phase 2: T^T goes to shared memory in P-layout (it is the B operand),
//                                             Winv_ii's live lower triangle is resident (the A operand)
// -> W (normal) and WT (transposed).  Same shared-memory plan as chol_panel_kernel with the operand roles swapped:
// there Winv multiplies from the right (its rows are output columns), here from the left (its rows are output rows).
__global__ void __launch_bounds__(GEMM_THREADS, 1) trtri_fused_kernel(CholGemmParams p) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  const int jb = blockIdx.x, i = jb + p.j;
  const double *Lm = p.L + (size_t)blockIdx.y * p.L_stride;
  const double *WTm = p.WT + (size_t)blockIdx.y * p.W_stride;
  LinearIt it{Lm + ((size_t)i * p.ktiles + (size_t)jb * KT_PER_BLOCK) * TILE_ELEMS,
              WTm + ((size_t)jb * p.ktiles + (size_t)jb * KT_PER_BLOCK) * TILE_ELEMS, p.j * KT_PER_BLOCK};
  double *dW = p.W + (size_t)blockIdx.y * p.W_stride + ((size_t)i * p.ktiles + (size_t)jb * KT_PER_BLOCK) * TILE_ELEMS;
  double *dWT = p.WT + (size_t)blockIdx.y * p.W_stride + ((size_t)jb * p.ktiles + (size_t)i * KT_PER_BLOCK) * TILE_ELEMS;
  const unsigned char *wi = reinterpret_cast<const unsigned char *>(p.Winv + (size_t)blockIdx.y * p.Winv_stride +
                                                                    (size_t)i * (TM * TM));
  uint64_t *wbar = reinterpret_cast<uint64_t *>(smem_raw + GEMM_RING_BYTES + GEMM_SCRATCH_BYTES) + 2 * GEMM_STAGES;
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  if (tid == 32 || tid == 33) {
    mbar_init(smem_u32(&wbar[tid - 32]), 1);
    mbar_fence_init();
  }
  auto prefetch_whi = [&]() {
    if (tid == 0) {
      mbar_arrive_expect_tx(smem_u32(&wbar[0]), PANEL_WHI_BYTES);
#pragma unroll
      for (int g = 2; g < 8; ++g)
        bulk_g2s(smem_u32(smem_raw + panel_w_off(g)), wi + (size_t)g * TILE_BYTES + g * 2048, TILE_BYTES - g * 2048,
                 smem_u32(&wbar[0]));
    }
  };
  gemm_pipeline<true>(it, it, [&](int, double(&acc)[8][4][2], const FragCoord &fc) {
    __syncthreads();   // every warp has consumed its last ring stage
    if (tid == 0) {
      mbar_arrive_expect_tx(smem_u32(&wbar[1]), 2 * TILE_BYTES - 2048);
      bulk_g2s(smem_u32(smem_raw + panel_w_off(0)), wi, TILE_BYTES, smem_u32(&wbar[1]));
      bulk_g2s(smem_u32(smem_raw + panel_w_off(1)), wi + TILE_BYTES + 2048, TILE_BYTES - 2048, smem_u32(&wbar[1]));
    }
    double *Ts = reinterpret_cast<double *>(smem_raw);   // T^T: row = column n of T, col = k
#pragma unroll
    for (int fm = 0; fm < 8; ++fm)
#pragma unroll
      for (int fn = 0; fn < 4; ++fn)
        p_store_cfrag_t(Ts, 8 * fc.wm + fm, 4 * fc.wn + fn, lane, acc[fm][fn][0], acc[fm][fn][1]);
    __syncthreads();
    mbar_wait(smem_u32(&wbar[0]), 0);

    // phase 2: warp w owns column slabs 4 (w & 3) .. + 3 of the output and the eight ROW slabs of group rg = w >> 2:
    // {4 rg + i} and {15 - 4 rg - i}, i < 4; row slab R of Winv_ii is live for k micro-steps kk <= R.
    const int cgp = w & 3, rg = w >> 2;
    double o[8][4][2];
#pragma unroll
    for (int m = 0; m < 8; ++m)
#pragma unroll
      for (int c = 0; c < 4; ++c) o[m][c][0] = o[m][c][1] = 0.0;
#pragma unroll
    for (int g = 7; g >= 0; --g) {
      if (g == 1) mbar_wait(smem_u32(&wbar[1]), 0);
      const double *Bs = Ts + g * TILE_ELEMS + (8 * cgp) * 64 + 2 * lane;
      const double *As = reinterpret_cast<const double *>(smem_raw + panel_w_off(g) - g * 2048) + 2 * lane;
#pragma unroll
      for (int mc = 0; mc < 2; ++mc) {
        const int kk = 2 * g + mc;
        double2 b[4];
#pragma unroll
        for (int c = 0; c < 4; ++c) b[c] = lds128(Bs + (c * 2 + mc) * 64);
#pragma unroll
        for (int half = 0; half < 2; ++half) {
          const int rfirst = half ? 15 - 4 * rg : 4 * rg, rstep = half ? -1 : 1;
          const int rmin = half ? rfirst - 3 : rfirst;
          if (kk <= rmin) {
            double2 aq[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) aq[q] = lds128(As + ((rfirst + rstep * q) * 2 + mc) * 64);
#pragma unroll
            for (int q = 0; q < 4; ++q)
#pragma unroll
              for (int c = 0; c < 4; ++c) dmma884(o[4 * half + q][c][0], o[4 * half + q][c][1], aq[q].x, b[c].x);
#pragma unroll
            for (int q = 0; q < 4; ++q)
#pragma unroll
              for (int c = 0; c < 4; ++c) dmma884(o[4 * half + q][c][0], o[4 * half + q][c][1], aq[q].y, b[c].y);
          } else if (kk <= rmin + 3) {
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              const int R = rfirst + rstep * q;
              if (kk <= R) {
                const double2 aa = lds128(As + (R * 2 + mc) * 64);
#pragma unroll
                for (int c = 0; c < 4; ++c) dmma884(o[4 * half + q][c][0], o[4 * half + q][c][1], aa.x, b[c].x);
#pragma unroll
                for (int c = 0; c < 4; ++c) dmma884(o[4 * half + q][c][0], o[4 * half + q][c][1], aa.y, b[c].y);
              }
            }
          }
        }
      }
    }
#pragma unroll
    for (int m = 0; m < 8; ++m) {
      const int R = m < 4 ? 4 * rg + m : 15 - 4 * rg - (m - 4);
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        p_store_cfrag(dW, R, 4 * cgp + c, lane, -o[m][c][0], -o[m][c][1]);
        p_store_cfrag_t(dWT, R, 4 * cgp + c, lane, -o[m][c][0], -o[m][c][1]);
      }
    }
  }, prefetch_whi);
}

// Generic C = A B^T on P-layout operands: grid (N/128, M/128).  Used by boss_gp_cov (V^T V, lower tiles only) and by
// the test hook boss_dbg_gemm_nt.
struct GemmNtParams {
  const double *A, *B;
  double *C;
  int ktilesAB;  // K/16
  int ktilesC;   // N/16
  int lower_only;  // skip tiles above the block diagonal (symmetric products: boss_gp_cov)
};
__global__ void __launch_bounds__(GEMM_THREADS, 1) gemm_nt_kernel(GemmNtParams p) {
  const int cb = blockIdx.x, rb = blockIdx.y;
  if (p.lower_only && cb > rb) return;
  LinearIt it{p.A + (size_t)rb * p.ktilesAB * TILE_ELEMS, p.B + (size_t)cb * p.ktilesAB * TILE_ELEMS, p.ktilesAB};
  double *dst = p.C + ((size_t)rb * p.ktilesC + (size_t)cb * KT_PER_BLOCK) * TILE_ELEMS;
  gemm_pipeline(it, it, [&](int, const double(&acc)[8][4][2], const FragCoord &fc) {
    store_block(dst, false, 1.0, nullptr, acc, fc);
  });
}

// ---------------------------------------------------------------------------------------------
// y = M x for a P-layout n_pad x n_pad matrix (one warp per 8-row micro-row).  Used for
// w = W delta and alpha = W^T w in the posterior fit.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) matvec_p_kernel(const double *__restrict__ Mx, const double *__restrict__ x,
                                                       double *__restrict__ y, int ktiles, size_t m_stride = 0,
                                                       size_t x_stride = 0, size_t y_stride = 0) {
  Mx += (size_t)blockIdx.y * m_stride;   // blockIdx.y = matrix of the batch
  x += (size_t)blockIdx.y * x_stride;
  y += (size_t)blockIdx.y * y_stride;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int mrow = blockIdx.x * 8 + warp;      // global micro-row
  const int rb = mrow >> 4, mr = mrow & 15;
  const int c4 = lane & 3;
  const double *base = Mx + (size_t)rb * ktiles * TILE_ELEMS + (mr * 2) * 64 + lane * 2;
  double acc = 0.0;
  for (int kt = 0; kt < ktiles; ++kt) {
#pragma unroll
    for (int mc = 0; mc < 2; ++mc) {
      const double2 v = *reinterpret_cast<const double2 *>(base + (size_t)kt * TILE_ELEMS + mc * 64);
      const int k = kt * 16 + mc * 8 + c4;
      acc = fma(v.x, x[k], acc);
      acc = fma(v.y, x[k + 4], acc);
    }
  }
  acc += __shfl_xor_sync(0xffffffffu, acc, 1);
  acc += __shfl_xor_sync(0xffffffffu, acc, 2);
  if (c4 == 0) y[mrow * 8 + (lane >> 2)] = acc;
}

// ---------------------------------------------------------------------------------------------
// Log-likelihood assembly.  The forward substitution  w_i = Winv_ii (delta_i - sum_{k<i} L_ik w_k)  runs inside the
// factorisation (fwd_* fields of CholGemmParams / PotrfParams), so no kernel re-reads L:
//   ll = -(n log 2pi + 2 sum log L_kk + |w|^2)/2
// (AbstractGPs logpdf(::FiniteGP, y), reference call site src/models/gaussian_process.jl:278-279)
// ---------------------------------------------------------------------------------------------
__global__ void loglik_finish_kernel(const double *logdet_blk, const double *ssq_blk, const int *status, int nblk, int n,
                                     int S, double *loglik) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= S) return;
  double ld = 0.0, mahal = 0.0;
  for (int b = 0; b < nblk; ++b) ld += logdet_blk[(size_t)s * nblk + b];
  for (int b = 0; b < nblk; ++b) mahal += ssq_blk[(size_t)s * nblk + b];
  double ll = -((double)n * 1.8378770664093453 + 2.0 * ld + mahal) * 0.5;
  const int st = status[s];
  if (st == 1) ll = -INFINITY;
  if (st < 0) ll = NAN;
  loglik[s] = ll;
}

// ---------------------------------------------------------------------------------------------
// Hyper-parameter gradient of the log marginal likelihood (SURVEY.md 8f rank 2):
//   d LML / d theta = 1/2 sum_ij G_ij dK_ij/dtheta,   G = alpha alpha^T - K^-1,  K^-1 = W^T W
// (what ForwardDiff yields through logpdf(::FiniteGP), src/model_fitters/optimization.jl:41,153)
// ---------------------------------------------------------------------------------------------
// zero-padded copy of delta = y - m(X): dst[s][n_pad]
__global__ void pad_delta_kernel(const double *ymm, long long ldy, int n, int n_pad, double *dst) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_pad) return;
  dst[(size_t)blockIdx.y * n_pad + i] = (i < n) ? ymm[(size_t)blockIdx.y * ldy + i] : 0.0;
}

// K^-1 lower block triangle: Kinv_ij = sum_{k >= i} WT_ik WT_jk^T  (i >= j), written over the factor's storage.
struct KinvParams {
  const double *WT;
  size_t W_stride;
  double *Kinv;
  size_t K_stride;
  int nblk, ktiles;
};
__global__ void __launch_bounds__(GEMM_THREADS, 1) kinv_wtw_kernel(KinvParams p) {
  int t = blockIdx.x, i = 0;
  while (t >= i + 1) {
    t -= i + 1;
    ++i;
  }
  const int j = t;
  // longest k-ranges first would balance better; the grid is large (S x tiles) so dynamic scheduling suffices
  const double *WTm = p.WT + (size_t)blockIdx.y * p.W_stride;
  LinearIt it{WTm + ((size_t)i * p.ktiles + (size_t)i * KT_PER_BLOCK) * TILE_ELEMS,
              WTm + ((size_t)j * p.ktiles + (size_t)i * KT_PER_BLOCK) * TILE_ELEMS, (p.nblk - i) * KT_PER_BLOCK};
  double *dst = p.Kinv + (size_t)blockIdx.y * p.K_stride + ((size_t)i * p.ktiles + (size_t)j * KT_PER_BLOCK) * TILE_ELEMS;
  gemm_pipeline(it, it, [&](int, const double(&acc)[8][4][2], const FragCoord &fc) {
    store_block(dst, false, 1.0, nullptr, acc, fc);
  });
}

// Per (lower tile, sample): partial sums  A1 = sum_{i>j} G_ij kappa_ij,  A2 = sum_i G_ii,  B_q = sum_{i>j} G_ij g_ij dq_ij^2
// with g = kappa'(r)/r and dq the scaled coordinate difference.  part[s][tile][DP + 2].


// grad[s][0..d-1] = -(a^2 / l_q) sum_t B_q ;  grad[s][d] = a (2 sum A1 + sum A2) ;  grad[s][d+1] = s sum A2
__global__ void loglik_grad_final_kernel(const double *part, int ntiles, int DP, int d, const double *ls, const double *amp,
                                         const double *noise, const int *status, double *grad, long long S) {
  const long long s = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (s >= S) return;
  const double a = amp[s] + MIN_PARAM_VALUE, sn = noise[s] + MIN_PARAM_VALUE;
  double a1 = 0.0, a2 = 0.0;
  const double *ps = part + (size_t)s * ntiles * (DP + 2);
  const bool ok = status[s] == 0;
  for (int t = 0; t < ntiles; ++t) {
    a1 += ps[(size_t)t * (DP + 2) + DP];
    a2 += ps[(size_t)t * (DP + 2) + DP + 1];
  }
  for (int q = 0; q < d; ++q) {
    double b = 0.0;
    for (int t = 0; t < ntiles; ++t) b += ps[(size_t)t * (DP + 2) + q];
    grad[(size_t)s * (d + 2) + q] = ok ? -(a * a) * b / (ls[(size_t)s * d + q] + MIN_PARAM_VALUE) : 0.0;
  }
  grad[(size_t)s * (d + 2) + d] = ok ? a * (2.0 * a1 + a2) : 0.0;
  grad[(size_t)s * (d + 2) + d + 1] = ok ? sn * a2 : 0.0;
}

// Gradient w.r.t. the parameters of the prior mean (DESIGN.md 2.13):  d LML / d theta_c = alpha^T J[:, c],  J = dm/dtheta
// at the training inputs, n x k column-major per sample (sample s at J + s*ldj; ldj == 0: shared).  Grid (k, S).  Thread t
// sums alpha_i J_ic over i = t, t + 128, ... < n in ascending i, then a fixed-order tree finishes: the result depends on
// the sample's alpha and J alone, never on the batch, window, stream group or device it was evaluated in.
__global__ void __launch_bounds__(128) loglik_mean_grad_kernel(const double *__restrict__ alpha, int n_pad,
                                                               const double *__restrict__ J, long long ldj, int n, int k,
                                                               const int *__restrict__ status, double *__restrict__ grad_mean) {
  __shared__ double red[128];
  const int c = blockIdx.x, s = blockIdx.y, t = threadIdx.x;
  const double *a = alpha + (size_t)s * n_pad;
  const double *Jc = J + (size_t)s * ldj + (size_t)c * n;
  double acc = 0.0;
  for (int i = t; i < n; i += 128) acc = fma(a[i], Jc[i], acc);
  red[t] = acc;
  __syncthreads();
#pragma unroll
  for (int w = 64; w > 0; w >>= 1) {
    if (t < w) red[t] += red[t + w];
    __syncthreads();
  }
  if (t == 0) grad_mean[(size_t)s * k + c] = status[s] == 0 ? red[0] : 0.0;   // not PD: alpha is garbage, the gradient 0
}

}  // namespace boss

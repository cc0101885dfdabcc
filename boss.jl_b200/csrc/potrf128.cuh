// potrf128.cuh -- Cholesky factor AND triangular inverse of one 128x128 diagonal block per CTA, on 8x8
// micro-tiles with FP64 tensor-core (DMMA.8x8x4) updates.
//
// This is the latency-critical step of the blocked factorisation (cholesky.cuh): every block column waits
// for it, and for batches of small matrices (BASELINE config C3: n = 512 -> 4 blocks per matrix) it is most
// of the run time.  Layout: the lower block triangle lives in shared memory as 136 packed 8x8 micro-tiles in
// the DMMA fragment order of the P-layout (common.cuh), 68 KB, so two CTAs share an SM and hide each other's
// dependency stalls.
//
//   factorisation  over the 16 tile columns s, with one column of look-ahead:
//                    finish   C_Is -= L_I,s-1 L_s,s-1^T                  DMMA, all warps (one k-step: short)
//                    potf2    8x8 diagonal tile, redundantly in the registers of every thread of warps 0-3
//                    trsm     rows of the panel below by forward substitution, one row per thread (warps 0-3)
//                    ahead    C_I,s+1 -= sum_{t<s} L_It L_s+1,t^T         DMMA, warps 4-7, while warps 0-3 are in
//                                                                        the latency-bound potf2 / trsm chain
//   inverse        8x8 diagonal inverses (one column per thread), then recursive doubling
//                    W21 = -W22 (L21 W11)   for block sizes 8, 16, 32, 64                DMMA
//
// Reference: LinearAlgebra.cholesky -> LAPACK dpotrf as called through AbstractGPs.posterior / logpdf
// (src/models/gaussian_process.jl:199-211, :269-280).
#pragma once
#include "common.cuh"
#include "kernel_fn.cuh"

namespace boss {

struct PotrfParams {
  double *L;
  size_t L_stride;
  double *Winv;
  size_t Winv_stride;
  int nblk, ktiles, j;
  double *logdet_blk;  // S x nblk : sum_k log L_kk of this block
  int *status;         // S : BOSS_NOT_POSDEF on a non-positive / NaN pivot
  double *W, *WT;      // optional: also deposit Winv_jj into W(j,j), its transpose into WT(j,j)
  size_t W_stride;     // per matrix of the batch
  // in-line forward substitution of the batched log-likelihood (fwd_w null = off):
  //   w_j = Winv_jj (delta_j - r_j),  r_j = sum_{k<j} L_jk w_k from the diagonal-tile SYRK (chol_update_kernel)
  const double *fwd_ymm;   // delta = y - m(X): shared (fwd_ldy = 0) or one column per matrix
  long long fwd_ldy;
  int fwd_n, n_pad;
  const double *fwd_r;     // [S][n_pad]
  double *fwd_w;           // [S][n_pad]
  double *fwd_ssq;         // [S][nblk]  |w_j|^2
  // fused diagonal step (potrf_fused_kernel, the left-looking batch paths): the CTA forms its own input tile
  //   A_jj = K_jj - sum_{k<j} L_jk L_jk^T
  // K_jj from the hyper-parameters (what build_k_kernel would have written), the SYRK from row block j of L, and
  // r_j = sum_{k<j} L_jk w_k of the forward substitution from the same stream of tiles; nothing of it touches HBM.
  const double *gen_X;     // d x n raw training inputs
  int gen_d, gen_dp, gen_n, gen_kid;
  const double *gen_ls, *gen_amp, *gen_noise;   // per-matrix raw hyper-parameters
  unsigned long long gen_disc;
  double gen_rq_a;         // RationalQuadratic shape parameter (gen_kid 4)
  int store_L;             // also write L_jj back to global (batched posterior fit: L is part of the handle)
};

constexpr int PT_TILES = 136;                        // 16*17/2 lower micro-tiles
constexpr int PT_TMP_ELEMS = 64 * 64;                // scratch for the inverse products (one 64x64 block)
constexpr int PT_SMEM_BYTES = (PT_TILES * 64 + PT_TMP_ELEMS + 128 + 128 + 8 + 128 + 8) * 8;   // 105 600 B -> 2 CTAs / SM
// the fused kernel adds: 12 mbarrier slots, the exp table (32), 1/l (32), per-row forward-substitution sums (128)
constexpr int PF_RING_STAGES = 6;                    // 6 x 16 KB single-tile stages live in the (not yet used) T | tmp area
constexpr int PF_BAR_SLOTS = 2 * PF_RING_STAGES;     // mbarrier slots of the SYRK ring: full[6], empty[6]
constexpr int PF_EXTRA_ELEMS = PF_BAR_SLOTS + EXPTAB_N + 32 + 128;
constexpr int PF_SMEM_BYTES = PT_SMEM_BYTES + PF_EXTRA_ELEMS * 8;   // 107 168 B -> still 2 CTAs / SM

// (I, J) of the t-th packed lower micro-tile
struct PtIJ {
  unsigned char I[PT_TILES], J[PT_TILES];
};
__host__ __device__ constexpr PtIJ pt_make_ij() {
  PtIJ r{};
  int t = 0;
  for (int I = 0; I < 16; ++I)
    for (int J = 0; J <= I; ++J) {
      r.I[t] = (unsigned char)I;
      r.J[t] = (unsigned char)J;
      ++t;
    }
  return r;
}
__constant__ PtIJ PT_IJ = pt_make_ij();

// packed lower-triangular micro-tile (I >= J)
__device__ __forceinline__ int pt_tile(int I, int J) { return ((I * (I + 1)) / 2 + J) * 64; }
// offset of element (r, c) inside a micro-tile (DMMA fragment order, see common.cuh)
__device__ __forceinline__ int pt_elem(int r, int c) { return (((r << 2) + (c & 3)) << 1) + (c >> 2); }
// offset of micro-tile (I, J) inside a 128x128 P-layout block (8 macro-tiles of 128 x 16)
__device__ __forceinline__ int pt_gtile(int I, int J) { return (J >> 1) * TILE_ELEMS + (((I << 1) + (J & 1)) << 6); }

// B operand of an "NN" product (B[k][n] = Q[k][n]): transposed fragment load of a stored tile
__device__ __forceinline__ double2 pt_ldT(const double *tile, int lane) {
  const int o = ((lane & 3) << 3) + (((lane >> 2) & 3) << 1) + (lane >> 4);
  return make_double2(tile[o], tile[o + 32]);
}

// C-fragment (lane holds (r = lane/4, c = 2(lane%4) + e)) <-> storage offsets
__device__ __forceinline__ int pt_cpos(int lane, int e) {
  const int r = lane >> 2, q = lane & 3;
  return (r << 3) + ((q & 1) << 2) + (e << 1) + (q >> 1);
}

// K values of the thread's 17 live micro-tiles of the diagonal block (accumulator fragment positions), minus the SYRK
// accumulators, into the packed tile store.  Same arithmetic as build_k_kernel followed by chol_update_kernel's
// `A - acc`, so the fused path reproduces the unfused one bit for bit.
// On entry the tile store holds the SYRK accumulators at the same positions (the loop over the tiles is not unrolled,
// and a dynamically indexed accumulator array would be demoted to local memory for the whole kernel).
template <int KID>
__device__ __forceinline__ void pf_generate_tile(double *T, const double *xs, int dp, int warp, int lane, int row0, int n,
                                                 double a2, double s2, const double *etab, double rq_a) {
#pragma unroll 1
  for (int t = 0; t < 17; ++t) {
    const int R = t < 16 - warp ? warp + t : t - 1, Cs = t < 16 - warp ? warp : 15 - warp;
    const int r = 8 * R + (lane >> 2), c0 = 8 * Cs + 2 * (lane & 3);
    const double *xr = xs + r * dp, *xc = xs + c0 * dp;
    double d20 = 0.0, d21 = 0.0;
    for (int i = 0; i < dp; ++i) {
      const double x = xr[i], df0 = x - xc[i], df1 = x - xc[dp + i];
      d20 = fma(df0, df0, d20);
      d21 = fma(df1, df1, d21);
    }
    double v0 = a2 * kappa_fast<KID>(d20, etab, rq_a), v1 = a2 * kappa_fast<KID>(d21, etab, rq_a);
    const int gi = row0 + r, gj = row0 + c0;
    if (gi < n && gj < n) {
      if (gi == gj) v0 += s2;
    } else {
      v0 = (gi == gj) ? 1.0 : 0.0;   // identity padding: L_pad = I, log-det contribution 0
    }
    if (gi < n && gj + 1 < n) {
      if (gi == gj + 1) v1 += s2;
    } else {
      v1 = (gi == gj + 1) ? 1.0 : 0.0;
    }
    double *dst = T + ((R * (R + 1)) / 2 + Cs) * 64;
    dst[pt_cpos(lane, 0)] = v0 - dst[pt_cpos(lane, 0)];
    dst[pt_cpos(lane, 1)] = v1 - dst[pt_cpos(lane, 1)];
  }
}

// live micro-tiles T0 .. T1-1 of the warp, one k micro-step (8 wide): fragments, then both halves of the DMMAs
template <int T0, int T1>
__device__ __forceinline__ void pf_syrk_batch(double (&acc)[17][2], const double *st, int warp, int n0, double2 b0, double2 b1) {
  double2 a[T1 - T0];
#pragma unroll
  for (int t = T0; t < T1; ++t) a[t - T0] = lds128(st + (t < n0 ? warp + t : t - 1) * 128);
#pragma unroll
  for (int t = T0; t < T1; ++t) dmma884(acc[t][0], acc[t][1], a[t - T0].x, t < n0 ? b0.x : b1.x);
#pragma unroll
  for (int t = T0; t < T1; ++t) dmma884(acc[t][0], acc[t][1], a[t - T0].y, t < n0 ? b0.y : b1.y);
}

// FUSED = false: the diagonal tile is read from global memory (posterior fit, right-looking steps).
// FUSED = true : the CTA generates K_jj, subtracts the SYRK of row block j of L (streamed through a 6-stage TMA ring
//                that lives in the tile store before it is needed) and carries the forward substitution's r_j.
// s_mat: matrix of the batch; jc: block column (p.j for the stand-alone kernels).
template <bool FUSED>
__device__ __forceinline__ void potrf_tile_body(const PotrfParams &p, const int s_mat, const int jc) {
  extern __shared__ __align__(16) double sm[];
  double *T = sm;                          // [136][64] packed lower tiles: A -> L -> W
  double *tmp = sm + PT_TILES * 64;        // [64][64] as 8x8 tiles (row-major tile grid, 8 tiles per row)
  double *dinv = tmp + PT_TMP_ELEMS;       // [128] 1 / L_kk
  double *lg = dinv + 128;                 // [128] log L_kk
  int *flag = reinterpret_cast<int *>(lg + 128);
  double *fv = lg + 128 + 8;               // [128] delta_j - r_j, then [8] warp partials of |w_j|^2
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  double *blk = p.L + (size_t)s_mat * p.L_stride + ((size_t)jc * p.ktiles + (size_t)jc * KT_PER_BLOCK) * TILE_ELEMS;

  if (tid == 0) *flag = 0;
  if constexpr (!FUSED) {
    // ---- load the lower block triangle: 136 micro-tiles of 512 B, one per warp pass (coalesced 16 B per lane;
    //      all 17 loads of a thread are in flight together) ----
    double2 buf[PT_TILES / 8];
#pragma unroll
    for (int k = 0; k < PT_TILES / 8; ++k) {
      const int t = warp + 8 * k;
      buf[k] = *reinterpret_cast<const double2 *>(blk + pt_gtile(PT_IJ.I[t], PT_IJ.J[t]) + 2 * lane);
    }
#pragma unroll
    for (int k = 0; k < PT_TILES / 8; ++k) *reinterpret_cast<double2 *>(T + (warp + 8 * k) * 64 + 2 * lane) = buf[k];
  } else {
    uint64_t *bars = reinterpret_cast<uint64_t *>(fv + 136);          // full[6], empty[6]
    double *etab = fv + 136 + PF_BAR_SLOTS;
    double *invl = etab + EXPTAB_N;
    double *rsum = invl + 32;                                         // [128] r_j = sum_{k<j} L_jk w_k
    exptab_init(etab);
    if (tid >= 32 && tid < 64) {
      const int i = tid - 32;
      double l = (i < p.gen_d) ? p.gen_ls[(size_t)s_mat * p.gen_d + i] : 1.0;
      if (i < p.gen_d && !(l >= 0.0)) p.status[s_mat] = -1;
      invl[i] = (i < p.gen_d) ? 1.0 / (l + MIN_PARAM_VALUE) : 0.0;
    }
    const double a_raw = p.gen_amp[s_mat], s_raw = p.gen_noise[s_mat];
    if (tid == 64 && (!(a_raw >= 0.0) || !(s_raw >= 0.0))) p.status[s_mat] = -1;
    const double amp = a_raw + MIN_PARAM_VALUE, sn = s_raw + MIN_PARAM_VALUE;
    double acc[17][2];
#pragma unroll
    for (int t = 0; t < 17; ++t) acc[t][0] = acc[t][1] = 0.0;
    if (jc > 0) {
      // ---- SYRK of the diagonal tile: both operands are row block j of L, so a stage is ONE 16 KB macro-tile ----
      uint64_t *full = bars, *empty = bars + PF_RING_STAGES;
      int pos0 = 0;   // stage index the ring starts at (a variable: folding it away changes ptxas' register allocation)
      if (tid < 2 * PF_RING_STAGES) {
        mbar_init(smem_u32(&bars[tid]), tid < PF_RING_STAGES ? 1u : 8u);
        mbar_fence_init();
      }
      __syncthreads();
      const double *src = p.L + (size_t)s_mat * p.L_stride + (size_t)jc * p.ktiles * TILE_ELEMS;
      const int nk = jc * KT_PER_BLOCK;
      int issued = 0;
      auto try_issue = [&](bool blocking) -> bool {
        const int ai = pos0 + issued, slot = ai % PF_RING_STAGES;
        if (ai >= PF_RING_STAGES) {
          const uint32_t eb = smem_u32(&empty[slot]);
          const uint32_t par = (uint32_t)((ai / PF_RING_STAGES - 1) & 1);
          if (blocking)
            mbar_wait(eb, par);
          else if (!mbar_try_wait(eb, par))
            return false;
        }
        const uint32_t bar = smem_u32(&full[slot]);
        mbar_arrive_expect_tx(bar, TILE_BYTES);
        bulk_g2s(smem_u32(sm + (size_t)slot * TILE_ELEMS), src + (size_t)issued * TILE_ELEMS, TILE_BYTES, bar);
        ++issued;
        return true;
      };
      if (tid == 0)
        while (issued < nk && issued < PF_RING_STAGES) try_issue(false);
      const int n0 = 16 - warp, c4 = lane & 3;
      const int b0off = warp * 128 + 2 * lane, b1off = (15 - warp) * 128 + 2 * lane;
      const bool fwd = p.fwd_w != nullptr;
      const double *wv = fwd ? p.fwd_w + (size_t)s_mat * p.n_pad + c4 : nullptr;
      double r0 = 0.0, r1 = 0.0;
      for (int g = 0; g < nk; ++g) {
        const int slot = (pos0 + g) % PF_RING_STAGES;
        if (tid == 0) {
          while (issued < nk && issued < g + PF_RING_STAGES) {
            if (!try_issue(issued <= g)) break;
          }
        }
        mbar_wait(smem_u32(&full[slot]), (uint32_t)(((pos0 + g) / PF_RING_STAGES) & 1));
        const double *st = sm + (size_t)slot * TILE_ELEMS;
#pragma unroll
        for (int mc = 0; mc < 2; ++mc) {
          const double2 b0 = lds128(st + b0off + mc * 64), b1 = lds128(st + b1off + mc * 64);
          // two batches of fragments (9 + 8 tiles) keep the kernel inside its 128-register budget (2 CTAs / SM)
          pf_syrk_batch<0, 9>(acc, st + 2 * lane + mc * 64, warp, n0, b0, b1);
          pf_syrk_batch<9, 17>(acc, st + 2 * lane + mc * 64, warp, n0, b0, b1);
          if (mc == 1) {
            if (fwd) {
              // warp w owns micro-rows 2w and 2w+1 of the row block; lane T holds (row T/4, k = T%4 and 4 + T%4)
              const double *ar = st + (4 * warp) * 64 + 2 * lane;
              const double *wk = wv + g * 16;
              const double w0 = wk[0], w1 = wk[4], w2 = wk[8], w3 = wk[12];
              const double2 a00 = lds128(ar), a01 = lds128(ar + 64), a10 = lds128(ar + 128), a11 = lds128(ar + 192);
              r0 = fma(a00.x, w0, r0);
              r0 = fma(a00.y, w1, r0);
              r0 = fma(a01.x, w2, r0);
              r0 = fma(a01.y, w3, r0);
              r1 = fma(a10.x, w0, r1);
              r1 = fma(a10.y, w1, r1);
              r1 = fma(a11.x, w2, r1);
              r1 = fma(a11.y, w3, r1);
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(smem_u32(&empty[slot]));
          }
        }
      }
      if (fwd) {
        r0 += __shfl_xor_sync(0xffffffffu, r0, 1);
        r0 += __shfl_xor_sync(0xffffffffu, r0, 2);
        r1 += __shfl_xor_sync(0xffffffffu, r1, 1);
        r1 += __shfl_xor_sync(0xffffffffu, r1, 2);
        if (c4 == 0) {
          rsum[16 * warp + (lane >> 2)] = r0;
          rsum[16 * warp + 8 + (lane >> 2)] = r1;
        }
      }
    } else if (tid < 128) {
      rsum[tid] = 0.0;
    }
    __syncthreads();   // every warp is through the ring: the tile store and tmp are free
    // ---- scaled (and rounded) training inputs of this block into tmp, then K_jj - acc into the tile store ----
    const int dp = p.gen_dp, row0 = jc * 128;
    for (int e = tid; e < 128 * dp; e += 256) {
      const int rr = e / dp, i = e - rr * dp, gi = row0 + rr;
      double v = 0.0;
      if (gi < p.gen_n && i < p.gen_d) {
        v = p.gen_X[(size_t)gi * p.gen_d + i];
        if ((p.gen_disc >> i) & 1ull) v = rint(v);
        v *= invl[i];
      }
      tmp[e] = v;
    }
    __syncthreads();
    // accumulators -> tile store (static indices), each thread re-reads only its own elements below
#pragma unroll
    for (int t = 0; t < 17; ++t) {
      const int R = t < 16 - warp ? warp + t : t - 1, Cs = t < 16 - warp ? warp : 15 - warp;
      double *dst = T + ((R * (R + 1)) / 2 + Cs) * 64;
      dst[pt_cpos(lane, 0)] = acc[t][0];
      dst[pt_cpos(lane, 1)] = acc[t][1];
    }
    const double a2 = amp * amp, s2 = sn * sn;
    switch (p.gen_kid) {   // every KID explicitly: an unknown id generates nothing (the host decodes ids first)
      case 0: pf_generate_tile<0>(T, tmp, dp, warp, lane, row0, p.gen_n, a2, s2, etab, p.gen_rq_a); break;
      case 1: pf_generate_tile<1>(T, tmp, dp, warp, lane, row0, p.gen_n, a2, s2, etab, p.gen_rq_a); break;
      case 2: pf_generate_tile<2>(T, tmp, dp, warp, lane, row0, p.gen_n, a2, s2, etab, p.gen_rq_a); break;
      case 3: pf_generate_tile<3>(T, tmp, dp, warp, lane, row0, p.gen_n, a2, s2, etab, p.gen_rq_a); break;
      case 4: pf_generate_tile<4>(T, tmp, dp, warp, lane, row0, p.gen_n, a2, s2, etab, p.gen_rq_a); break;
      default: break;
    }
  }
  __syncthreads();

  // ---- factorisation ----
  // C(I, col) -= sum_{t in [t0, t1)} L(I, t) L(col, t)^T, four independent accumulator pairs
  auto apply = [&](int I, int col, int t0, int t1) {
    double c[4][2];
#pragma unroll
    for (int q = 0; q < 4; ++q) c[q][0] = c[q][1] = 0.0;
    const double *ti = T + pt_tile(I, 0) + 2 * lane, *ts = T + pt_tile(col, 0) + 2 * lane;
    for (int t = t0; t < t1; t += 4) {
      double2 a[4], b[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        if (t + q < t1) {
          a[q] = lds128(ti + (t + q) * 64);
          b[q] = lds128(ts + (t + q) * 64);
        }
      }
#pragma unroll
      for (int q = 0; q < 4; ++q)
        if (t + q < t1) dmma884(c[q][0], c[q][1], a[q].x, b[q].x);
#pragma unroll
      for (int q = 0; q < 4; ++q)
        if (t + q < t1) dmma884(c[q][0], c[q][1], a[q].y, b[q].y);
    }
    double *dst = T + pt_tile(I, col);
    dst[pt_cpos(lane, 0)] -= (c[0][0] + c[1][0]) + (c[2][0] + c[3][0]);
    dst[pt_cpos(lane, 1)] -= (c[0][1] + c[1][1]) + (c[2][1] + c[3][1]);
  };
  for (int s = 0; s < 16; ++s) {
    // (a) finish column s: the terms t < s-1 were applied ahead of time during step s-1
    if (s > 0) {
      for (int I = s + warp; I < 16; I += 8) apply(I, s, s - 1, s);
      __syncthreads();
    }
    if (warp < 4) {
      // (b) every participating thread factors the 8x8 diagonal tile redundantly in registers (no shuffles, no
      //     extra barrier), then solves its own row of the panel below:  x L_ss^T = c.  Thread 0 publishes L_ss.
      const int nrows = (15 - s) * 8;
      double *d = T + pt_tile(s, s);
      double l[8][8];
      double rsv[8];
      bool bad = false;
      if (tid < (nrows > 32 ? nrows : 32)) {
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
          for (int c = 0; c <= i; ++c) l[i][c] = d[(i << 3) + ((c & 3) << 1) + (c >> 2)];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const double piv = l[k][k];
          bad |= !(piv > 1e-300);   // LAPACK dpotrf info > 0 (also catches NaN and pivots the flush-to-zero seed
                                    // cannot take); off the dependent chain: a bad pivot only poisons this matrix
                                    // with NaN / Inf, and its status reports it
          // 1/sqrt(piv) and sqrt(piv): MUFU seed (2^-22) + two coupled Newton steps on (g, y) -> (sqrt, rsqrt);
          // five dependent FP64 operations (the pivot chain is this kernel's critical path)
          double y;
          asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(piv));
          double gq = piv * y;
          double rq = fma(-gq, y, 1.0);
          gq = fma(0.5 * gq, rq, gq);
          y = fma(0.5 * y, rq, y);
          rq = fma(-gq, y, 1.0);
          gq = fma(0.5 * gq, rq, gq);
          const double rs = fma(0.5 * y, rq, y);
          rsv[k] = rs;
          l[k][k] = gq;
#pragma unroll
          for (int i = k + 1; i < 8; ++i) l[i][k] *= rs;
#pragma unroll
          for (int jj = k + 1; jj < 8; ++jj)
#pragma unroll
            for (int i = jj; i < 8; ++i) l[i][jj] = fma(-l[i][k], l[jj][k], l[i][jj]);
        }
        if (tid < nrows) {
          const int I = s + 1 + (tid >> 3), r = tid & 7;
          double *row = T + pt_tile(I, s) + (r << 3);
          double x[8];
#pragma unroll
          for (int c = 0; c < 8; ++c) x[c] = row[((c & 3) << 1) + (c >> 2)];
#pragma unroll
          for (int k = 0; k < 8; ++k) {
            double acc = x[k];
#pragma unroll
            for (int m = 0; m < k; ++m) acc = fma(-x[m], l[k][m], acc);
            x[k] = acc * rsv[k];
          }
#pragma unroll
          for (int c = 0; c < 8; ++c) row[((c & 3) << 1) + (c >> 2)] = x[c];
        }
      }
      // Thread 0 overwrites the diagonal tile with L_ss.  Every other thread of warps 0-3 reads that tile above, and
      // the compiler is free to fetch those values late (re-materialised shared-memory loads under register
      // pressure), so the overwrite needs its own barrier over the four warps: without it a lagging warp factored
      // a half-published tile once in a few hundred launches (tests: test_loglik_is_repeatable_and_split_invariant).
      asm volatile("bar.sync 1, 128;" ::: "memory");
      if (tid == 0) {
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
          for (int c = 0; c < 8; ++c) d[(i << 3) + ((c & 3) << 1) + (c >> 2)] = (c <= i) ? l[i][c] : 0.0;
#pragma unroll
        for (int k = 0; k < 8; ++k) dinv[s * 8 + k] = rsv[k];
        if (bad) *flag = 1;
      }
    } else if (s > 0 && s < 15) {
      // (c) look-ahead on the otherwise idle warps: columns t < s are final, apply them to column s+1 now
      //     (tiles (I, s+1) and columns < s are not touched by (b), which works on column s)
      for (int I = s + 1 + (warp - 4); I < 16; I += 4) apply(I, s + 1, 0, s);
    }
    __syncthreads();
  }

  // ---- log L_kk in parallel, L -> global (upper part zero); the fixed-order sum runs on an idle thread below ----
  if (tid < 128) lg[tid] = -log(dinv[tid]);
  if (!FUSED || p.store_L) {   // the left-looking batch paths never read L_jj again (only Winv_jj)
    for (int e = 2 * tid; e < TM * TM; e += 512) {   // 16 B per lane, a micro-tile per warp pass
      const int kt = e >> 11, micro = (e >> 6) & 31, w = e & 63;
      const int I = micro >> 1, J = (kt << 1) + (micro & 1);
      *reinterpret_cast<double2 *>(blk + e) = (J <= I) ? lds128(T + pt_tile(I, J) + w) : make_double2(0.0, 0.0);
    }
  }
  __syncthreads();
  if (tid == 255) {
    if (*flag && p.status[s_mat] == 0) p.status[s_mat] = 1;
    double ld = 0.0;
    for (int k = 0; k < 128; ++k) ld += lg[k];
    p.logdet_blk[(size_t)s_mat * p.nblk + jc] = ld;
  }

  // ---- inverse, level 0: 8x8 diagonal tiles, one column per thread (threads 0..127) -> tmp, then back ----
  if (tid < 128) {
    const int u = tid >> 3, c = tid & 7;
    const double *ld = T + pt_tile(u, u);
    double w[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      double acc = (i == c) ? 1.0 : 0.0;
#pragma unroll
      for (int m = 0; m < i; ++m) acc = fma(-ld[(i << 3) + ((m & 3) << 1) + (m >> 2)], w[m], acc);
      w[i] = (i >= c) ? acc * dinv[u * 8 + i] : 0.0;
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) tmp[u * 64 + (i << 3) + ((c & 3) << 1) + (c >> 2)] = w[i];
  }
  __syncthreads();
  if (tid < 128) {
    const int u = tid >> 3, r = tid & 7;
    double *d = T + pt_tile(u, u) + (r << 3);
    const double *sv = tmp + u * 64 + (r << 3);
#pragma unroll
    for (int q = 0; q < 8; ++q) d[q] = sv[q];
  }
  __syncthreads();

  // ---- inverse, recursive doubling: diagonal blocks of mt tiles are inverted; merge pairs.  A warp works on two
  //      output tiles with the same k-range at a time (four independent DMMA chains) ----
  for (int mt = 1; mt < 16; mt <<= 1) {
    const int npair = 16 / (2 * mt), per = mt * mt;
    const int hm = mt > 1 ? mt / 2 : 1, two = mt > 1 ? 2 : 1;   // tiles per unit: 2 (mt >= 2) or 1
    // step A: Tm(I, J) = sum_{t = J}^{mt-1} L21(I, t) W11(t, J)        -> tmp tile (pair, I, J);  unit = (pair, J, I/2)
    for (int u = warp; u < npair * mt * hm; u += 8) {
      const int pr = u / (mt * hm), J = (u / hm) % mt, I0 = two * (u % hm);
      const int R0 = 2 * pr * mt + mt, C0 = 2 * pr * mt;
      double c0 = 0.0, c1 = 0.0, e0 = 0.0, e1 = 0.0, f0 = 0.0, f1 = 0.0, g0 = 0.0, g1 = 0.0;
      const int I1 = I0 + two - 1;   // == I0 when mt == 1 (second tile skipped below)
      int t = J;
      for (; t + 1 < mt; t += 2) {
        const double2 b = pt_ldT(T + pt_tile(C0 + t, C0 + J), lane), b2 = pt_ldT(T + pt_tile(C0 + t + 1, C0 + J), lane);
        const double2 a = lds128(T + pt_tile(R0 + I0, C0 + t) + 2 * lane), a2 = lds128(T + pt_tile(R0 + I0, C0 + t + 1) + 2 * lane);
        const double2 p = lds128(T + pt_tile(R0 + I1, C0 + t) + 2 * lane), p2 = lds128(T + pt_tile(R0 + I1, C0 + t + 1) + 2 * lane);
        dmma884(c0, c1, a.x, b.x);
        dmma884(e0, e1, a2.x, b2.x);
        dmma884(f0, f1, p.x, b.x);
        dmma884(g0, g1, p2.x, b2.x);
        dmma884(c0, c1, a.y, b.y);
        dmma884(e0, e1, a2.y, b2.y);
        dmma884(f0, f1, p.y, b.y);
        dmma884(g0, g1, p2.y, b2.y);
      }
      if (t < mt) {
        const double2 b = pt_ldT(T + pt_tile(C0 + t, C0 + J), lane);
        const double2 a = lds128(T + pt_tile(R0 + I0, C0 + t) + 2 * lane), p = lds128(T + pt_tile(R0 + I1, C0 + t) + 2 * lane);
        dmma884(c0, c1, a.x, b.x);
        dmma884(f0, f1, p.x, b.x);
        dmma884(c0, c1, a.y, b.y);
        dmma884(f0, f1, p.y, b.y);
      }
      double *dst = tmp + (size_t)(pr * per + I0 * mt + J) * 64;
      dst[pt_cpos(lane, 0)] = c0 + e0;
      dst[pt_cpos(lane, 1)] = c1 + e1;
      if (two == 2) {
        dst += (size_t)mt * 64;
        dst[pt_cpos(lane, 0)] = f0 + g0;
        dst[pt_cpos(lane, 1)] = f1 + g1;
      }
    }
    __syncthreads();
    // step B: W21(I, J) = - sum_{t = 0}^{I} W22(I, t) Tm(t, J)          -> overwrites L21;  unit = (pair, I, J/2)
    for (int u = warp; u < npair * mt * hm; u += 8) {
      const int pr = u / (mt * hm), I = (u / hm) % mt, J0 = two * (u % hm);
      const int R0 = 2 * pr * mt + mt, C0 = 2 * pr * mt;
      const double *tm = tmp + (size_t)pr * per * 64;
      const int J1 = J0 + two - 1;
      double c0 = 0.0, c1 = 0.0, e0 = 0.0, e1 = 0.0, f0 = 0.0, f1 = 0.0, g0 = 0.0, g1 = 0.0;
      int t = 0;
      for (; t + 1 <= I; t += 2) {
        const double2 a = lds128(T + pt_tile(R0 + I, R0 + t) + 2 * lane), a2 = lds128(T + pt_tile(R0 + I, R0 + t + 1) + 2 * lane);
        const double2 b = pt_ldT(tm + (t * mt + J0) * 64, lane), b2 = pt_ldT(tm + ((t + 1) * mt + J0) * 64, lane);
        const double2 q = pt_ldT(tm + (t * mt + J1) * 64, lane), q2 = pt_ldT(tm + ((t + 1) * mt + J1) * 64, lane);
        dmma884(c0, c1, a.x, b.x);
        dmma884(e0, e1, a2.x, b2.x);
        dmma884(f0, f1, a.x, q.x);
        dmma884(g0, g1, a2.x, q2.x);
        dmma884(c0, c1, a.y, b.y);
        dmma884(e0, e1, a2.y, b2.y);
        dmma884(f0, f1, a.y, q.y);
        dmma884(g0, g1, a2.y, q2.y);
      }
      if (t <= I) {
        const double2 a = lds128(T + pt_tile(R0 + I, R0 + t) + 2 * lane);
        const double2 b = pt_ldT(tm + (t * mt + J0) * 64, lane), q = pt_ldT(tm + (t * mt + J1) * 64, lane);
        dmma884(c0, c1, a.x, b.x);
        dmma884(f0, f1, a.x, q.x);
        dmma884(c0, c1, a.y, b.y);
        dmma884(f0, f1, a.y, q.y);
      }
      double *dst = T + pt_tile(R0 + I, C0 + J0);
      dst[pt_cpos(lane, 0)] = -(c0 + e0);
      dst[pt_cpos(lane, 1)] = -(c1 + e1);
      if (two == 2) {
        dst += 64;   // tile (R0 + I, C0 + J0 + 1)
        dst[pt_cpos(lane, 0)] = -(f0 + g0);
        dst[pt_cpos(lane, 1)] = -(f1 + g1);
      }
    }
    __syncthreads();
  }

  // ---- Winv_jj -> global (and, for a posterior fit, into W(j,j) and transposed into WT(j,j)) ----
  double *wi = p.Winv + (size_t)s_mat * p.Winv_stride + (size_t)jc * (TM * TM);
  double *wfull = p.W ? p.W + (size_t)s_mat * p.W_stride + ((size_t)jc * p.ktiles + (size_t)jc * KT_PER_BLOCK) * TILE_ELEMS : nullptr;
  double *wtfull = p.WT ? p.WT + (size_t)s_mat * p.W_stride + ((size_t)jc * p.ktiles + (size_t)jc * KT_PER_BLOCK) * TILE_ELEMS : nullptr;
  for (int e = 2 * tid; e < TM * TM; e += 512) {   // 16 B per lane, a micro-tile per warp pass
    const int kt = e >> 11, micro = (e >> 6) & 31, w = e & 63;
    const int I = micro >> 1, J = (kt << 1) + (micro & 1);
    const double2 v = (J <= I) ? lds128(T + pt_tile(I, J) + w) : make_double2(0.0, 0.0);
    *reinterpret_cast<double2 *>(wi + e) = v;
    if (wfull) *reinterpret_cast<double2 *>(wfull + e) = v;
    if (wtfull) {
      // element (r, c) of tile (I, J) of W^T is element (c, r) of tile (J, I) of W; w and w+1 are (r, c) and (r, c+4)
      const int r = w >> 3, c = (w >> 1) & 3;
      const double *src = T + pt_tile(J, I);
      *reinterpret_cast<double2 *>(wtfull + e) =
          (I <= J) ? make_double2(src[pt_elem(c, r)], src[pt_elem(c + 4, r)]) : make_double2(0.0, 0.0);
    }
  }

  // ---- forward substitution step of the log-likelihood: w_j = Winv_jj (delta_j - r_j), |w_j|^2 ----
  if (p.fwd_w) {
    if (tid < 128) {
      const int row = jc * 128 + tid;
      const double dl = (row < p.fwd_n) ? p.fwd_ymm[(size_t)s_mat * p.fwd_ldy + row] : 0.0;
      double rj;
      if constexpr (FUSED)
        rj = (fv + 136 + PF_BAR_SLOTS + EXPTAB_N + 32)[tid];
      else
        rj = jc > 0 ? p.fwd_r[(size_t)s_mat * p.n_pad + row] : 0.0;
      fv[tid] = dl - rj;
    }
    __syncthreads();
    // warp w: micro-rows 2w, 2w+1; lane T holds (row T/4, columns T%4 and 4 + T%4) of each 8x8 tile
    const int c4 = lane & 3;
    double sq = 0.0;
#pragma unroll
    for (int m = 0; m < 2; ++m) {
      const int I = 2 * warp + m;
      double acc = 0.0;
      for (int J = 0; J <= I; ++J) {
        const double2 a = lds128(T + pt_tile(I, J) + 2 * lane);
        acc = fma(a.x, fv[J * 8 + c4], acc);
        acc = fma(a.y, fv[J * 8 + c4 + 4], acc);
      }
      acc += __shfl_xor_sync(0xffffffffu, acc, 1);
      acc += __shfl_xor_sync(0xffffffffu, acc, 2);
      if (c4 == 0) {
        p.fwd_w[(size_t)s_mat * p.n_pad + jc * 128 + I * 8 + (lane >> 2)] = acc;
        sq = fma(acc, acc, sq);
      }
    }
    sq += __shfl_xor_sync(0xffffffffu, sq, 4);    // lanes with c4 == 0 hold the rows; fixed tree
    sq += __shfl_xor_sync(0xffffffffu, sq, 8);
    sq += __shfl_xor_sync(0xffffffffu, sq, 16);
    if (lane == 0) fv[128 + warp] = sq;
    __syncthreads();
    if (tid == 0) {
      double t = 0.0;
      for (int q = 0; q < 8; ++q) t += fv[128 + q];
      p.fwd_ssq[(size_t)s_mat * p.nblk + jc] = t;
    }
  }
}

__global__ void __launch_bounds__(256, 2) potrf_tile_kernel(PotrfParams p) { potrf_tile_body<false>(p, blockIdx.x, p.j); }
__global__ void __launch_bounds__(256, 2) potrf_fused_kernel(PotrfParams p) { potrf_tile_body<true>(p, blockIdx.x, p.j); }

}  // namespace boss

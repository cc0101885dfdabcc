// chol_matrix.cuh -- batched log marginal likelihood for small kernel matrices (n_pad <= 512: 1..4 diagonal blocks),
// ONE persistent CTA per matrix, two CTAs per SM.
//
// BASELINE config C3 (4096 hyper-parameter samples x n = 512) spends its time in launch-level dependencies when the
// block-column steps are separate kernels: every step waits for the slowest matrix of its group, the latency-bound
// diagonal-block factorisation (potf2 chain) owns its SMs while the tensor pipe idles, and GEMM CTAs with K = 128..384
// are half pipeline fill.  Here a CTA takes a whole matrix through the left-looking factorisation without leaving
// the SM:
//
//   for block column j:   U(i,j)  T_ij = K_ij - sum_{k<j} L_ik L_jk^T   (i > j)    K_ij generated from the hyper-parameters
//                                                                                  in the epilogue (K never exists in HBM)
//                         D(j)    K_jj - SYRK, potf2, Winv_jj = L_jj^-1, log-det, forward-substitution block
//                                 (potrf128.cuh: potrf_tile_body<true, true>; Winv_jj stays in shared memory)
//                         S(i,j)  L_ij = T_ij Winv_jj^T                  (i > j)    B operand = the resident Winv_jj
//
// L tiles travel through global memory (L2) between the steps -- they are the operands of later block columns -- but
// there is no launch boundary, no inter-CTA dependency and no HBM trip for K, the diagonal tiles or Winv.  With 128
// registers per thread and 107 KB of shared memory two matrices share an SM, so one matrix's potf2 / inverse chain
// overlaps the other's DMMA work: the overlap the multi-kernel pipeline could only get between different SMs.
// GEMM-shaped steps work on 128 x 64 half tiles (8 warps x (32 x 32), 64 accumulator registers); the update ring has
// 4 stages of 24 KB (A 128 x 16, B 64 x 16) in the not-yet-used tile store, the solve ring 2 stages of 16 KB.
//
// Reference: gp_data_loglike_slice (src/models/gaussian_process.jl:269-280) -> logpdf(::FiniteGP, y) evaluated for
// the hyper-parameter batches of SamplingMAP (src/model_fitters/sampling.jl:59-78) and ext/TuringExt.jl:54-68.
#pragma once
#include "gemm_core.cuh"
#include "potrf128.cuh"

namespace boss {

constexpr int CM_MAX_NBLK = 4;
constexpr int CM_U_STAGES = 4, CM_U_STAGE_ELEMS = TILE_ELEMS + TILE_ELEMS / 2;   // A 128x16 + B 64x16 = 24 KB
constexpr int CM_S_STAGES = 2;                                                    // A 128x16 = 16 KB each, in tmp
constexpr int CM_SMEM_BYTES = PF_SMEM_BYTES;

__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async;" ::: "memory"); }

// A small TMA ring whose stages hold one or two bulk copies.  Each ring shape owns its barriers (initialised once at
// kernel start) and carries the absolute index of its next stage from job to job, so the phases just keep counting.
template <int NST>
struct CmRing {
  double *base;
  uint64_t *full, *empty;
  int stage_elems, pos0, issued;   // pos0: absolute index of this job's stage 0; issued: stages issued in this job
  __device__ __forceinline__ void begin(double *b, uint64_t *bars, int se, int pos) {
    base = b;
    full = bars;
    empty = bars + NST;
    stage_elems = se;
    pos0 = pos;
    issued = 0;
    fence_proxy_async();   // generic-proxy accesses of the ring area (tile store / scratch) precede the bulk copies
    __syncthreads();
  }
  // thread 0: issue stage `issued` = (srcA, bytesA) [+ (srcB, bytesB) behind it]
  __device__ __forceinline__ bool try_issue(const double *srcA, uint32_t bytesA, const double *srcB, uint32_t bytesB, bool blocking) {
    const int ai = pos0 + issued, slot = ai % NST;
    if (ai >= NST) {
      const uint32_t eb = smem_u32(&empty[slot]);
      const uint32_t par = (uint32_t)((ai / NST - 1) & 1);
      if (blocking)
        mbar_wait(eb, par);
      else if (!mbar_try_wait(eb, par))
        return false;
    }
    const uint32_t bar = smem_u32(&full[slot]);
    double *dst = base + (size_t)slot * stage_elems;
    mbar_arrive_expect_tx(bar, bytesA + bytesB);
    bulk_g2s(smem_u32(dst), srcA, bytesA, bar);
    if (bytesB) bulk_g2s(smem_u32(dst + bytesA / 8), srcB, bytesB, bar);
    ++issued;
    return true;
  }
  __device__ __forceinline__ const double *wait(int g) const {
    const int ai = pos0 + g;
    mbar_wait(smem_u32(&full[ai % NST]), (uint32_t)((ai / NST) & 1));
    return base + (size_t)(ai % NST) * stage_elems;
  }
  __device__ __forceinline__ void release(int g) const {
    __syncwarp();
    if ((threadIdx.x & 31) == 0) mbar_arrive(smem_u32(&empty[(pos0 + g) % NST]));
  }
};

// running stage counters of the three rings of a CTA (uniform across its threads)
struct CmPos {
  int d, u, s;
};

struct CmParams {
  PotrfParams pp;     // L, strides, nblk, ktiles, status, logdet_blk, fwd_*, gen_* (see potrf128.cuh); pp.j is not used
  long long S;        // matrices in the batch
};

// ---- U(i, j, h): half tile h (columns 64h .. 64h+63) of T_ij = K_ij - sum_{k<j} L_ik L_jk^T  ->  global block (i, j) ----
template <int KID>
__device__ __forceinline__ void cm_update_job(const PotrfParams &p, const int s_mat, const int i, const int j, const int h,
                                              double *sm, uint64_t *bars, int &pos, const double *etab, const double *invl,
                                              const double a2) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, wm = warp >> 1, wn = warp & 1;
  double *Lm = p.L + (size_t)s_mat * p.L_stride;
  double acc[4][4][2];
#pragma unroll
  for (int fm = 0; fm < 4; ++fm)
#pragma unroll
    for (int fn = 0; fn < 4; ++fn) acc[fm][fn][0] = acc[fm][fn][1] = 0.0;
  const int nk = j * KT_PER_BLOCK;
  if (nk > 0) {
    CmRing<CM_U_STAGES> rg;
    rg.begin(sm, bars + 12, CM_U_STAGE_ELEMS, pos);
    pos += nk;
    const double *srcA = Lm + (size_t)i * p.ktiles * TILE_ELEMS;                            // row block i, k-tiles 0..
    const double *srcB = Lm + (size_t)j * p.ktiles * TILE_ELEMS + (size_t)h * (TILE_ELEMS / 2);   // rows 64h.. of row block j
    auto feed = [&](int g) {
      while (rg.issued < nk && rg.issued < g + CM_U_STAGES) {
        const size_t o = (size_t)rg.issued * TILE_ELEMS;
        if (!rg.try_issue(srcA + o, TILE_BYTES, srcB + o, TILE_BYTES / 2, rg.issued <= g)) break;
      }
    };
    if (tid == 0) feed(0);
    const int a_off = (4 * wm) * 128 + 2 * lane, b_off = TILE_ELEMS + (4 * wn) * 128 + 2 * lane;
    for (int g = 0; g < nk; ++g) {
      if (tid == 0) feed(g);
      const double *st = rg.wait(g);
#pragma unroll
      for (int mc = 0; mc < 2; ++mc) {
        double2 a[4], b[4];
#pragma unroll
        for (int fm = 0; fm < 4; ++fm) a[fm] = lds128(st + a_off + fm * 128 + mc * 64);
#pragma unroll
        for (int fn = 0; fn < 4; ++fn) b[fn] = lds128(st + b_off + fn * 128 + mc * 64);
#pragma unroll
        for (int fm = 0; fm < 4; ++fm)
#pragma unroll
          for (int fn = 0; fn < 4; ++fn) dmma884(acc[fm][fn][0], acc[fm][fn][1], a[fm].x, b[fn].x);
        if (mc == 1) rg.release(g);
#pragma unroll
        for (int fm = 0; fm < 4; ++fm)
#pragma unroll
          for (int fn = 0; fn < 4; ++fn) dmma884(acc[fm][fn][0], acc[fm][fn][1], a[fm].y, b[fn].y);
      }
    }
  }
  __syncthreads();   // every warp is through the ring
  // scaled (and rounded) inputs of row block i (128 points) and of columns 64h.. of block j (64 points) -> shared memory
  const int dp = p.gen_dp;
  double *xi = sm, *xj = sm + 128 * dp;
  for (int e = tid; e < 192 * dp; e += 256) {
    const int rr = e / dp, q = e - rr * dp;
    const int gi = rr < 128 ? i * 128 + rr : j * 128 + 64 * h + (rr - 128);
    double v = 0.0;
    if (gi < p.gen_n && q < p.gen_d) {
      v = p.gen_X[(size_t)gi * p.gen_d + q];
      if ((p.gen_disc >> q) & 1ull) v = rint(v);
      v *= invl[q];
    }
    sm[e] = v;
  }
  __syncthreads();
  double *dst = Lm + ((size_t)i * p.ktiles + (size_t)j * KT_PER_BLOCK) * TILE_ELEMS;
  // The accumulators go to their destination first (static indices, 16-byte lane-pair stores); the kernel values are
  // then generated in a rolled loop by the thread that holds each pair and combined in place -- generating them with the
  // 64 accumulator registers still live does not fit the 128-register budget of a 2-CTA/SM kernel.
#pragma unroll
  for (int fm = 0; fm < 4; ++fm)
#pragma unroll
    for (int fn = 0; fn < 4; ++fn) p_store_cfrag(dst, 4 * wm + fm, 8 * h + 4 * wn + fn, lane, acc[fm][fn][0], acc[fm][fn][1]);
  const int q4 = lane & 3, k3 = q4 < 2 ? 2 * q4 : 2 * q4 - 3;   // the pair a lane stored: columns k3 and k3 + 4 of its row
#pragma unroll 1
  for (int t = 0; t < 16; ++t) {
    const int fm = t >> 2, fn = t & 3;
    const int rslab = 4 * wm + fm, cslab = 8 * h + 4 * wn + fn;
    const int r = 8 * rslab + (lane >> 2), c = 32 * wn + 8 * fn + k3;      // c: column inside this half (0..63)
    const double *xr = xi + r * dp, *xc = xj + c * dp;
    double d20 = 0.0, d21 = 0.0;
    for (int q = 0; q < dp; ++q) {
      const double x = xr[q], df0 = x - xc[q], df1 = x - xc[4 * dp + q];
      d20 = fma(df0, df0, d20);
      d21 = fma(df1, df1, d21);
    }
    double v0 = a2 * kappa_fast<KID>(d20, etab, p.gen_rq_a), v1 = a2 * kappa_fast<KID>(d21, etab, p.gen_rq_a);
    const bool row_live = i * 128 + r < p.gen_n;
    const int gj = j * 128 + 64 * h + c;
    if (!(row_live && gj < p.gen_n)) v0 = 0.0;            // padding rows / columns of an off-diagonal block are zero
    if (!(row_live && gj + 4 < p.gen_n)) v1 = 0.0;
    double2 *pq = reinterpret_cast<double2 *>(dst + (cslab >> 1) * TILE_ELEMS + (((rslab << 1) + (cslab & 1)) << 6) +
                                              ((((lane >> 2) << 2) + k3) << 1));
    const double2 sacc = *pq;
    *pq = make_double2(v0 - sacc.x, v1 - sacc.y);
  }
  fence_proxy_async();   // these tiles are read back by bulk copies (solve step, later block columns)
  __syncthreads();
}

// live column slabs LO..3 of the warp in one k micro-step of the solve (Winv_jj is lower triangular)
template <int LO>
__device__ __forceinline__ void cm_solve_step(double (&acc)[4][4][2], const double2 (&a)[4], const double *T, const int c0,
                                              const int kk, const int lane) {
  double2 b[4];
#pragma unroll
  for (int fn = LO; fn < 4; ++fn) b[fn] = lds128(T + pt_tile(c0 + fn, kk) + 2 * lane);
#pragma unroll
  for (int fm = 0; fm < 4; ++fm)
#pragma unroll
    for (int fn = LO; fn < 4; ++fn) dmma884(acc[fm][fn][0], acc[fm][fn][1], a[fm].x, b[fn].x);
#pragma unroll
  for (int fm = 0; fm < 4; ++fm)
#pragma unroll
    for (int fn = LO; fn < 4; ++fn) dmma884(acc[fm][fn][0], acc[fm][fn][1], a[fm].y, b[fn].y);
}

// ---- S(i, j, h): columns 64h .. 64h+63 of L_ij = T_ij Winv_jj^T, in place in global block (i, j).  Winv_jj is the
//      packed lower-triangular tile store in shared memory; T_ij streams through a 2-stage ring in tmp.  Half 1 must run
//      before half 0 (it still needs the T values of columns 0..63). ----
__device__ __forceinline__ void cm_solve_job(const PotrfParams &p, const int s_mat, const int i, const int j, const int h,
                                             double *sm, uint64_t *bars, int &pos) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, wm = warp >> 1, wn = warp & 1;
  double *blk = p.L + (size_t)s_mat * p.L_stride + ((size_t)i * p.ktiles + (size_t)j * KT_PER_BLOCK) * TILE_ELEMS;
  const double *T = sm;
  double acc[4][4][2];
#pragma unroll
  for (int fm = 0; fm < 4; ++fm)
#pragma unroll
    for (int fn = 0; fn < 4; ++fn) acc[fm][fn][0] = acc[fm][fn][1] = 0.0;
  const int nk = 4 * (h + 1);   // k-tiles 0 .. 4(h+1)-1: Winv rows 64h.. have no entries beyond column 64h+63
  CmRing<CM_S_STAGES> rg;
  rg.begin(sm + PT_TILES * 64, bars + 12 + 2 * CM_U_STAGES, TILE_ELEMS, pos);
  pos += nk;
  auto feed = [&](int g) {
    while (rg.issued < nk && rg.issued < g + CM_S_STAGES) {
      if (!rg.try_issue(blk + (size_t)rg.issued * TILE_ELEMS, TILE_BYTES, nullptr, 0, rg.issued <= g)) break;
    }
  };
  if (tid == 0) feed(0);
  const int a_off = (4 * wm) * 128 + 2 * lane, c0 = 8 * h + 4 * wn;
  for (int g = 0; g < nk; ++g) {
    if (tid == 0) feed(g);
    const double *st = rg.wait(g);
#pragma unroll 1
    for (int mc = 0; mc < 2; ++mc) {
      const int kk = 2 * g + mc;
      if (kk <= c0 + 3) {                       // warp-uniform: real branches (a predicated-off DMMA still costs its slot)
        double2 a[4];
#pragma unroll
        for (int fm = 0; fm < 4; ++fm) a[fm] = lds128(st + a_off + fm * 128 + mc * 64);
        const int lo = kk - c0;
        if (lo <= 0)
          cm_solve_step<0>(acc, a, T, c0, kk, lane);
        else if (lo == 1)
          cm_solve_step<1>(acc, a, T, c0, kk, lane);
        else if (lo == 2)
          cm_solve_step<2>(acc, a, T, c0, kk, lane);
        else
          cm_solve_step<3>(acc, a, T, c0, kk, lane);
      }
    }
    rg.release(g);
  }
  __syncthreads();   // every warp has read its last stage: the in-place stores below cannot overtake a pending copy
#pragma unroll
  for (int fm = 0; fm < 4; ++fm)
#pragma unroll
    for (int fn = 0; fn < 4; ++fn) p_store_cfrag(blk, 4 * wm + fm, c0 + fn, lane, acc[fm][fn][0], acc[fm][fn][1]);
  fence_proxy_async();
  __syncthreads();
}

template <int KID>
__device__ __forceinline__ void cm_matrix(const PotrfParams &pp, const int s_mat, double *sm, CmPos &pos) {
  double *fv = sm + PT_TILES * 64 + PT_TMP_ELEMS + 128 + 128 + 8;
  uint64_t *bars = reinterpret_cast<uint64_t *>(fv + 136);
  double *etab = fv + 136 + PF_BAR_SLOTS, *invl = etab + EXPTAB_N;
  const int nblk = pp.nblk, tid = threadIdx.x;
  // per-matrix constants of the kernel-value generation (the diagonal step rewrites the same values)
  exptab_init(etab);
  if (tid >= 32 && tid < 64) {
    const int q = tid - 32;
    invl[q] = (q < pp.gen_d) ? 1.0 / (pp.gen_ls[(size_t)s_mat * pp.gen_d + q] + MIN_PARAM_VALUE) : 0.0;
  }
  const double amp = pp.gen_amp[s_mat] + MIN_PARAM_VALUE;
  const double a2 = amp * amp;
  __syncthreads();
#pragma unroll 1
  for (int j = 0; j < nblk; ++j) {
    // T_ij for the rows below the diagonal block (for j = 0 this is just K_i0): independent of the diagonal step
#pragma unroll 1
    for (int ih = 2 * (j + 1); ih < 2 * nblk; ++ih) cm_update_job<KID>(pp, s_mat, ih >> 1, j, ih & 1, sm, bars, pos.u, etab, invl, a2);
    fence_proxy_async();   // the tile store was written through the generic proxy; the SYRK ring reuses it
    __syncthreads();
    potrf_tile_body<true, true>(pp, s_mat, j, &pos.d);     // ends with a CTA-wide barrier; Winv_jj is in the tile store
#pragma unroll 1
    for (int ih = 2 * (j + 1); ih < 2 * nblk; ++ih) cm_solve_job(pp, s_mat, ih >> 1, j, 1 - (ih & 1), sm, bars, pos.s);   // half 1 first
  }
}

template <int KID>
__global__ void __launch_bounds__(256, 2) chol_matrix_kernel(const __grid_constant__ CmParams p) {
  extern __shared__ __align__(16) double sm[];
  {
    // all rings' barriers, once: SYRK ring full[6] empty[6] | update ring full[4] empty[4] | solve ring full[2] empty[2]
    uint64_t *bars = reinterpret_cast<uint64_t *>(sm + PT_TILES * 64 + PT_TMP_ELEMS + 128 + 128 + 8 + 136);
    const int t = threadIdx.x;
    if (t < PF_BAR_SLOTS) {
      const bool is_full = t < 6 || (t >= 12 && t < 16) || (t >= 20 && t < 22);
      mbar_init(smem_u32(&bars[t]), is_full ? 1u : 8u);
      mbar_fence_init();
    }
    __syncthreads();
  }
  CmPos pos{0, 0, 0};
  for (int s = blockIdx.x; s < (int)p.S; s += gridDim.x) {
    cm_matrix<KID>(p.pp, s, sm, pos);
    __syncthreads();
  }
}

}  // namespace boss

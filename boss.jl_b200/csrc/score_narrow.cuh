// score_narrow.cuh -- the triangular products of the scoring path for SMALL candidate batches: 32 candidates per CTA.
//
// score_trmm_kernel / wtv_kernel (score.cuh, grad.cuh) give a CTA 128 candidates; a batch of a few dozen points -- the
// unfinished starts of the multi-start optimiser after its first rounds, single-point calls of the reference's
// one-x-at-a-time access pattern -- then still pays 128-wide DMMA work on every stage of the longest row block
// (0.56 ms per pass at n = 4096, whatever the batch size).  Here a CTA owns 32 candidates: a stage is the same 16 KB
// tile of W plus a 4 KB slice of K*^T, the tensor work per stage is a quarter, and four times as many CTAs share the
// row blocks.  The two kernels produce THE SAME BITS as their wide twins: identical accumulation order inside a tile
// (k ascending, the same structurally-zero fragments skipped) and, for the column sums of squares, the wide kernel's
// reduction order is replayed explicitly (rows of one parity in fragment order, then the 3-level butterfly over the
// eight rows of a slab) -- a candidate scores identically alone, in a 1 000-start batch or in a 40 000-point grid
// (tests/test_gpu_parity.py::test_small_batch_split_is_bitwise_invariant).
#pragma once
#include "grad.cuh"
#include "score.cuh"

namespace boss {

constexpr int NW_NB = 32;                                   // candidates per CTA
constexpr int NW_STAGES = 6;
constexpr int NW_STAGE_ELEMS = TILE_ELEMS + TILE_ELEMS / 4;  // A: 128 x 16 tile of W (16 KB) + B: 32 x 16 slice (4 KB)
constexpr int NW_V_ELEMS = 128 * NW_NB;                      // one tile of V (or U) staged for the ordered reduction
constexpr int NW_SMEM_BYTES = (NW_STAGES * NW_STAGE_ELEMS + NW_V_ELEMS + 2 * 8 * NW_NB) * 8 + 2 * NW_STAGES * 8;

struct NarrowParams {
  const double *A;      // W (MODE 0, lower triangular) or W^T (MODE 1, upper triangular), P-layout
  const double *B;      // K*^T chunk (MODE 0) or V^T chunk (MODE 1): rows = candidates, P-layout blocks of 128
  int nblk, ktiles;
  double *ss_part;      // MODE 0: [2*nblk][ld] partial column sums of squares (same layout as score_trmm_kernel)
  int ld;
  double *OT;           // MODE 0: optional V^T chunk (gradient mode); MODE 1: U^T chunk
};

// MODE 0:  V = W K*  (row block i uses k-tiles 0 .. 8(i+1)-1, the last 8 are the lower-triangular diagonal block)
// MODE 1:  U = W^T V (row block i uses k-tiles 8i .. ktiles-1, the first 8 are the upper-triangular diagonal block)
// grid = (32-candidate blocks, row-block splits); row blocks are dealt in the same zig-zag order as the wide kernels.
template <int MODE>
__global__ void __launch_bounds__(256, 1) score_narrow_kernel(const __grid_constant__ NarrowParams p) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  double *ring = reinterpret_cast<double *>(smem_raw);
  double *Vst = ring + NW_STAGES * NW_STAGE_ELEMS;          // [16 slabs][8 rows][32 candidates]
  double *chn = Vst + NW_V_ELEMS;                           // [2 parities][8 rows][32 candidates]
  uint64_t *full = reinterpret_cast<uint64_t *>(chn + 2 * 8 * NW_NB), *empty = full + NW_STAGES;
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int cb32 = blockIdx.x, cb = cb32 >> 2, sub = cb32 & 3, y = blockIdx.y, ns2 = 2 * gridDim.y;
  if (tid < 2 * NW_STAGES) {
    mbar_init(smem_u32(tid < NW_STAGES ? &full[tid] : &empty[tid - NW_STAGES]), tid < NW_STAGES ? 1u : 8u);
    mbar_fence_init();
  }
  __syncthreads();

  // producer state (thread 0): the stream of (row block, k-tile) pairs of this CTA
  int pj = 0, pi = zigzag_row(0, y, ns2), pkt = MODE == 0 ? 0 : pi * KT_PER_BLOCK, issued = 0;
  const double *Bblk = p.B + (size_t)cb * p.ktiles * TILE_ELEMS + (size_t)sub * (TILE_ELEMS / 4);
  auto try_issue = [&](bool blocking) -> bool {
    const int slot = issued % NW_STAGES;
    if (issued >= NW_STAGES) {
      const uint32_t eb = smem_u32(&empty[slot]);
      const uint32_t par = (uint32_t)((issued / NW_STAGES - 1) & 1);
      if (blocking)
        mbar_wait(eb, par);
      else if (!mbar_try_wait(eb, par))
        return false;
    }
    const uint32_t bar = smem_u32(&full[slot]);
    double *dst = ring + (size_t)slot * NW_STAGE_ELEMS;
    mbar_arrive_expect_tx(bar, TILE_BYTES + TILE_BYTES / 4);
    bulk_g2s(smem_u32(dst), p.A + ((size_t)pi * p.ktiles + pkt) * TILE_ELEMS, TILE_BYTES, bar);
    bulk_g2s(smem_u32(dst + TILE_ELEMS), Bblk + (size_t)pkt * TILE_ELEMS, TILE_BYTES / 4, bar);
    ++issued;
    const int last = MODE == 0 ? (pi + 1) * KT_PER_BLOCK - 1 : p.ktiles - 1;
    if (pkt == last) {
      ++pj;
      pi = zigzag_row(pj, y, ns2);
      pkt = MODE == 0 ? 0 : pi * KT_PER_BLOCK;
    } else {
      ++pkt;
    }
    return true;
  };
  if (tid == 0)
    while (pi < p.nblk && issued < NW_STAGES) try_issue(false);

  const int R0 = 2 * w;   // this warp's row slabs R0, R0 + 1 of the current row block
  int g = 0;
  for (int j = 0;; ++j) {
    const int i = zigzag_row(j, y, ns2);
    if (i >= p.nblk) break;
    const int kt0 = MODE == 0 ? 0 : i * KT_PER_BLOCK, kt1 = MODE == 0 ? (i + 1) * KT_PER_BLOCK : p.ktiles;
    double acc[2][4][2];
#pragma unroll
    for (int fm = 0; fm < 2; ++fm)
#pragma unroll
      for (int fn = 0; fn < 4; ++fn) acc[fm][fn][0] = acc[fm][fn][1] = 0.0;
    for (int kt = kt0; kt < kt1; ++kt, ++g) {
      if (tid == 0) {
        while (pi < p.nblk && issued < g + NW_STAGES) {
          if (!try_issue(issued <= g)) break;
        }
      }
      const int slot = g % NW_STAGES;
      mbar_wait(smem_u32(&full[slot]), (uint32_t)((g / NW_STAGES) & 1));
      const double *As = ring + (size_t)slot * NW_STAGE_ELEMS + 2 * lane, *Bs = As + TILE_ELEMS;
      const int dg = kt - i * KT_PER_BLOCK;          // k-tile inside the diagonal block when 0 <= dg < 8
      const bool diag = dg >= 0 && dg < KT_PER_BLOCK;
#pragma unroll 1
      for (int mc = 0; mc < 2; ++mc) {
        // live row slabs (warp-uniform, real branches): lower block R >= kk, upper block R <= kk
        bool l0 = true, l1 = true;
        if (diag) {
          const int kk = 2 * dg + mc;
          l0 = MODE == 0 ? R0 >= kk : R0 <= kk;
          l1 = MODE == 0 ? R0 + 1 >= kk : R0 + 1 <= kk;
        }
        if (!(l0 || l1)) continue;
        double2 b[4];
#pragma unroll
        for (int fn = 0; fn < 4; ++fn) b[fn] = lds128(Bs + fn * 128 + mc * 64);
        if (l0) {
          const double2 a = lds128(As + R0 * 128 + mc * 64);
#pragma unroll
          for (int fn = 0; fn < 4; ++fn) dmma884(acc[0][fn][0], acc[0][fn][1], a.x, b[fn].x);
#pragma unroll
          for (int fn = 0; fn < 4; ++fn) dmma884(acc[0][fn][0], acc[0][fn][1], a.y, b[fn].y);
        }
        if (l1) {
          const double2 a = lds128(As + (R0 + 1) * 128 + mc * 64);
#pragma unroll
          for (int fn = 0; fn < 4; ++fn) dmma884(acc[1][fn][0], acc[1][fn][1], a.x, b[fn].x);
#pragma unroll
          for (int fn = 0; fn < 4; ++fn) dmma884(acc[1][fn][0], acc[1][fn][1], a.y, b[fn].y);
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(&empty[slot]));
    }
    // ---- tile (row block i) finished ----
    if (p.OT) {   // transposed store: rows = candidates (block cb, slabs 4 sub + fn), columns = row index of block i
      double *ot = p.OT + (size_t)cb * p.ktiles * TILE_ELEMS + (size_t)i * KT_PER_BLOCK * TILE_ELEMS;
#pragma unroll
      for (int fm = 0; fm < 2; ++fm)
#pragma unroll
        for (int fn = 0; fn < 4; ++fn) p_store_cfrag_t(ot, R0 + fm, 4 * sub + fn, lane, acc[fm][fn][0], acc[fm][fn][1]);
    }
    if (MODE == 0) {
      // column sums of squares in the wide kernel's order: for each parity pr of the row slab, the chain
      // v = fma(x, x, v) over the slabs R = pr, pr + 2, ..., pr + 14 (fixed row-in-slab r), then the butterfly over r
      const int r = lane >> 2, c2 = 2 * (lane & 3);
#pragma unroll
      for (int fm = 0; fm < 2; ++fm)
#pragma unroll
        for (int fn = 0; fn < 4; ++fn) {
          Vst[((R0 + fm) * 8 + r) * NW_NB + 8 * fn + c2] = acc[fm][fn][0];
          Vst[((R0 + fm) * 8 + r) * NW_NB + 8 * fn + c2 + 1] = acc[fm][fn][1];
        }
      __syncthreads();
      for (int e = tid; e < 2 * 8 * NW_NB; e += 256) {
        const int pr = e / (8 * NW_NB), rr = (e / NW_NB) & 7, cc = e % NW_NB;
        double v = 0.0;
#pragma unroll
        for (int fmw = 0; fmw < 8; ++fmw) {
          const double x = Vst[((2 * fmw + pr) * 8 + rr) * NW_NB + cc];
          v = fma(x, x, v);
        }
        chn[e] = v;
      }
      __syncthreads();
      if (tid < 2 * NW_NB) {
        const int pr = tid / NW_NB, cc = tid % NW_NB;
        const double *q = chn + pr * 8 * NW_NB + cc;
        const double s = ((q[0] + q[NW_NB]) + (q[2 * NW_NB] + q[3 * NW_NB])) + ((q[4 * NW_NB] + q[5 * NW_NB]) + (q[6 * NW_NB] + q[7 * NW_NB]));
        p.ss_part[(size_t)(2 * i + pr) * p.ld + (size_t)cb * 128 + 32 * sub + cc] = s;
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Quarter-row-block CTAs: built for TINY batches (a handful of unfinished multi-start runs, the reference's one-x-per-call
// access pattern) and, as it turned out, the fastest shape up to a few thousand candidates (its many short CTAs balance
// better than the row-split wide kernels: 10 % faster up to 8192 candidates at n = 2048; the cost model in score_slice decides).  With one 32-candidate block the kernels above expose only nblk CTAs and the longest of them walks
// all 8 nblk stages of the last row block alone: 218 us at n = 4096 whatever the batch holds.  Here a CTA owns 32 rows
// (4 row slabs) of one row block x 32 candidates (warp = 1 slab x 2 candidate slabs), 4 nblk CTAs per candidate block,
// launched longest first; the structurally dead head / tail k-tiles of a quarter are not even loaded.
// What bounds such a CTA is the rate at which ONE SM can pull its operands, and that is set by the number of
// requests, not bytes (measured, tools/bulk_copy_rate.cu -> profiles/r02_bulk_copy_rate.json): a TMA / mbarrier ring
// stage costs ~310 ns + 15 ns per 4 KB bulk copy whatever the ring depth or the source (L2 or HBM) -- 24 GB/s per SM
// with 8 KB stages, 75 GB/s with 32 KB stages; direct LDG.128 fragment loads four k-tiles ahead in registers reach
// ~28 GB/s (both tried here: 0.53 and 0.43 us per k-tile).  So a stage carries 4 k-tiles (8 bulk copies of
// 4 KB, 32 KB), issued by a dedicated producer warp, 3 stages in flight, two CTAs per SM.  (8 k-tiles per stage with one
// CTA per SM is as fast for a single 32-candidate block and 10-15 % slower from 256 candidates on; 2 k-tiles per stage
// with three CTAs per SM changes nothing: the SM's operand rate saturates.)
// Accumulation order inside a fragment is unchanged (k ascending, same fragments skipped), V^T is always stored, and
// quarter_sumsq_kernel replays the wide kernel's reduction over the stored tile -- THE SAME BITS again (DMMA.8x8x4
// itself accumulates k ascending like an FMA chain: tools/dmma_order_test.cu, profiles/r02_dmma_order.json).
// ---------------------------------------------------------------------------------------------
// The kernel is a template over the CTA tile: RS row slabs (of 8 rows) x NC 32-candidate slices.  <4, 1> is the quarter
// shape above and the only one instantiated: <8, 2> (64 rows x 64 candidates, half the operand bytes per output) was
// measured and is slower up to 512 candidates (n = 4096, 256 candidates: 519 vs 378 us per value + gradient call) --
// four times fewer CTAs with a four times longer DMMA chain each balance worse than the bytes they save.
constexpr int NQ_STAGES = 3;
constexpr int NQ_STAGE_ELEMS = 4096;                         // 32 KB per stage, whole k-tiles of [A part | B slices]
constexpr int NQ_SMEM_BYTES = NQ_STAGES * NQ_STAGE_ELEMS * 8 + 2 * NQ_STAGES * 8;
constexpr int NQ_THREADS = 288;                              // 8 consumer warps + 1 producer warp

// grid = (NC x 32-candidate blocks, (16 / RS) nblk): blockIdx.y = (16 / RS) * (rank of the row block, longest k-range
// first) + part of the row block
template <int MODE, int RS, int NC>
__global__ void __launch_bounds__(NQ_THREADS, 2) score_quarter_kernel(const __grid_constant__ NarrowParams p) {
  constexpr int PARTS = 16 / RS;                     // CTAs per row block
  constexpr int A_EL = RS * 128, B_EL = NC * 512;    // doubles per k-tile: RS row slabs of W, NC candidate slices of K*^T
  constexpr int KT_EL = A_EL + B_EL;
  constexpr int KT = NQ_STAGE_ELEMS / KT_EL;         // k-tiles per ring stage: 4 (quarter) or 2 (half)
  constexpr int SW = RS / 4, FW = 2 * NC;            // a warp: SW row slabs x FW candidate slabs
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  double *ring = reinterpret_cast<double *>(smem_raw);
  uint64_t *full = reinterpret_cast<uint64_t *>(ring + NQ_STAGES * NQ_STAGE_ELEMS), *empty = full + NQ_STAGES;
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int s32 = blockIdx.x * NC, cb = s32 >> 2, sub = s32 & 3, part = blockIdx.y % PARTS;
  const int i = MODE == 0 ? p.nblk - 1 - (int)(blockIdx.y / PARTS) : (int)(blockIdx.y / PARTS);
  // live k-tiles of the part: lower block (MODE 0) slab R sees k micro-steps kk <= R, R < RS (part + 1);
  // upper block (MODE 1) slab R sees kk >= R, R >= RS part
  const int kt0 = MODE == 0 ? 0 : i * KT_PER_BLOCK + (RS * part) / 2;
  const int kt1 = MODE == 0 ? i * KT_PER_BLOCK + (RS * part + RS) / 2 : p.ktiles;
  const int nk = kt1 - kt0, nst = (nk + KT - 1) / KT;
  if (tid < 2 * NQ_STAGES) {
    mbar_init(smem_u32(tid < NQ_STAGES ? &full[tid] : &empty[tid - NQ_STAGES]), tid < NQ_STAGES ? 1u : 8u);
    mbar_fence_init();
  }
  __syncthreads();
  if (w == 8) {   // producer warp: one lane streams the stages, blocking only on the slot it is about to refill
    if (lane == 0) {
      const double *Ablk = p.A + ((size_t)i * p.ktiles + kt0) * TILE_ELEMS + (size_t)part * A_EL;
      const double *Bblk = p.B + ((size_t)cb * p.ktiles + kt0) * TILE_ELEMS + (size_t)sub * 512;
      for (int s = 0; s < nst; ++s) {
        const int slot = s % NQ_STAGES;
        if (s >= NQ_STAGES) mbar_wait(smem_u32(&empty[slot]), (uint32_t)((s / NQ_STAGES - 1) & 1));
        const int cnt = min(KT, nk - s * KT);
        const uint32_t bar = smem_u32(&full[slot]);
        double *dst = ring + (size_t)slot * NQ_STAGE_ELEMS;
        mbar_arrive_expect_tx(bar, (uint32_t)(cnt * KT_EL * 8));
        for (int t = 0; t < cnt; ++t) {
          const size_t off = (size_t)(s * KT + t) * TILE_ELEMS;
          bulk_g2s(smem_u32(dst + (size_t)t * KT_EL), Ablk + off, A_EL * 8, bar);
          bulk_g2s(smem_u32(dst + (size_t)t * KT_EL + A_EL), Bblk + off, B_EL * 8, bar);
        }
      }
    }
    return;
  }
  const int sl0 = (w >> 1) * SW, R0 = RS * part + sl0, fn0 = FW * (w & 1);   // this warp: slabs R0.. x candidate slabs fn0..
  double acc[SW][FW][2];
#pragma unroll
  for (int a = 0; a < SW; ++a)
#pragma unroll
    for (int f = 0; f < FW; ++f) acc[a][f][0] = acc[a][f][1] = 0.0;
  for (int s = 0; s < nst; ++s) {
    const int slot = s % NQ_STAGES;
    mbar_wait(smem_u32(&full[slot]), (uint32_t)((s / NQ_STAGES) & 1));
    const int cnt = min(KT, nk - s * KT);
    const double *st = ring + (size_t)slot * NQ_STAGE_ELEMS + 2 * lane + sl0 * 128;
    const double *sb = ring + (size_t)slot * NQ_STAGE_ELEMS + 2 * lane + A_EL + fn0 * 128;
    const int dgs = kt0 + s * KT - i * KT_PER_BLOCK;   // k-tile t of the stage is k-tile dgs + t of the diagonal block (if in 0..7)
    // fragments: [mc][slab] of W, [mc][candidate slab] of K*^T
    auto fetch = [&](int t, double2(&fa)[2][SW], double2(&fb)[2][FW]) {
      const double *As = st + (size_t)t * KT_EL, *Bs = sb + (size_t)t * KT_EL;
#pragma unroll
      for (int mc = 0; mc < 2; ++mc) {
#pragma unroll
        for (int a = 0; a < SW; ++a) fa[mc][a] = lds128(As + a * 128 + mc * 64);
#pragma unroll
        for (int f = 0; f < FW; ++f) fb[mc][f] = lds128(Bs + f * 128 + mc * 64);
      }
    };
    auto mma = [&](int t, const double2(&fa)[2][SW], const double2(&fb)[2][FW]) {
      const int dg = dgs + t;
      const bool diag = dg >= 0 && dg < KT_PER_BLOCK;
#pragma unroll
      for (int mc = 0; mc < 2; ++mc) {
        const int kk = 2 * dg + mc;
#pragma unroll
        for (int a = 0; a < SW; ++a) {
          const bool live = !diag || (MODE == 0 ? R0 + a >= kk : R0 + a <= kk);   // warp-uniform
          if (live) {
#pragma unroll
            for (int f = 0; f < FW; ++f) dmma884(acc[a][f][0], acc[a][f][1], fa[mc][a].x, fb[mc][f].x);
#pragma unroll
            for (int f = 0; f < FW; ++f) dmma884(acc[a][f][0], acc[a][f][1], fa[mc][a].y, fb[mc][f].y);
          }
        }
      }
    };
    if constexpr (SW * FW <= 2) {
      // quarter shape: the fragments of k-tile t + 1 are fetched before the (short) DMMA chain of k-tile t starts
      double2 a0[2][SW], b0[2][FW], a1[2][SW], b1[2][FW];
      fetch(0, a0, b0);
#pragma unroll
      for (int t = 0; t < KT; t += 2) {
        if (t < cnt) {
          if (t + 1 < cnt) fetch(t + 1, a1, b1);
          mma(t, a0, b0);
        }
        if (t + 1 < cnt) {
          if (t + 2 < cnt) fetch(t + 2, a0, b0);
          mma(t + 1, a1, b1);
        }
      }
    } else {
      double2 a0[2][SW], b0[2][FW];
#pragma unroll
      for (int t = 0; t < KT; ++t)
        if (t < cnt) {
          fetch(t, a0, b0);
          mma(t, a0, b0);
        }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(smem_u32(&empty[slot]));
  }
  // transposed store: rows = candidates (block cb, slabs 4 sub + fn), columns = rows of block i
  double *ot = p.OT + (size_t)cb * p.ktiles * TILE_ELEMS + (size_t)i * KT_PER_BLOCK * TILE_ELEMS;
#pragma unroll
  for (int a = 0; a < SW; ++a)
#pragma unroll
    for (int f = 0; f < FW; ++f) p_store_cfrag_t(ot, R0 + a, 4 * sub + fn0 + f, lane, acc[a][f][0], acc[a][f][1]);
}

// Column sums of squares of the stored V^T in the wide kernel's order: per row block and slab parity the fma chain over
// the 8 slabs of the parity at a fixed row-in-slab r, then the 3-level butterfly over r; the partials land in ss_part
// exactly where score_trmm_kernel / score_narrow_kernel<0> put theirs (reduce_rows2_kernel folds them).
// grid = (32-candidate blocks, nblk), 256 threads = 32 candidates x 8 rows-in-slab.
__global__ void __launch_bounds__(256) quarter_sumsq_kernel(const double *__restrict__ VT, int ktiles, double *__restrict__ ss_part,
                                                            int ld) {
  const int r = threadIdx.x & 7, c = blockIdx.x * NW_NB + (threadIdx.x >> 3), i = blockIdx.y;
  const double *base = VT + (size_t)(c >> 7) * ktiles * TILE_ELEMS;
  const int cc = c & 127;
#pragma unroll
  for (int pr = 0; pr < 2; ++pr) {
    double x[8];
#pragma unroll
    for (int fmw = 0; fmw < 8; ++fmw) x[fmw] = base[p_index(cc, i * TM + (2 * fmw + pr) * 8 + r, ktiles)];
    double v = 0.0;
#pragma unroll
    for (int fmw = 0; fmw < 8; ++fmw) v = fma(x[fmw], x[fmw], v);
    v += __shfl_xor_sync(0xffffffffu, v, 1);
    v += __shfl_xor_sync(0xffffffffu, v, 2);
    v += __shfl_xor_sync(0xffffffffu, v, 4);
    if (r == 0) ss_part[(size_t)(2 * i + pr) * ld + c] = v;
  }
}

}  // namespace boss

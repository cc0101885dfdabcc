// tk_build.cu -- kernel-matrix construction (SURVEY.md 8 row a1) and the tile pass of the hyper-parameter gradient
// (row f2), instantiated for every (covariance function, padded input dimension).
#include "common.cuh"
#include "tk_params.cuh"

namespace boss {

// ---------------------------------------------------------------------------------------------
// K2: fused ARD kernel-matrix construction (lower block triangle, P-layout), per hyper-parameter sample
// Reference: finite_gp, src/models/gaussian_process.jl:216-248 (+1e-8 on every hyper-parameter, a^2 kappa, s^2 I).
// ---------------------------------------------------------------------------------------------
template <int KID, int DP>
__global__ void __launch_bounds__(256) build_k_kernel(BuildKParams p) {
  __shared__ double xcol[128 * DP];
  __shared__ double invl[DP];
  __shared__ double etab[EXPTAB_N];
  exptab_init(etab);
  const int s = blockIdx.y;
  // decode (rb >= cb) from the linear lower-triangle index
  int t = blockIdx.x, rb = 0;
  while (t >= rb + 1) {
    t -= rb + 1;
    ++rb;
  }
  const int cb = t;
  if (p.skip_diag && rb == cb) return;
  const int tid = threadIdx.x;
  if (tid < DP) {
    double l = (tid < p.d) ? p.ls[(size_t)s * p.d + tid] : 1.0;
    if (tid < p.d && !(l >= 0.0)) p.status[s] = -1;
    invl[tid] = (tid < p.d) ? 1.0 / (l + MIN_PARAM_VALUE) : 0.0;
  }
  __syncthreads();
  const double a_raw = p.amp[s], s_raw = p.noise[s];
  if (tid == 0 && (!(a_raw >= 0.0) || !(s_raw >= 0.0))) p.status[s] = -1;
  const double a = a_raw + MIN_PARAM_VALUE, sn = s_raw + MIN_PARAM_VALUE;
  const double a2 = a * a, s2 = sn * sn;

  // column points of this block -> smem (scaled)
  for (int e = tid; e < 128 * DP; e += 256) {
    const int jj = e / DP, i = e % DP;
    const int j = cb * 128 + jj;
    double v = 0.0;
    if (j < p.n && i < p.d) {
      v = p.X[(size_t)j * p.d + i];
      if ((p.disc_bits >> i) & 1ull) v = rint(v);
      v *= invl[i];
    }
    xcol[e] = v;
  }
  const int r = tid & 127, kh = tid >> 7;
  const int gi = rb * 128 + r;
  double xr[DP];
  load_scaled_point<DP>(xr, p.X + (size_t)gi * p.d, p.d, invl, p.disc_bits, gi < p.n);
  __syncthreads();

  double *blk = p.K + (size_t)s * p.K_stride + ((size_t)rb * p.ktiles + (size_t)cb * KT_PER_BLOCK) * TILE_ELEMS;
  for (int mcol = kh; mcol < 16; mcol += 2) {
    // diagonal blocks: micro-columns entirely above this row are never read (the factorisation only touches the
    // lower triangle) -> skip their exp / sqrt work
    if (rb == cb && mcol * 8 > r) continue;
    double v[8];
#pragma unroll
    for (int kk = 0; kk < 8; ++kk) {   // eight independent, branch-free chains: the scheduler interleaves them
      const int jj = mcol * 8 + kk;
      double d2 = 0.0;
#pragma unroll
      for (int i = 0; i < DP; ++i) {
        const double df = xr[i] - xcol[jj * DP + i];
        d2 = fma(df, df, d2);
      }
      v[kk] = a2 * kappa_fast<KID>(d2, etab, p.rq_a);
    }
    if (rb == cb || rb == p.nblk - 1) {   // diagonal tile (noise) or last row block (padding): per-element fix-up
#pragma unroll
      for (int kk = 0; kk < 8; ++kk) {
        const int gj = cb * 128 + mcol * 8 + kk;
        if (gi < p.n && gj < p.n) {
          if (gi == gj) v[kk] += s2;
        } else {
          v[kk] = (gi == gj) ? 1.0 : 0.0;  // identity padding: L_pad = I, log-det contribution 0
        }
      }
    }
    double *dst = blk + (mcol >> 1) * TILE_ELEMS + ((((r >> 3) << 1) + (mcol & 1)) << 6) + ((r & 7) << 3);
#pragma unroll
    for (int q = 0; q < 4; ++q) *reinterpret_cast<double2 *>(dst + 2 * q) = make_double2(v[q], v[q + 4]);
  }
}

// Per (lower tile, sample): partial sums  A1 = sum_{i>j} G_ij kappa_ij,  A2 = sum_i G_ii,  B_q = sum_{i>j} G_ij g_ij dq_ij^2
// with g = kappa'(r)/r and dq the scaled coordinate difference.  part[s][tile][DP + 2].
template <int KID, int DP>
__global__ void __launch_bounds__(256) loglik_grad_tile_kernel(LlGradParams p) {
  __shared__ double xcol[128 * DP];
  __shared__ double acol[128];
  __shared__ double invl[DP];
  __shared__ double red[256];
  __shared__ double etab[EXPTAB_N];
  exptab_init(etab);
  const int s = blockIdx.y, tid = threadIdx.x;
  int t = blockIdx.x, rb = 0;
  while (t >= rb + 1) {
    t -= rb + 1;
    ++rb;
  }
  const int cb = t;
  if (tid < DP) invl[tid] = (tid < p.d) ? 1.0 / (p.ls[(size_t)s * p.d + tid] + MIN_PARAM_VALUE) : 0.0;
  __syncthreads();
  const int n_pad = p.nblk * 128;
  const double *al = p.alpha + (size_t)s * n_pad;
  for (int e = tid; e < 128 * DP; e += 256) {
    const int jj = e / DP, i = e % DP, j = cb * 128 + jj;
    double v = 0.0;
    if (j < p.n && i < p.d) {
      v = p.X[(size_t)j * p.d + i];
      if ((p.disc_bits >> i) & 1ull) v = rint(v);
      v *= invl[i];
    }
    xcol[e] = v;
  }
  if (tid < 128) acol[tid] = al[cb * 128 + tid];
  const int r = tid & 127, kh = tid >> 7, gi = rb * 128 + r;
  double xr[DP];
  load_scaled_point<DP>(xr, p.X + (size_t)gi * p.d, p.d, invl, p.disc_bits, gi < p.n);
  const double ai = al[gi];
  __syncthreads();
  const double *blk = p.Kinv + (size_t)s * p.K_stride + ((size_t)rb * p.ktiles + (size_t)cb * KT_PER_BLOCK) * TILE_ELEMS;
  double a1 = 0.0, a2 = 0.0, bq[DP];
#pragma unroll
  for (int q = 0; q < DP; ++q) bq[q] = 0.0;
  for (int mcol = kh; mcol < 16; mcol += 2) {
    if (rb == cb && mcol * 8 > r) continue;
    const double *src = blk + (mcol >> 1) * TILE_ELEMS + ((((r >> 3) << 1) + (mcol & 1)) << 6) + ((r & 7) << 3);
    double kv[8];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const double2 v = *reinterpret_cast<const double2 *>(src + 2 * q);
      kv[q] = v.x;
      kv[q + 4] = v.y;
    }
    double kap[8], wgt[8];
#pragma unroll
    for (int kk = 0; kk < 8; ++kk) {   // independent, branch-free chains
      const int jj = mcol * 8 + kk;
      double d2 = 0.0;
#pragma unroll
      for (int q = 0; q < DP; ++q) {
        const double df = xr[q] - xcol[jj * DP + q];
        d2 = fma(df, df, d2);
      }
      kappa_and_dr_fast<KID>(d2, etab, p.rq_a, kap[kk], wgt[kk]);
    }
#pragma unroll
    for (int kk = 0; kk < 8; ++kk) {
      const int jj = mcol * 8 + kk, gj = cb * 128 + jj;
      const double G = ai * acol[jj] - kv[kk];
      const double Gd = (gi < p.n && gj == gi) ? G : 0.0;   // selects, not branches: adding 0.0 changes nothing
      const double Go = (gi < p.n && gj < gi) ? G : 0.0;
      a2 += Gd;
      a1 = fma(Go, kap[kk], a1);
      const double w = Go * wgt[kk];
#pragma unroll
      for (int q = 0; q < DP; ++q) {
        const double df = xr[q] - xcol[jj * DP + q];
        bq[q] = fma(w * df, df, bq[q]);
      }
    }
  }
  // block reductions in a fixed order, one quantity at a time
  double *out = p.part + ((size_t)s * gridDim.x + blockIdx.x) * (DP + 2);
#pragma unroll
  for (int q = 0; q < DP + 2; ++q) {
    const double v = (q < DP) ? bq[q < DP ? q : 0] : (q == DP ? a1 : a2);
    __syncthreads();
    red[tid] = v;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
      if (tid < o) red[tid] += red[tid + o];
      __syncthreads();
    }
    if (tid == 0) out[q] = red[0];
  }
}

bool launch_build_k(int kid, int dp, const BuildKParams &p, dim3 grid, cudaStream_t st) {
#define CALL(K, D) build_k_kernel<K, D><<<grid, 256, 0, st>>>(p)
  BOSS_DISPATCH_KID_DP(CALL, kid, dp)
#undef CALL
}
bool launch_loglik_grad_tile(int kid, int dp, const LlGradParams &p, dim3 grid, cudaStream_t st) {
#define CALL(K, D) loglik_grad_tile_kernel<K, D><<<grid, 256, 0, st>>>(p)
  BOSS_DISPATCH_KID_DP(CALL, kid, dp)
#undef CALL
}

}  // namespace boss

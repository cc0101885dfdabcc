// tk_score.cu -- the FP64-pipe kernels of the scoring path that evaluate the covariance function: cross-covariance
// K*^T + posterior mean (row a3), the finish of the full posterior covariance, and the kernel derivatives of the
// x-gradient (row g1); instantiated for every (covariance function, padded input dimension), the FP32 mean tier for
// KIDs 0-2 only.
#include "common.cuh"
#include "tk_params.cuh"

namespace boss {

// grid = (candidate blocks, splits over the 128-point training chunks).  Every chunk's contribution to
// mu is written as its own partial (fixed summation order downstream), so results do not depend on the split.
// STORE_KS = false: the mean partials only (argmax screening needs mu, not K*^T); same partials, same bits.
template <int KID, int DP, bool STORE_KS = true>
__global__ void __launch_bounds__(256) xcov_kernel(XcovParams p) {
  __shared__ double xt[XCOV_KC * DP];
  __shared__ double al[XCOV_KC];
  __shared__ double etab[EXPTAB_N];
  exptab_init(etab);
  const int tid = threadIdx.x, r = tid & 127, kh = tid >> 7;
  const int cb = blockIdx.x;
  const long long m = p.m0 + (long long)cb * 128 + r;
  double xc[DP];
  load_scaled_point<DP>(xc, p.Xs + (size_t)(m - p.in_off) * p.d, p.d, p.invl, p.disc_bits, m < p.M);

  double *rowbase = p.Ks + (size_t)cb * p.ktiles * TILE_ELEMS + (((r >> 3) << 1) << 6) + ((r & 7) << 3);
  for (int k0 = blockIdx.y * XCOV_KC; k0 < p.n_pad; k0 += gridDim.y * XCOV_KC) {
    double mu_acc = 0.0;
    __syncthreads();
    for (int e = tid; e < XCOV_KC * DP; e += 256) xt[e] = p.Xt[(size_t)k0 * DP + e];
    if (tid < XCOV_KC) al[tid] = p.alpha[k0 + tid];
    __syncthreads();
    // the last chunk may run past n: its padded columns must be exactly 0 (W is identity there)
    const int live = p.n - k0;
    for (int mcol = kh; mcol < XCOV_KC / 8; mcol += 2) {
      double v[8];
#pragma unroll
      for (int kk = 0; kk < 8; ++kk) {   // eight independent, branch-free chains: the scheduler interleaves them
        const int kl = mcol * 8 + kk;
        double d2 = 0.0;
#pragma unroll
        for (int i = 0; i < DP; ++i) {
          const double df = xc[i] - xt[kl * DP + i];
          d2 = fma(df, df, d2);
        }
        v[kk] = p.a2 * kappa_fast<KID>(d2, etab, p.rq_a);
      }
      if (live < XCOV_KC) {
#pragma unroll
        for (int kk = 0; kk < 8; ++kk) v[kk] = (mcol * 8 + kk < live) ? v[kk] : 0.0;
      }
#pragma unroll
      for (int kk = 0; kk < 8; ++kk) mu_acc = fma(v[kk], al[mcol * 8 + kk], mu_acc);
      if (!STORE_KS) continue;
      const int kg = k0 + mcol * 8;  // global training index of v[0]
      double *dst = rowbase + (size_t)(kg >> 4) * TILE_ELEMS + (((kg >> 3) & 1) << 6);
#pragma unroll
      for (int q = 0; q < 4; ++q) *reinterpret_cast<double2 *>(dst + 2 * q) = make_double2(v[q], v[q + 4]);
    }
    p.mu_part[(size_t)(2 * (k0 / XCOV_KC) + kh) * p.ld + (size_t)cb * 128 + r] = mu_acc;
  }
}

// D += A B for one m16n8k8 tile: A (16 x 8, row-major) and B (8 x 8, column-major) in TF32, D in FP32
__device__ __forceinline__ void mma_tf32(float (&d)[4], const unsigned (&a)[4], unsigned b0, unsigned b1) {
  asm("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, "
      "{%0, %1, %2, %3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// 16-byte asynchronous copy global -> shared (L2 only), and the waits on its commit groups
__device__ __forceinline__ void cp_async16(void *dst, const void *src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// The FP32 mean tier of argmax screening (DESIGN.md 2.9), one CTA per 128 candidates over every training point of
// every slice, then the bound verdicts of those candidates.
//
// Means: d2 = |u~|^2 + |t~_j|^2 - 2 u~.t~_j from centred FP32 points.  The cross term runs on the tensor cores
// (mma.sync TF32, 3-term hi / lo split, accumulated in FP32); the norms are added and kappa_f32x2 evaluated on the
// accumulator fragments, training points 2t and 2t + 1 as the two lanes of the packed FP32 instructions.  Warp w takes candidates 16w..16w+15 against the 16 eight-point tiles of each 128-point stage of
// training points.  A thread holds candidates g and g + 8 (g = lane / 4) against training points 2t, 2t + 1 of each tile
// (t = lane % 4); each run of 4 tiles (8 points per candidate) is summed in FP32 and added to an FP64 accumulator, the
// four lanes of a candidate are combined by a fixed butterfly, and the stage's two halves (tiles 0-7, 8-15) are scaled
// by a^2 and added to mu~ in ascending (stage, half) order.  So mu~ does not depend on scheduling, and equals the
// ordered sum of per-(stage, half) partials that reduce_rows_kernel forms on the FP64 tier.  A stage's B fragments and
// (|t~|^2, alpha) are copied into a 2-deep ring while the previous stage computes.
//
// Verdicts, one thread per candidate: per slice mu~ +- E', E' = E with the sign of the slice's output coefficient (NaN
// for both if mu~ or E is not finite), so that EI is at least as large at mu~ + E' as at the FP64 mean and no larger at
// mu~ - E'; the EI bound at each (acq_candidate under p.hi and p.lo, into hi.acq and lo.acq); and, unless p.cnt is
// null, the CTA's survivors, !(hi < p.thr), to p.cnt[blockIdx.x].  With p.mu_out set the CTA writes mu~ and E to
// p.mu_out / p.e_out instead.
template <int KID, int DP>
__global__ void __launch_bounds__(256) screen_mean_bound_kernel(ScreenF32Params p) {
  constexpr int KS = (DP + 7) / 8, KP = 8 * KS;       // k-steps of the MMA, the padded dimension
  constexpr int NF = XCOV_KC / 8 * KS * 32, NS = NF + XCOV_KC / 2;   // float4 of one stage: B fragments, (|t~|^2, alpha)
  extern __shared__ float4 ring[];                     // [2][NS]; then mu~ and E, [nsl][128] each
  double *smu = reinterpret_cast<double *>(ring + 2 * NS), *se = smu + p.nsl * 128;
  __shared__ float snu[128];
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5, g = lane >> 2, t = lane & 3;
  const long long mb = p.m0 + (long long)blockIdx.x * 128;   // the CTA's first candidate
  for (int q = 0; q < p.nsl; ++q) {
    const ScreenSlice &sl = p.sl[q];
    const int nst = sl.n_pad / XCOV_KC;
    auto stage = [&](int st) {   // stage st of the slice into ring slot st & 1, one commit group
      float4 *dst = ring + (st & 1) * NS;
      const float4 *tf = sl.tfrag + (size_t)st * NF, *ta = sl.tn_al + (size_t)st * (XCOV_KC / 2);
      for (int e = tid; e < NS; e += 256) cp_async16(dst + e, e < NF ? tf + e : ta + (e - NF));
      cp_async_commit();
    };
    stage(0);
    if (tid < 128) {   // the candidates' -2 u~ (hi, lo; [128][KP] each) in slot 1, |u~|^2, E
      const long long m = mb + tid;
      double x64[DP];
      load_scaled_point<DP>(x64, p.Xs + (size_t)(m - p.in_off) * p.d, p.d, sl.invl, sl.disc_bits, m < p.M);
      double n2 = 0.0;
#pragma unroll
      for (int i = 0; i < DP; ++i) {
        x64[i] -= sl.A[2 + i];
        n2 = fma(x64[i], x64[i], n2);
      }
      float *ua = reinterpret_cast<float *>(ring + NS);
#pragma unroll
      for (int i = 0; i < KP; ++i) {
        float hi, lo;
        tf32_split(i < DP ? (float)x64[i] : 0.0f, hi, lo);
        ua[tid * KP + i] = -2.0f * hi;
        ua[128 * KP + tid * KP + i] = -2.0f * lo;
      }
      snu[tid] = (float)n2;
      se[q * 128 + tid] =
          sl.a2 * 0x1p-24 * (SCREEN_C_EVAL * sl.A[0] + screen_l2(KID) * screen_k_dot(DP) * fma(n2, sl.A[0], sl.A[1]));
    }
    __syncthreads();
    unsigned ahi[KS][4], alo[KS][4];
    {
      const float *ua = reinterpret_cast<const float *>(ring + NS);
      const int r0 = 16 * w + g;
#pragma unroll
      for (int ks = 0; ks < KS; ++ks)
#pragma unroll
        for (int e = 0; e < 4; ++e) {   // a0: (g, t), a1: (g + 8, t), a2: (g, t + 4), a3: (g + 8, t + 4)
          const int o = (r0 + 8 * (e & 1)) * KP + ks * 8 + t + 4 * (e >> 1);
          ahi[ks][e] = __float_as_uint(ua[o]);
          alo[ks][e] = __float_as_uint(ua[128 * KP + o]);
        }
    }
    const float2 nu0 = f2(snu[16 * w + g]), nu1 = f2(snu[16 * w + g + 8]);
    double mu0 = 0.0, mu1 = 0.0;   // candidates g and g + 8
    for (int st = 0; st < nst; ++st) {
      __syncthreads();   // slot (st + 1) & 1 is no longer read (stage st - 1, or the candidates' fragments)
      if (st + 1 < nst) stage(st + 1);
      else cp_async_commit();
      cp_async_wait<1>();
      __syncthreads();   // stage st has landed for every thread's copies
      const float4 *sbuf = ring + (st & 1) * NS, *snt = sbuf + NF;
#pragma unroll
      for (int kh = 0; kh < 2; ++kh) {
        double acc0 = 0.0, acc1 = 0.0;
#pragma unroll
        for (int run = 0; run < 2; ++run) {
          float2 s0 = f2(0.0f), s1 = f2(0.0f);   // points 2t and 2t + 1 of the run's tiles, summed apart
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const int nt = kh * 8 + run * 4 + u;
            float c[4] = {0.0f, 0.0f, 0.0f, 0.0f};
#pragma unroll
            for (int ks = 0; ks < KS; ++ks) {   // b = (b0 hi, b1 hi, b0 lo, b1 lo): B(t, g), B(t + 4, g)
              const float4 b = sbuf[(nt * KS + ks) * 32 + lane];
              mma_tf32(c, alo[ks], __float_as_uint(b.x), __float_as_uint(b.y));
              mma_tf32(c, ahi[ks], __float_as_uint(b.z), __float_as_uint(b.w));
              mma_tf32(c, ahi[ks], __float_as_uint(b.x), __float_as_uint(b.y));
            }
            const float4 na = snt[nt * 4 + t];   // points 2t, 2t + 1 of the tile
            const float2 tn = make_float2(na.x, na.y), al = make_float2(na.z, na.w);
            float2 d0 = __fadd2_rn(__fadd2_rn(make_float2(c[0], c[1]), nu0), tn);
            float2 d1 = __fadd2_rn(__fadd2_rn(make_float2(c[2], c[3]), nu1), tn);
            d0 = make_float2(fmaxf(d0.x, 1e-30f), fmaxf(d0.y, 1e-30f));
            d1 = make_float2(fmaxf(d1.x, 1e-30f), fmaxf(d1.y, 1e-30f));
            s0 = __ffma2_rn(al, kappa_f32x2<KID>(d0), s0);
            s1 = __ffma2_rn(al, kappa_f32x2<KID>(d1), s1);
          }
          acc0 += (double)(s0.x + s0.y);
          acc1 += (double)(s1.x + s1.y);
        }
        acc0 += __shfl_xor_sync(0xffffffffu, acc0, 1);
        acc1 += __shfl_xor_sync(0xffffffffu, acc1, 1);
        acc0 += __shfl_xor_sync(0xffffffffu, acc0, 2);
        acc1 += __shfl_xor_sync(0xffffffffu, acc1, 2);
        // the partial a^2 acc is rounded before it is added (no fused multiply-add), as in the ordered sum
        mu0 = __dadd_rn(mu0, __dmul_rn(sl.a2, acc0));
        mu1 = __dadd_rn(mu1, __dmul_rn(sl.a2, acc1));
      }
    }
    if (t == 0) {
      smu[q * 128 + 16 * w + g] = mu0;
      smu[q * 128 + 16 * w + g + 8] = mu1;
    }
    __syncthreads();   // mu~ complete; the ring and snu are free for the next slice
  }
  const long long m = mb + tid;
  if (p.mu_out) {
    if (tid < 128 && m < p.M)
      for (int q = 0; q < p.nsl; ++q) {
        p.mu_out[(size_t)q * p.ld + (m - p.m0)] = smu[q * 128 + tid];
        p.e_out[(size_t)q * p.ld + (m - p.m0)] = se[q * 128 + tid];
      }
    return;
  }
  bool keep = false;
  if (tid < 128 && m < p.M) {
    for (int q = 0; q < p.nsl; ++q) {   // smu <- mu~ + E', se <- mu~ - E'
      const double mq = smu[q * 128 + tid], E = p.hi.coefs[q % p.hi.y_dim] < 0.0 ? -se[q * 128 + tid] : se[q * 128 + tid];
      const bool ok = isfinite(mq) && isfinite(E);
      smu[q * 128 + tid] = ok ? mq + E : NAN;
      se[q * 128 + tid] = ok ? mq - E : NAN;
    }
    keep = !(acq_candidate<true>(p.hi, 0, m, smu + tid, 128) < p.thr);
    acq_candidate<true>(p.lo, 0, m, se + tid, 128);
  }
  if (!p.cnt) return;
  const int k = __syncthreads_count(keep);
  if (tid == 0) p.cnt[blockIdx.x] = k;
}

// The tensor-core d2 of screen_mean_bound_kernel for given FP32 points, for the tests of its error model: u [16 gridDim.x]
// [8 KS] and t [8 gridDim.y][8 KS] row-major, nu / nt their norms; one warp per 16 x 8 tile, the same split, MMA chain
// and assembly (without the clamp at 0), d2 [16 gridDim.x][8 gridDim.y] row-major.
template <int KS>
__global__ void mma_d2_kernel(const float *u, const float *t, const float *nu, const float *nt, float *d2) {
  const int lane = threadIdx.x, g = lane >> 2, tq = lane & 3, KP = 8 * KS;
  const int r0 = blockIdx.x * 16 + g, j = blockIdx.y * 8 + g, N = gridDim.y * 8;
  float c[4] = {0.0f, 0.0f, 0.0f, 0.0f};
  for (int ks = 0; ks < KS; ++ks) {
    unsigned ahi[4], alo[4], bhi[2], blo[2];
    for (int e = 0; e < 4; ++e) {
      float hi, lo;
      tf32_split(u[(size_t)(r0 + 8 * (e & 1)) * KP + ks * 8 + tq + 4 * (e >> 1)], hi, lo);
      ahi[e] = __float_as_uint(-2.0f * hi);
      alo[e] = __float_as_uint(-2.0f * lo);
    }
    for (int e = 0; e < 2; ++e) {
      float hi, lo;
      tf32_split(t[(size_t)j * KP + ks * 8 + tq + 4 * e], hi, lo);
      bhi[e] = __float_as_uint(hi);
      blo[e] = __float_as_uint(lo);
    }
    mma_tf32(c, alo, bhi[0], bhi[1]);
    mma_tf32(c, ahi, blo[0], blo[1]);
    mma_tf32(c, ahi, bhi[0], bhi[1]);
  }
  const int row = blockIdx.x * 16 + g, col = blockIdx.y * 8 + 2 * tq;
  for (int e = 0; e < 4; ++e) {
    const int rr = row + 8 * (e >> 1), cc = col + (e & 1);
    d2[(size_t)rr * N + cc] = c[e] + nu[rr] + nt[cc];
  }
}

bool launch_mma_d2(int dp, const float *u, const float *t, const float *nu, const float *nt, int mt, int nt_, float *d2,
                   cudaStream_t st) {
  const dim3 grid(mt, nt_);
  switch ((dp + 7) / 8) {
    case 1: mma_d2_kernel<1><<<grid, 32, 0, st>>>(u, t, nu, nt, d2); return true;
    case 2: mma_d2_kernel<2><<<grid, 32, 0, st>>>(u, t, nu, nt, d2); return true;
    case 4: mma_d2_kernel<4><<<grid, 32, 0, st>>>(u, t, nu, nt, d2); return true;
    default: return false;
  }
}

// The FP32 tier's kappa_f32x2 at d2 = max(fp32(r^2), 1e-30), as the tier clamps it, for the error-bound sweep of the
// tests: thread i evaluates distances 2i and 2i + 1 as the two lanes
template <int KID>
__global__ void kappa_f32_sweep_kernel(const double *r, int n, double *out) {
  const int i = 2 * (blockIdx.x * blockDim.x + threadIdx.x);
  if (i >= n) return;
  const double r1 = i + 1 < n ? r[i + 1] : 0.0;
  const float2 k = kappa_f32x2<KID>(make_float2(fmaxf((float)(r[i] * r[i]), 1e-30f), fmaxf((float)(r1 * r1), 1e-30f)));
  out[i] = (double)k.x;
  if (i + 1 < n) out[i + 1] = (double)k.y;
}

// full posterior covariance of a small candidate batch (cov / mean_and_cov, gaussian_process.jl:163-167,180-184)
//   cov[i][j] = k(x*_i, x*_j) - (V^T V)[i][j] + 1e-18 [i == j],   diagonal through _clip_var
template <int KID, int DP>
__global__ void __launch_bounds__(256) cov_finish_kernel(CovFinishParams p) {
  __shared__ double etab[EXPTAB_N];
  exptab_init(etab);
  __syncthreads();
  const int i = blockIdx.x * 16 + (threadIdx.x & 15), j = blockIdx.y * 16 + (threadIdx.x >> 4);
  if (i >= p.M || j >= p.M) return;
  double xi[DP], xj[DP];
  load_scaled_point<DP>(xi, p.Xs + (size_t)i * p.d, p.d, p.invl, p.disc_bits, true);
  load_scaled_point<DP>(xj, p.Xs + (size_t)j * p.d, p.d, p.invl, p.disc_bits, true);
  double d2 = 0.0;
#pragma unroll
  for (int q = 0; q < DP; ++q) {
    const double df = xi[q] - xj[q];
    d2 = fma(df, df, d2);
  }
  const int hi = max(i, j), lo = min(i, j);
  double v = p.a2 * kappa_fast<KID>(d2, etab, p.rq_a) - p.C[p_index(hi, lo, p.ktilesC)];
  if (i == j) {
    v += VAR_JITTER;
    if (!clip_var(v)) *p.any_fail = 1;
    if (p.mu_out) p.mu_out[i] = p.prior_mean ? p.prior_mean[i] + p.mu[i] : p.mu[i];
  }
  p.cov[(size_t)j * p.M + i] = v;
}

// d mu / dx and d var / dx for one slice and one chunk (see grad.cuh).
template <int KID, int DP>
__global__ void __launch_bounds__(256) grad_kernel(GradParams p) {
  __shared__ double xt[XCOV_KC * DP];
  __shared__ double al[XCOV_KC];
  __shared__ double etab[EXPTAB_N];
  exptab_init(etab);
  const int tid = threadIdx.x, r = tid & 127, kh = tid >> 7;
  const int cb = blockIdx.x;
  const long long m = p.m0 + (long long)cb * 128 + r;
  double xc[DP];
  load_scaled_point<DP>(xc, p.Xs + (size_t)(m - p.in_off) * p.d, p.d, p.invl, p.disc_bits, m < p.M);
  const double *rowbase = p.UT + (size_t)cb * p.ktiles * TILE_ELEMS + (((r >> 3) << 1) << 6) + ((r & 7) << 3);
  for (int k0 = blockIdx.y * XCOV_KC; k0 < p.n_pad; k0 += gridDim.y * XCOV_KC) {
    double gm[DP], gv[DP];
#pragma unroll
    for (int i = 0; i < DP; ++i) gm[i] = gv[i] = 0.0;
    __syncthreads();
    for (int e = tid; e < XCOV_KC * DP; e += 256) xt[e] = p.Xt[(size_t)k0 * DP + e];
    if (tid < XCOV_KC) al[tid] = p.alpha[k0 + tid];
    __syncthreads();
    for (int mcol = kh; mcol < XCOV_KC / 8; mcol += 2) {
      const int kg = k0 + mcol * 8;
      const double *src = rowbase + (size_t)(kg >> 4) * TILE_ELEMS + (((kg >> 3) & 1) << 6);
      double u[8];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const double2 v = *reinterpret_cast<const double2 *>(src + 2 * q);
        u[q] = v.x;
        u[q + 4] = v.y;
      }
      double gk[8];
#pragma unroll
      for (int kk = 0; kk < 8; ++kk) {   // independent, branch-free chains
        const int kl = mcol * 8 + kk;
        double d2 = 0.0;
#pragma unroll
        for (int i = 0; i < DP; ++i) {
          const double df = xc[i] - xt[kl * DP + i];
          d2 = fma(df, df, d2);
        }
        gk[kk] = p.a2 * kappa_dr_over_r_fast<KID>(d2, etab, p.rq_a);
      }
      if (p.n - k0 < XCOV_KC) {
#pragma unroll
        for (int kk = 0; kk < 8; ++kk) gk[kk] = (k0 + mcol * 8 + kk < p.n) ? gk[kk] : 0.0;
      }
#pragma unroll
      for (int kk = 0; kk < 8; ++kk) {
        const int kl = mcol * 8 + kk;
        const double t1 = gk[kk] * al[kl], t2 = gk[kk] * u[kk];
#pragma unroll
        for (int i = 0; i < DP; ++i) {
          const double df = xc[i] - xt[kl * DP + i];
          gm[i] = fma(t1, df, gm[i]);
          gv[i] = fma(t2, df, gv[i]);
        }
      }
    }
    const size_t prow = (size_t)(2 * (k0 / XCOV_KC) + kh) * p.d;
#pragma unroll
    for (int i = 0; i < DP; ++i) {
      if (i < p.d) {
        p.gm_part[(prow + i) * p.chunk_ld + cb * 128 + r] = gm[i];
        p.gv_part[(prow + i) * p.chunk_ld + cb * 128 + r] = gv[i];
      }
    }
  }
}

bool launch_xcov(int kid, int dp, const XcovParams &p, dim3 grid, cudaStream_t st) {
#define CALL(K, D) xcov_kernel<K, D><<<grid, 256, 0, st>>>(p)
  BOSS_DISPATCH_KID_DP(CALL, kid, dp)
#undef CALL
}
bool launch_xcov_mean(int kid, int dp, const XcovParams &p, dim3 grid, cudaStream_t st) {
#define CALL(K, D) xcov_kernel<K, D, false><<<grid, 256, 0, st>>>(p)
  BOSS_DISPATCH_KID_DP(CALL, kid, dp)
#undef CALL
}
size_t screen_mean_bound_smem(int dp, int nsl) {
  return (size_t)2 * (XCOV_KC / 8 * ((dp + 7) / 8) * 32 + XCOV_KC / 2) * 16 + (size_t)nsl * 2 * 128 * 8;
}
bool launch_screen_mean_bound(int kid, int dp, const ScreenF32Params &p, int nblocks, cudaStream_t st) {
  const size_t smem = screen_mean_bound_smem(dp, p.nsl);
#define CALL(K, D)                                                                                                 \
  do {                                                                                                             \
    cudaFuncSetAttribute(screen_mean_bound_kernel<K, D>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
    screen_mean_bound_kernel<K, D><<<nblocks, 256, smem, st>>>(p);                                               \
  } while (0)
  BOSS_DISPATCH_KID_DP_F32(CALL, kid, dp)
#undef CALL
}
bool launch_kappa_f32_sweep(int kid, const double *r, int n, double *out, cudaStream_t st) {
  const int nb = (n + 511) / 512;
  if (n < 1) return true;
  if (kid == 0) kappa_f32_sweep_kernel<0><<<nb, 256, 0, st>>>(r, n, out);
  else if (kid == 1) kappa_f32_sweep_kernel<1><<<nb, 256, 0, st>>>(r, n, out);
  else if (kid == 2) kappa_f32_sweep_kernel<2><<<nb, 256, 0, st>>>(r, n, out);
  else return false;
  return true;
}
bool launch_cov_finish(int kid, int dp, const CovFinishParams &p, dim3 grid, cudaStream_t st) {
#define CALL(K, D) cov_finish_kernel<K, D><<<grid, 256, 0, st>>>(p)
  BOSS_DISPATCH_KID_DP(CALL, kid, dp)
#undef CALL
}
bool launch_grad(int kid, int dp, const GradParams &p, dim3 grid, cudaStream_t st) {
#define CALL(K, D) grad_kernel<K, D><<<grid, 256, 0, st>>>(p)
  BOSS_DISPATCH_KID_DP(CALL, kid, dp)
#undef CALL
}

}  // namespace boss

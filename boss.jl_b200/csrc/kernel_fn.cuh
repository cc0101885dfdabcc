// kernel_fn.cuh -- covariance function evaluation shared by the kernel-matrix builder (a1) and the
// cross-covariance generator (a3).  Mirrors KernelFunctions' kappa for SqExponential / Matern32 /
// Matern52 / Exponential (Matern12) / RationalQuadratic composed with ARDTransform(1/l) and ScaledKernel(a^2)  (reference call site:
// src/models/gaussian_process.jl:243), optional DiscreteKernel rounding (src/models/utils/kernels.jl:56-64).
#pragma once
#include "common.cuh"

namespace boss {

constexpr double MIN_PARAM_VALUE = 1e-8;  // src/models/gaussian_process.jl:5
constexpr double MAX_NEG_VAR = 1e-8;      // src/models/gaussian_process.jl:13
constexpr double VAR_JITTER = 1e-18;      // AbstractGPs default FiniteGP observation noise

#ifdef __CUDACC__
// exp(-t) for t >= 0 with a 32-entry table of 2^(j/32) in shared memory and a degree-6 polynomial on
// |r| <= ln2/64: 11 FP64 instructions instead of libm's ~17 and no branches, so the eight independent elements
// a thread evaluates per pass interleave (the FP64 pipe is shared with the DMMA kernels: every instruction
// counts).  Relative error < 4e-16 (measured, tests/test_gpu_parity.py::test_fast_kernel_fn).  t >= 700 and
// t = +Inf return 0 (the true value is below 1e-304), NaN returns NaN; the range test is one integer compare on
// the high word (valid because t >= 0), and whatever the polynomial computed from an out-of-range t is discarded.
constexpr int EXPTAB_N = 32;
__device__ __forceinline__ void exptab_init(double *tab) {   // call with all threads, then __syncthreads()
  if (threadIdx.x < EXPTAB_N) tab[threadIdx.x] = exp2((double)threadIdx.x * (1.0 / EXPTAB_N));
}
__device__ __forceinline__ double fast_exp_neg(double t, const double *tab) {
  const double MAGIC = 6755399441055744.0;                    // 1.5 * 2^52: rounds to nearest integer in the low bits
  const double kf = fma(t, -46.16624130844682903551758979206054839765 /* -32/ln2 */, MAGIC);
  const int ki = __double2loint(kf);
  const double kd = kf - MAGIC;
  double r = fma(kd, -0.021660849392446835 /* ln2/32, top 38 bits: kd * hi is exact */, -t);
  r = fma(kd, -5.145609244655338e-14 /* ln2/32 - hi */, r);
  double p = fma(r, 1.0 / 720.0, 1.0 / 120.0);
  p = fma(p, r, 1.0 / 24.0);
  p = fma(p, r, 1.0 / 6.0);
  p = fma(p, r, 0.5);
  p = fma(p, r, 1.0);
  p = fma(p, r, 1.0);
  const double v = tab[ki & (EXPTAB_N - 1)] * p;
  // scale by 2^(ki >> 5): exponent-field add (v in [1, 2.1), result >= 2^-1010 stays normal)
  const int thi = __double2hiint(t), vhi = __double2hiint(v) + ((ki >> 5) << 20), vlo = __double2loint(v);
  int hi, lo;   // big = t >= 700, +Inf or NaN -> 0, 0, NaN; written as selects so that no branch splits the chain
  asm("{\n\t.reg .pred big, nan;\n\t.reg .b32 alt;\n\t"
      "setp.ge.s32 big, %2, 0x4085E000;\n\t"
      "setp.gt.s32 nan, %2, 0x7FF00000;\n\t"
      "selp.b32 alt, %2, 0, nan;\n\t"
      "selp.b32 %0, alt, %3, big;\n\t"
      "selp.b32 %1, 0, %4, big;\n\t}"
      : "=r"(hi), "=r"(lo)
      : "r"(thi), "r"(vhi), "r"(vlo));
  return __hiloint2double(hi, lo);
}

// sqrt(x) for x >= 0: MUFU.RSQ64H seed (~2^-22), one coupled Goldschmidt step and one residual correction:
// 8 FP64 instructions instead of libm's 19, no branches.  Error <= 1 ulp for x >= 1e-270 (measured,
// test_fast_kernel_fn); the seed needs a normal, non-zero input, so 1e-290 is added first: x = 0 returns 1e-145,
// which every caller multiplies into exp(-t) ~ 1.  NaN -> NaN, +Inf -> NaN (callers: kappa(Inf) is Inf * 0 in the
// reference's Matern kernels too).
__device__ __forceinline__ double fast_sqrt(double x) {
  x += 1e-290;
  double y;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
  double g = x * y, h = 0.5 * y;
  const double r = fma(-g, h, 0.5);
  g = fma(g, r, g);
  h = fma(h, r, h);
  return fma(fma(-g, g, x), h, g);
}

// 1/sqrt(x) for x >= 0: MUFU.RSQ64H seed (~2^-22) and two Newton steps, a few ulp for every normal x.  The seed flushes
// subnormals, so x is raised to the smallest normal double first: x = 0 returns 6.7e153 (the one caller selects 0 there).
__device__ __forceinline__ double fast_rsqrt(double x) {
  x = fmax(x, 2.2250738585072014e-308);
  double y;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
  const double h = 0.5 * x;
  y = y * fma(-h * y, y, 1.5);
  return y * fma(-h * y, y, 1.5);
}

// log1p(u) for u >= 0 without branches (libm's log1p inlines a slow path that, eight chains wide, costs the tile kernels
// their registers): w = 1 + u = 2^k m with m in [sqrt(1/2), sqrt(2)), log m = 2 atanh(s), s = (m - 1) / (m + 1), |s| <=
// 0.172, by an odd series through s^21; the reciprocals are MUFU.RCP64H seeds refined by Newton steps, and the
// rounding of 1 + u is put back as -((w - 1) - u) / w.  A few ulp (measured against mpmath,
// tests/test_gpu_kernels_more.py::test_kernel_functions).  Finite u only.
__device__ __forceinline__ double rcp_newton(double x, int steps) {
  double y;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
  for (int i = 0; i < steps; ++i) y = fma(y, fma(-x, y, 1.0), y);
  return y;
}
__device__ __forceinline__ double fast_log1p(double u) {
  const double w = 1.0 + u, c = (w - 1.0) - u;
  const int hi = __double2hiint(w);
  const int k = ((hi + (0x3FF00000 - 0x3FE6A09E)) >> 20) - 1023;
  const double m = __hiloint2double(hi - (k << 20), __double2loint(w));
  const double f = m - 1.0, q = 2.0 + f;
  const double rq = rcp_newton(q, 2);
  double sv = f * rq;
  sv = fma(fma(-sv, q, f), rq, sv);
  const double z = sv * sv;
  double p = fma(z, 1.0 / 21.0, 1.0 / 19.0);
  p = fma(p, z, 1.0 / 17.0);
  p = fma(p, z, 1.0 / 15.0);
  p = fma(p, z, 1.0 / 13.0);
  p = fma(p, z, 1.0 / 11.0);
  p = fma(p, z, 1.0 / 9.0);
  p = fma(p, z, 1.0 / 7.0);
  p = fma(p, z, 1.0 / 5.0);
  p = fma(p, z, 1.0 / 3.0);
  const double s2 = 2.0 * sv, lm = fma(s2 * z, p, s2);
  const double kd = (double)k;
  const double corr = fma(kd, 1.9082149292705877e-10 /* ln2 - ln2_hi */, lm) - c * rcp_newton(w, 1);
  return fma(kd, 6.93147180369123816490e-01 /* ln2_hi: 32 bits, kd * ln2_hi is exact */, corr);
}

// The covariance functions kappa(d2) of the ARD-scaled squared distance d2 = r^2 (DESIGN.md 2.14 for KIDs 3 and 4):
//   KID 0 SqExponential  exp(-r^2 / 2)          KID 3 Matern12 / Exponential  exp(-r)
//   KID 1 Matern32       (1 + sqrt3 r) exp(-sqrt3 r)   KID 4 RationalQuadratic  (1 + r^2 / (2 a))^-a,  a = rq_a > 0
//   KID 2 Matern52       (1 + sqrt5 r + 5 r^2 / 3) exp(-sqrt5 r)
// rq_a is the RQ shape parameter (KernelFunctions' alpha, not BOSS's amplitude); KIDs 0-3 ignore it.  kappa(0) = 1 for
// every KID.  RQ's 0.5 / rq_a is loop-invariant in every caller and hoisted out of the training-point loops.
template <int KID>
__device__ __forceinline__ double kappa_fast(double d2, const double *tab, double rq_a) {
  if (KID == 0) {
    return fast_exp_neg(0.5 * d2, tab);
  } else if (KID == 1) {
    const double t = 1.7320508075688772 * fast_sqrt(d2);
    return (1.0 + t) * fast_exp_neg(t, tab);
  } else if (KID == 2) {
    const double t = 2.23606797749979 * fast_sqrt(d2);
    return (1.0 + t + (5.0 / 3.0) * d2) * fast_exp_neg(t, tab);
  } else if (KID == 3) {
    return fast_exp_neg(fast_sqrt(d2), tab);
  } else {
    static_assert(KID >= 0 && KID <= 4, "kernel id");
    return fast_exp_neg(rq_a * fast_log1p(d2 * (0.5 / rq_a)), tab);
  }
}

// (d kappa / d r) / r, fast variant (see kappa_dr_over_r below)
template <int KID>
__device__ __forceinline__ double kappa_dr_over_r_fast(double d2, const double *tab, double rq_a) {
  if (KID == 0) {
    return -fast_exp_neg(0.5 * d2, tab);
  } else if (KID == 1) {
    return -3.0 * fast_exp_neg(1.7320508075688772 * fast_sqrt(d2), tab);
  } else if (KID == 2) {
    const double t = 2.23606797749979 * fast_sqrt(d2);
    return -(5.0 / 3.0) * (1.0 + t) * fast_exp_neg(t, tab);
  } else if (KID == 3) {
    const double ri = fast_rsqrt(d2);
    const double v = -fast_exp_neg(d2 * ri, tab) * ri;
    return d2 == 0.0 ? 0.0 : v;   // the r = 0 convention (DESIGN.md 2.14): a select, not a branch
  } else {
    static_assert(KID >= 0 && KID <= 4, "kernel id");
    return -fast_exp_neg((rq_a + 1.0) * fast_log1p(d2 * (0.5 / rq_a)), tab);
  }
}

// kappa_fast and kappa_dr_over_r_fast at the same d2 (the log-likelihood gradient's tile pass needs both): RQ shares
// its log1p between the two, every other KID evaluates the two functions above unchanged.
template <int KID>
__device__ __forceinline__ void kappa_and_dr_fast(double d2, const double *tab, double rq_a, double &k, double &g) {
  if (KID == 4) {
    const double l = fast_log1p(d2 * (0.5 / rq_a));
    k = fast_exp_neg(rq_a * l, tab);
    g = -fast_exp_neg((rq_a + 1.0) * l, tab);
  } else {
    k = kappa_fast<KID>(d2, tab, rq_a);
    g = kappa_dr_over_r_fast<KID>(d2, tab, rq_a);
  }
}

template <int KID>
__device__ __forceinline__ double kappa(double d2, double rq_a) {
  if (KID == 0) {
    return exp(-0.5 * d2);
  } else if (KID == 1) {
    const double t = 1.7320508075688772 * sqrt(d2);
    return (1.0 + t) * exp(-t);
  } else if (KID == 2) {
    const double t = 2.23606797749979 * sqrt(d2);
    return (1.0 + t + (5.0 / 3.0) * d2) * exp(-t);
  } else if (KID == 3) {
    return exp(-sqrt(d2));
  } else {
    static_assert(KID >= 0 && KID <= 4, "kernel id");
    return exp(-rq_a * log1p(d2 * (0.5 / rq_a)));
  }
}

// The FP32 mean tier of argmax screening (DESIGN.md 2.9) evaluates kappa two lanes at a time with the packed FP32
// instructions of sm_100 (FADD2 / FMUL2 / FFMA2: one issue slot for two results).
__device__ __forceinline__ float2 f2(float a) { return make_float2(a, a); }
__device__ __forceinline__ float ex2_mufu(float x) {
  float e;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x));
  return e;
}

// FP32 kappa of two squared distances d2 >= 1e-30 (the tier clamps d2 at 1e-30 once, which is also the rsqrt's
// floor: r~ = d2 rsqrt(d2) is below 1e-15 there): one MUFU.RSQ (Matern only) and one MUFU.EX2 per lane, the rest
// packed.  exp(-t) flushes to 0 for t >= ~87.  Absolute error against kappa at the same d2, measured over r in
// [0, 40]: tests/test_gpu_screen_f32.py.
template <int KID>
__device__ __forceinline__ float2 kappa_f32x2(float2 d2) {
  constexpr float C = KID == 0 ? -0.72134752044448170f    /* -log2(e)/2 */
                    : KID == 1 ? -2.4988211106473432f     /* -sqrt3 log2(e) */
                               : -3.2259641822295610f;    /* -sqrt5 log2(e) */
  float2 r = d2;   // SE: the exponent is C d2
  if (KID != 0) {
    float y0, y1;
    asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(y0) : "f"(d2.x));
    asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(y1) : "f"(d2.y));
    r = __fmul2_rn(d2, make_float2(y0, y1));
  }
  const float2 x = __fmul2_rn(r, f2(C));
  const float2 e = make_float2(ex2_mufu(x.x), ex2_mufu(x.y));
  if (KID == 0) return e;
  if (KID == 1) return __ffma2_rn(__fmul2_rn(f2(1.7320508075688772f), r), e, e);
  const float2 t = __fmul2_rn(f2(2.2360679774997896f), r);
  return __ffma2_rn(__ffma2_rn(f2(1.6666666666666667f), d2, t), e, e);
}

// x = hi + lo + r with hi, lo TF32 (round to nearest, ties away): |x - hi| <= 2^-11 |x|, |r| <= 2^-22 |x|.  x - hi is
// exact in FP32.  Non-finite x gives lo = NaN.
__device__ __forceinline__ void tf32_split(float x, float &hi, float &lo) {
  unsigned h, l;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(h) : "f"(x));
  hi = __uint_as_float(h);
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(l) : "f"(x - hi));
  lo = __uint_as_float(l);
}

// (d kappa / d r) / r as a function of d2 = r^2: finite at r = 0 for KIDs 0-2 and 4.  Matern12's -exp(-r) / r is
// unbounded there; it is defined as 0 at d2 == 0 (DESIGN.md 2.14), as a select, so no -Inf * 0 = NaN can reach a sum.
// RQ: -kappa / (1 + r^2 / (2a)) = -(1 + r^2 / (2a))^-(a+1).
template <int KID>
__device__ __forceinline__ double kappa_dr_over_r(double d2, double rq_a) {
  if (KID == 0) {
    return -exp(-0.5 * d2);
  } else if (KID == 1) {
    return -3.0 * exp(-1.7320508075688772 * sqrt(d2));
  } else if (KID == 2) {
    const double t = 2.23606797749979 * sqrt(d2);
    return -(5.0 / 3.0) * (1.0 + t) * exp(-t);
  } else if (KID == 3) {
    const double r = sqrt(d2);
    const double v = -exp(-r) / r;
    return d2 == 0.0 ? 0.0 : v;
  } else {
    static_assert(KID >= 0 && KID <= 4, "kernel id");
    return -exp(-(rq_a + 1.0) * log1p(d2 * (0.5 / rq_a)));
  }
}

// _clip_var, src/models/gaussian_process.jl:186-194.  returns false where the reference throws.
__device__ __forceinline__ bool clip_var(double &v) {
  if (v >= 0.0) return true;
  if (v >= -MAX_NEG_VAR) {
    v = 0.0;
    return true;
  }
  return false;
}

// Load point `p` (d raw coordinates), round flagged dims (ties-to-even like Julia's round), scale by 1/l.
template <int DP>
__device__ __forceinline__ void load_scaled_point(double (&x)[DP], const double *p, int d, const double *invl,
                                                  unsigned long long disc_bits, bool valid) {
#pragma unroll
  for (int i = 0; i < DP; ++i) {
    double v = 0.0;
    if (valid && i < d) {
      v = p[i];
      if ((disc_bits >> i) & 1ull) v = rint(v);
      v *= invl[i];
    }
    x[i] = v;
  }
}
#endif

}  // namespace boss

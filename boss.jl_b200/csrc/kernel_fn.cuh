// kernel_fn.cuh -- covariance function evaluation shared by the kernel-matrix builder (a1) and the
// cross-covariance generator (a3).  Mirrors KernelFunctions' kappa for SqExponential / Matern32 /
// Matern52 composed with ARDTransform(1/l) and ScaledKernel(a^2)  (reference call site:
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

template <int KID>
__device__ __forceinline__ double kappa_fast(double d2, const double *tab) {
  if (KID == 0) {
    return fast_exp_neg(0.5 * d2, tab);
  } else if (KID == 1) {
    const double t = 1.7320508075688772 * fast_sqrt(d2);
    return (1.0 + t) * fast_exp_neg(t, tab);
  } else {
    const double t = 2.23606797749979 * fast_sqrt(d2);
    return (1.0 + t + (5.0 / 3.0) * d2) * fast_exp_neg(t, tab);
  }
}

// (d kappa / d r) / r, fast variant (see kappa_dr_over_r below)
template <int KID>
__device__ __forceinline__ double kappa_dr_over_r_fast(double d2, const double *tab) {
  if (KID == 0) {
    return -fast_exp_neg(0.5 * d2, tab);
  } else if (KID == 1) {
    return -3.0 * fast_exp_neg(1.7320508075688772 * fast_sqrt(d2), tab);
  } else {
    const double t = 2.23606797749979 * fast_sqrt(d2);
    return -(5.0 / 3.0) * (1.0 + t) * fast_exp_neg(t, tab);
  }
}

template <int KID>
__device__ __forceinline__ double kappa(double d2) {
  if (KID == 0) {
    return exp(-0.5 * d2);
  } else if (KID == 1) {
    const double t = 1.7320508075688772 * sqrt(d2);
    return (1.0 + t) * exp(-t);
  } else {
    const double t = 2.23606797749979 * sqrt(d2);
    return (1.0 + t + (5.0 / 3.0) * d2) * exp(-t);
  }
}

// FP32 kappa for the FP32 mean tier of argmax screening (DESIGN.md 2.9): one MUFU.RSQ (Matern only) and one MUFU.EX2.
// r = d2 rsqrt(max(d2, 1e-30)) is 0 at d2 = 0 (|r~ - r| <= 1e-15 below the floor); t >= ~87 flushes exp to 0.
// Absolute error against kappa at the same d2, measured over r in [0, 40]: tests/test_gpu_screen_f32.py.
template <int KID>
__device__ __forceinline__ float kappa_f32(float d2) {
  float e;
  if (KID == 0) {
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(d2 * -0.72134752044448170f /* -log2(e)/2 */));
    return e;
  }
  float y;
  asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(fmaxf(d2, 1e-30f)));
  const float r = d2 * y;
  if (KID == 1) {
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(r * -2.4988211106473432f /* -sqrt3 log2(e) */));
    const float t = 1.7320508075688772f * r;
    return fmaf(t, e, e);
  } else {
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(r * -3.2259641822295610f /* -sqrt5 log2(e) */));
    const float t = 2.2360679774997896f * r;
    return fmaf(fmaf(1.6666666666666667f, d2, t), e, e);
  }
}

// (d kappa / d r) / r as a function of d2 = r^2 : finite at r = 0 for all three kernels.
template <int KID>
__device__ __forceinline__ double kappa_dr_over_r(double d2) {
  if (KID == 0) {
    return -exp(-0.5 * d2);
  } else if (KID == 1) {
    return -3.0 * exp(-1.7320508075688772 * sqrt(d2));
  } else {
    const double t = 2.23606797749979 * sqrt(d2);
    return -(5.0 / 3.0) * (1.0 + t) * exp(-t);
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

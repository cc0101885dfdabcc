// boss_b200.cu -- host runtime + C ABI of libboss_b200.so (see include/boss_b200.h).
//
// One process drives one B200.  All numerics run in the hand-written sm_100a kernels of
// cholesky.cuh / score.cuh on the library's stream; this file owns device memory (grow-only
// workspaces sized for 180 GB HBM3e), the fitted-GP handles (the factor cache) and the chunked
// candidate pipeline.  There is no CPU fallback: every entry point fails with BOSS_ERR_STATE /
// BOSS_ERR_CUDA if the device is not usable.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <ctime>
#include <limits>
#include <map>
#include <mutex>
#include <set>
#include <thread>
#include <functional>
#include <string>
#include <vector>

#include "../../include/boss_b200.h"
#include "cholesky.cuh"
#include "score.cuh"
#include "grad.cuh"
#include "score_narrow.cuh"
#include "append.cuh"
#include "multistart.cuh"
#include "topk.cuh"

using namespace boss;

struct boss_gp;

// ---------------------------------------------------------------------------------------------
// context
// ---------------------------------------------------------------------------------------------
namespace {

// Red zones (BOSS_DEBUG_REDZONE=1; the home-grown stand-in for compute-sanitizer memcheck, which is closed on the
// build pool): every device allocation of the library is then made exactly as large as requested (no growth slack)
// and bracketed by two RZ_BYTES guard bands filled with 0xA5; boss_dbg_check_redzones() scans all live guard bands
// on the device and returns the number of bytes a kernel has overwritten.  Off by default: zero cost.
constexpr size_t RZ_BYTES = 64 << 10;
struct RzEntry {
  char *base;
  size_t bytes;   // user bytes (rounded up to 256)
  int device;
};
std::mutex g_rz_mu;
std::map<void *, RzEntry> g_rz;      // user pointer -> allocation
inline bool redzones_on() {
  static const bool on = getenv("BOSS_DEBUG_REDZONE") != nullptr;
  return on;
}
cudaError_t dev_malloc(void **out, size_t bytes) {
  if (!redzones_on()) return cudaMalloc(out, bytes);
  const size_t user = (bytes + 255) & ~(size_t)255;
  char *base = nullptr;
  cudaError_t e = cudaMalloc(reinterpret_cast<void **>(&base), user + 2 * RZ_BYTES);
  if (e != cudaSuccess) return e;
  cudaMemset(base, 0xA5, RZ_BYTES);
  // the bytes between the requested size and the 256-byte rounding belong to the upper guard band as well
  cudaMemset(base + RZ_BYTES + bytes, 0xA5, user - bytes + RZ_BYTES);
  int dev = -1;
  cudaGetDevice(&dev);
  std::lock_guard<std::mutex> lk(g_rz_mu);
  g_rz[base + RZ_BYTES] = RzEntry{base, bytes, dev};
  *out = base + RZ_BYTES;
  return cudaSuccess;
}
cudaError_t dev_free(void *p) {
  if (!p) return cudaSuccess;
  if (redzones_on()) {
    std::lock_guard<std::mutex> lk(g_rz_mu);
    auto it = g_rz.find(p);
    if (it != g_rz.end()) {
      void *base = it->second.base;
      g_rz.erase(it);
      return cudaFree(base);
    }
  }
  return cudaFree(p);
}

struct DevBuf {
  void *p = nullptr;
  size_t cap = 0;
  cudaError_t ensure(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (p) dev_free(p);
    p = nullptr;
    cap = 0;
    size_t want = redzones_on() ? bytes : bytes + bytes / 8;
    cudaError_t e = dev_malloc(&p, want);
    if (e != cudaSuccess) {
      e = dev_malloc(&p, bytes);
      want = bytes;
    }
    if (e == cudaSuccess) cap = want;
    return e;
  }
  void release() {
    if (p) dev_free(p);
    p = nullptr;
    cap = 0;
  }
  template <class T>
  T *as() const {
    return reinterpret_cast<T *>(p);
  }
};

constexpr int N_TIMERS = 4;
constexpr int LL_GROUPS = 16;  // max concurrent sub-batches of a log-likelihood window (separate streams)
constexpr int EV_POOL = 512;
constexpr int MAX_DEV = 16;

// One context per device.  A process may drive one GPU (boss_init: the torchrun-style one-process-per-GPU layout)
// or several (boss_init_multi: the single-process layout a Julia caller has, SURVEY.md 8b/5).  Every entry point
// works inside exactly one context at a time: it locks the context, makes its device current and publishes it as
// the calling thread's current context (tl_ctx), which is what C() returns to the launch helpers below.
struct Ctx {
  int device = -1;
  cudaStream_t stream = nullptr;
  std::recursive_mutex mu;
  int64_t launches = 0;
  bool timing = false;
  bool attrs_done = false;
  // workspaces
  DevBuf ks, muv, sumsq, xs_stage, pm_stage, acq_stage, mu_stage;
  DevBuf blk_val, blk_idx, small, chol_L, chol_Winv, chol_misc, tt, vt, ut, dmu, dvar;
  DevBuf part_mu, part_ss, part_gm, part_gv, cov_p, cov_stage, chol_W, chol_WT, ll_vec, ll_part, ms_buf;   // split-invariant partial sums (score.cuh / grad.cuh)
  DevBuf scr_misc, scr_pool;         // argmax screening: bounds, counts, seed batch / survivor pool (Screen)
  DevBuf scr_pool2;                  // argmax screening: the pool re-compacted after refinement and re-seed
  DevBuf topk;                       // top-k calls: running set, chunk scores, selection state, sorted result
  int64_t scr_stats[3] = {0, 0, 0};  // last scoring call: screened (1) or fell back (2), candidates bounded, pool size
  int64_t scr_amb[2] = {0, 0};       // last screened call: ambiguous candidates of the FP32 tier, pool before refinement and re-seed
  int64_t scr_var[2] = {0, 0};       // last screened call: pool rows into and out of the variance tier (0, 0: not run)
  int64_t score_paths[5] = {0, 0, 0, 0, 0};   // last scoring call's (chunk, slice) passes by path (boss_dbg_score_paths)
  // event pool for per-kernel-class timing
  cudaEvent_t ev_a[EV_POOL], ev_b[EV_POOL];
  int ev_class[EV_POOL];
  int ev_used = 0;
  bool ev_ready = false;
  double last_ms[N_TIMERS] = {0, 0, 0, 0};
  int last_cnt[N_TIMERS] = {0, 0, 0, 0};
  cudaEvent_t call_a = nullptr, call_b = nullptr;
  cudaEvent_t caller_ev = nullptr;   // orders the library stream after the caller's stream (_dev entry points)
  // handle-buffer pool: a BO loop refits GPs of the same size every iteration; cudaMalloc / cudaFree of the three
  // n_pad^2 factors cost more than the factorisation itself.  Freed buffers are kept (up to POOL_CAP bytes) by size.
  std::multimap<size_t, void *> pool;
  std::map<void *, size_t> pool_sizes;
  size_t pool_bytes = 0;
  cudaStream_t ll_stream[LL_GROUPS] = {};
  cudaEvent_t ll_fork = nullptr, ll_join[LL_GROUPS] = {};
  std::set<boss_gp *> live;          // handles whose buffers live on this device (boss_shutdown invalidates them)
  void *pinned = nullptr;            // pinned slots for chunks of host arrays (see HostStaging)
  size_t pinned_cap = 0;
  cudaEvent_t pin_ev[2] = {nullptr, nullptr};
  // the FP32 screening pass of device-resident calls runs here beside the first chunk's chain (Screen): the lowest
  // priority, the library stream the highest, so that the chain's kernels take SMs as the pass's CTAs retire
  cudaStream_t side = nullptr;
  cudaEvent_t side_fork = nullptr, side_join = nullptr;
};

Ctx *g_ctx[MAX_DEV] = {};            // created by boss_init / boss_init_multi, emptied by boss_shutdown
std::mutex g_reg_mu;                 // guards g_ctx / g_primary / g_ndev
int g_primary = -1;                  // device of boss_init, or the first device of boss_init_multi
int g_ndev = 0;                      // number of devices multi-device calls fan out to (0 or 1: single device)
thread_local Ctx *tl_ctx = nullptr;  // context the calling thread is working in
thread_local int tl_dev = -1;        // boss_set_device(): device of this thread's _dev calls and new handles
thread_local std::string tl_err;     // boss_last_error() of the calling thread

inline Ctx &C() { return *tl_ctx; }

Ctx *ctx_of(int dev) { return (dev >= 0 && dev < MAX_DEV && g_ctx[dev] && g_ctx[dev]->device == dev) ? g_ctx[dev] : nullptr; }
Ctx *ctx_current() { return ctx_of(tl_dev >= 0 ? tl_dev : g_primary); }

// RAII: lock a context, make it (and its device) current for this thread
struct Enter {
  Ctx *prev;
  std::unique_lock<std::recursive_mutex> lk;
  explicit Enter(Ctx *c) : prev(tl_ctx) {
    if (c) {
      lk = std::unique_lock<std::recursive_mutex>(c->mu);
      tl_ctx = c;
      cudaSetDevice(c->device);
    }
  }
  ~Enter() { tl_ctx = prev; }
  Enter(const Enter &) = delete;
  Enter &operator=(const Enter &) = delete;
};

constexpr size_t POOL_CAP = (size_t)16 << 30;

cudaError_t pool_alloc(double **out, size_t bytes) {
  auto it = C().pool.find(bytes);
  if (it != C().pool.end()) {
    *out = reinterpret_cast<double *>(it->second);
    C().pool_bytes -= bytes;
    C().pool.erase(it);
    return cudaSuccess;
  }
  void *p = nullptr;
  cudaError_t e = dev_malloc(&p, bytes);
  if (e != cudaSuccess && !C().pool.empty()) {   // out of memory: drop the pooled buffers and retry
    for (auto &kv : C().pool) {
      dev_free(kv.second);
      C().pool_sizes.erase(kv.second);
    }
    C().pool.clear();
    C().pool_bytes = 0;
    cudaGetLastError();
    e = dev_malloc(&p, bytes);
  }
  if (e == cudaSuccess) {
    C().pool_sizes[p] = bytes;
    *out = reinterpret_cast<double *>(p);
  }
  return e;
}
void pool_free(void *p) {
  if (!p) return;
  auto it = C().pool_sizes.find(p);
  if (it == C().pool_sizes.end() || C().pool_bytes + it->second > POOL_CAP || C().device < 0) {
    if (it != C().pool_sizes.end()) C().pool_sizes.erase(it);
    dev_free(p);
    return;
  }
  C().pool.emplace(it->second, p);
  C().pool_bytes += it->second;
}
void pool_release_all() {
  for (auto &kv : C().pool) dev_free(kv.second);
  C().pool.clear();
  C().pool_sizes.clear();
  C().pool_bytes = 0;
}

int fail(int code, const std::string &msg) {
  tl_err = msg;
  return code;
}

#define CUDA_TRY(expr)                                                                                 \
  do {                                                                                                 \
    cudaError_t _e = (expr);                                                                           \
    if (_e != cudaSuccess)                                                                             \
      return fail(BOSS_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e) + " (" __FILE__ ":" + \
                                     std::to_string(__LINE__) + ")");                                  \
  } while (0)

// timing helpers: bracket one launch with a pooled event pair, recorded on the stream the launch goes to
struct Timed {
  int slot = -1;
  cudaStream_t st;
  Timed(int cls, cudaStream_t s = nullptr) : st(s ? s : C().stream) {
    if (C().timing && C().ev_used < EV_POOL) {
      slot = C().ev_used++;
      C().ev_class[slot] = cls;
      cudaEventRecord(C().ev_a[slot], st);
    }
  }
  ~Timed() {
    if (slot >= 0) cudaEventRecord(C().ev_b[slot], st);
  }
};

void timing_begin() {
  C().ev_used = 0;
  if (C().timing) cudaEventRecord(C().call_a, C().stream);
}
void timing_end() {  // call after the stream has been synchronised
  for (int c = 0; c < N_TIMERS; ++c) {
    C().last_ms[c] = 0;
    C().last_cnt[c] = 0;
  }
  if (!C().timing) return;
  cudaEventRecord(C().call_b, C().stream);
  cudaEventSynchronize(C().call_b);
  float ms = 0;
  cudaEventElapsedTime(&ms, C().call_a, C().call_b);
  C().last_ms[3] = ms;
  C().last_cnt[3] = 1;
  for (int i = 0; i < C().ev_used; ++i) {
    cudaEventElapsedTime(&ms, C().ev_a[i], C().ev_b[i]);
    C().last_ms[C().ev_class[i]] += ms;
    C().last_cnt[C().ev_class[i]] += 1;
  }
}

int pick_dp(int d) {
  if (d <= 2) return 2;
  if (d <= 4) return 4;
  if (d <= 6) return 6;
  if (d <= 8) return 8;
  if (d <= 12) return 12;
  if (d <= 16) return 16;
  if (d <= 32) return 32;
  return -1;
}

unsigned long long mask_bits(const uint8_t *mask, int d) {
  unsigned long long b = 0;
  if (mask)
    for (int i = 0; i < d; ++i)
      if (mask[i]) b |= (1ull << i);
  return b;
}

// Number of zig-zag row-block splits per candidate block for the triangular products (score_trmm / wtv):
// minimise waves x (largest per-CTA share of the nblk(nblk+1)/2 block-steps + ~1 block-step of pipeline fill).
int pick_row_splits(int ncb, int nblk, double *cost = nullptr) {
  if (cost) *cost = ((ncb + 147) / 148) * (nblk * (nblk + 1) / 2 + 1.0);
  if (ncb >= 4 * 148 || nblk < 2) return 1;
  double best_t = 1e300;
  int best = 1;
  for (int ns = 1; ns <= nblk; ++ns) {
    int maxw = 0;
    for (int y = 0; y < ns; ++y) {
      int w = 0;
      for (int j = 0;; ++j) {
        const int i = (j >> 1) * 2 * ns + ((j & 1) ? 2 * ns - 1 - y : y);
        if (i >= nblk) break;
        w += i + 1;
      }
      maxw = std::max(maxw, w);
    }
    const long ctas = (long)ncb * ns, waves = (ctas + 147) / 148;
    const double t = (double)waves * (maxw + 1.0);
    if (t < best_t * (1.0 - 1e-9)) {
      best_t = t;
      best = ns;
    }
  }
  if (cost) *cost = best_t;
  return best;
}

// cost model of the quarter-row kernels (score_narrow.cuh) in pick_row_splits' unit (one 128-block step of the wide
// kernel on one SM, 17 us): per row block of the longest CTA's chain, per (32-candidate block x block step) of tensor
// work spread over the GPU, fixed cost of the extra reduction launch.  Calibrated on the B200 (tools/bench_small_batch.py).
constexpr long long MS_FAN_BATCH = 256;   // capacity of a multi-start round's batch once the step-size fan is on
constexpr double NQ_COST_CHAIN = 0.085, NQ_COST_WORK = 0.0019, NQ_COST_FIXED = 0.15;

// dynamic shared-memory opt-in is per device: once per context
int set_kernel_attrs() {
  if (C().attrs_done) return 0;
  CUDA_TRY(cudaFuncSetAttribute(chol_update_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_SMEM_BYTES));
  CUDA_TRY(cudaFuncSetAttribute(chol_trsm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_SMEM_BYTES));
  CUDA_TRY(cudaFuncSetAttribute(chol_panel_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, PANEL_SMEM_BYTES));
  CUDA_TRY(cudaFuncSetAttribute(trtri_fused_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, PANEL_SMEM_BYTES));
  CUDA_TRY(cudaFuncSetAttribute(gemm_nt_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_SMEM_BYTES));
  CUDA_TRY(cudaFuncSetAttribute(kinv_wtw_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_SMEM_BYTES));
  CUDA_TRY(cudaFuncSetAttribute(chol_update_rl_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_SMEM_BYTES));
  CUDA_TRY(cudaFuncSetAttribute(trtri_acc_rl_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_SMEM_BYTES));
  CUDA_TRY(cudaFuncSetAttribute(trtri_row_rl_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_SMEM_BYTES));
  CUDA_TRY(cudaFuncSetAttribute(score_trmm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_SMEM_BYTES));
  CUDA_TRY(cudaFuncSetAttribute(topk_sort_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, TOPK_SORT_SMEM));
  CUDA_TRY(cudaFuncSetAttribute(wtv_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_SMEM_BYTES));
  CUDA_TRY(cudaFuncSetAttribute(score_narrow_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, NW_SMEM_BYTES));
  CUDA_TRY(cudaFuncSetAttribute(score_narrow_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, NW_SMEM_BYTES));
  CUDA_TRY(cudaFuncSetAttribute(score_quarter_kernel<0, 4, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, NQ_SMEM_BYTES));
  CUDA_TRY(cudaFuncSetAttribute(score_quarter_kernel<1, 4, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, NQ_SMEM_BYTES));
  CUDA_TRY(cudaFuncSetAttribute(potrf_tile_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, PT_SMEM_BYTES));
  CUDA_TRY(cudaFuncSetAttribute(potrf_fused_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, PF_SMEM_BYTES));
  C().attrs_done = true;
  return 0;
}

// ---------------------------------------------------------------------------------------------
// batched blocked Cholesky driver (shared by fit and loglik)
// ---------------------------------------------------------------------------------------------
// On return L holds the factors, Winv the inverted diagonal blocks, logdet_blk / status are filled.
// W / WT non-null (S must be 1): also form the full triangular inverse.
// fwd non-null (left-looking only): the forward substitution w = L^-1 delta rides along (r_j in the diagonal-tile
// SYRK, w_j and |w_j|^2 in potrf_tile_kernel), so the log-likelihood needs no pass over L afterwards.
struct FwdInline {
  const double *ymm;   // delta of the first matrix; matrix s reads ymm + s * ldy
  long long ldy;
  int n, n_pad;
  double *r, *w;       // [S][n_pad] scratch / result
  double *ssq;         // [S][nblk]
};
// gen non-null (left-looking only): the diagonal-block kernel forms its own input tile (potrf_fused_kernel: K_jj from
// the hyper-parameters minus the SYRK of row block j) -- build_k must then have been launched with skip_diag.
int run_cholesky(double *L, size_t L_stride, double *Winv, size_t Winv_stride, int nblk, int ktiles, int S,
                 double *logdet_blk, int *status, double *W, double *WT, double *TT, size_t W_stride = 0,
                 size_t TT_stride = 0, bool single_fit = false, const FwdInline *fwd = nullptr,
                 const BuildKParams *gen = nullptr, int gen_kid = 0, int gen_dp = 0, bool store_L = true) {
  CholGemmParams gp{};
  gp.L = L;
  gp.L_stride = L_stride;
  gp.Winv = Winv;
  gp.Winv_stride = Winv_stride;
  gp.nblk = nblk;
  gp.ktiles = ktiles;
  gp.W = W;
  gp.WT = WT;
  gp.TT = TT;
  gp.W_stride = W_stride;
  gp.TT_stride = TT_stride;
  PotrfParams pp{};
  pp.L = L;
  pp.L_stride = L_stride;
  pp.Winv = Winv;
  pp.Winv_stride = Winv_stride;
  pp.nblk = nblk;
  pp.ktiles = ktiles;
  pp.logdet_blk = logdet_blk;
  pp.status = status;
  pp.W = W;
  pp.WT = WT;
  pp.W_stride = W_stride;
  if (fwd) {
    gp.fwd_w = fwd->w;
    gp.fwd_r = fwd->r;
    gp.n_pad = fwd->n_pad;
    pp.fwd_ymm = fwd->ymm;
    pp.fwd_ldy = fwd->ldy;
    pp.fwd_n = fwd->n;
    pp.n_pad = fwd->n_pad;
    pp.fwd_r = fwd->r;
    pp.fwd_w = fwd->w;
    pp.fwd_ssq = fwd->ssq;
  }
  // Left-looking keeps accumulators in registers over the whole k-range (best when S x nblk CTAs fill the GPU);
  // a small batch (a single posterior fit) cannot fill 148 SMs that way -> right-looking steps of K = 128 tiles.
  // Only the posterior fit takes this path: batched log-likelihoods always run left-looking, so a sample's value
  // never depends on how the batch was split (over sub-batches, streams or GPUs).
  const bool right_looking = single_fit && (long long)S * nblk <= 148;
  const bool fused_diag = gen != nullptr && !right_looking;
  if (fused_diag) {
    pp.gen_X = gen->X;
    pp.gen_d = gen->d;
    pp.gen_dp = gen_dp;
    pp.gen_n = gen->n;
    pp.gen_kid = gen_kid;
    pp.gen_rq_a = gen->rq_a;
    pp.gen_ls = gen->ls;
    pp.gen_amp = gen->amp;
    pp.gen_noise = gen->noise;
    pp.gen_disc = gen->disc_bits;
    pp.store_L = store_L ? 1 : 0;
  }
  for (int j = 0; j < nblk; ++j) {
    gp.j = j;
    pp.j = j;
    // left-looking, column j >= 1: SYRK of the diagonal tile + potrf (one kernel) -> fused update + panel solve of the rows below
    const bool fused_panel = j > 0 && !right_looking;
    if (fused_diag) {
      Timed t(2);
      potrf_fused_kernel<<<S, 256, PF_SMEM_BYTES, C().stream>>>(pp);
      ++C().launches;
    } else {
      if (fused_panel) {
        Timed t(2);
        chol_update_kernel<<<dim3(1, S), GEMM_THREADS, GEMM_SMEM_BYTES, C().stream>>>(gp);
        ++C().launches;
      }
      potrf_tile_kernel<<<S, 256, PT_SMEM_BYTES, C().stream>>>(pp);
      ++C().launches;
    }
    if (j < nblk - 1) {
      Timed t(2);
      if (fused_panel)
        chol_panel_kernel<<<dim3(nblk - j - 1, S), GEMM_THREADS, PANEL_SMEM_BYTES, C().stream>>>(gp);
      else
        chol_trsm_kernel<<<dim3(nblk - j - 1, S), GEMM_THREADS, GEMM_SMEM_BYTES, C().stream>>>(gp);
      ++C().launches;
      if (right_looking) {
        const int m = nblk - j - 1;
        chol_update_rl_kernel<<<dim3(m * (m + 1) / 2, S), GEMM_THREADS, GEMM_SMEM_BYTES, C().stream>>>(gp);
        ++C().launches;
      }
    }
  }
  if (W && right_looking) {
    for (int k = 0; k + 1 < nblk; ++k) {
      Timed t(2);
      gp.j = k;
      trtri_acc_rl_kernel<<<dim3((nblk - k - 1) * (k + 1), S), GEMM_THREADS, GEMM_SMEM_BYTES, C().stream>>>(gp);
      gp.j = k + 1;
      trtri_row_rl_kernel<<<dim3(k + 1, S), GEMM_THREADS, GEMM_SMEM_BYTES, C().stream>>>(gp);
      C().launches += 2;
    }
  } else if (W) {
    for (int delta = 1; delta < nblk; ++delta) {
      gp.j = delta;
      Timed t(2);
      trtri_fused_kernel<<<dim3(nblk - delta, S), GEMM_THREADS, PANEL_SMEM_BYTES, C().stream>>>(gp);
      ++C().launches;
    }
  }
  CUDA_TRY(cudaGetLastError());
  return 0;
}

}  // namespace

// ---------------------------------------------------------------------------------------------
// handle
// ---------------------------------------------------------------------------------------------
struct boss_gp {
  int n = 0, d = 0, n_pad = 0, nblk = 0, ktiles = 0, kernel_id = 0, dp = 0;   // kernel_id: the decoded KID (0-4)
  double rq_a = 0.0;                                                         // RationalQuadratic shape (KID 4)
  unsigned long long disc = 0;
  double amp = 0, noise = 0, a2 = 0;
  double loglik = 0;
  double *W = nullptr, *WT = nullptr, *L = nullptr, *alpha = nullptr, *Xt = nullptr, *invl = nullptr;
  double *wvec = nullptr, *ymm = nullptr;   // w = L^-1 delta and delta = y - m(X), kept for boss_gp_append
  int dev = -1;                             // device the buffers live on (-1: invalidated by boss_shutdown)
  // multi-device mode (boss_init_multi): the handle the caller holds is the replica on the primary device; rep[k]
  // is the bit-identical replica on device k (rep[dev] == this).  Replicas are owned by the primary handle.
  boss_gp *rep[MAX_DEV] = {};
  void free_dev() {   // call inside the handle's context
    for (double **q : {&W, &WT, &L, &alpha, &Xt, &invl, &wvec, &ymm}) {
      if (*q) pool_free(*q);
      *q = nullptr;
    }
  }
};

namespace {

// the replica of `h` that lives on device `dev` (nullptr if there is none)
const boss_gp *replica_on(const boss_gp *h, int dev) {
  if (!h) return nullptr;
  if (h->dev == dev) return h;
  return (dev >= 0 && dev < MAX_DEV) ? h->rep[dev] : nullptr;
}

int init_device(int device) {   // g_reg_mu held
  int count = 0;
  CUDA_TRY(cudaGetDeviceCount(&count));
  if (device < 0 || device >= count || device >= MAX_DEV) return fail(BOSS_ERR_ARG, "boss_init: no such CUDA device");
  if (g_ctx[device] && g_ctx[device]->device == device) return 0;
  if (!g_ctx[device]) g_ctx[device] = new Ctx();
  Ctx *cx = g_ctx[device];
  Enter en(cx);
  CUDA_TRY(cudaSetDevice(device));
  cudaDeviceProp prop;
  CUDA_TRY(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) return fail(BOSS_ERR_STATE, std::string("boss_init: built for sm_100a, device is ") + prop.name);
  int prio_lo = 0, prio_hi = 0;
  CUDA_TRY(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
  CUDA_TRY(cudaStreamCreateWithPriority(&cx->stream, cudaStreamNonBlocking, prio_hi));
  CUDA_TRY(cudaStreamCreateWithPriority(&cx->side, cudaStreamNonBlocking, prio_lo));
  CUDA_TRY(cudaEventCreateWithFlags(&cx->side_fork, cudaEventDisableTiming));
  CUDA_TRY(cudaEventCreateWithFlags(&cx->side_join, cudaEventDisableTiming));
  for (int i = 0; i < EV_POOL; ++i) {
    CUDA_TRY(cudaEventCreate(&cx->ev_a[i]));
    CUDA_TRY(cudaEventCreate(&cx->ev_b[i]));
  }
  CUDA_TRY(cudaEventCreate(&cx->call_a));
  CUDA_TRY(cudaEventCreate(&cx->call_b));
  CUDA_TRY(cudaEventCreateWithFlags(&cx->caller_ev, cudaEventDisableTiming));
  CUDA_TRY(cudaEventCreateWithFlags(&cx->ll_fork, cudaEventDisableTiming));
  for (int i = 0; i < 2; ++i) CUDA_TRY(cudaEventCreateWithFlags(&cx->pin_ev[i], cudaEventDisableTiming));
  for (int i = 0; i < LL_GROUPS; ++i) {
    CUDA_TRY(cudaStreamCreateWithFlags(&cx->ll_stream[i], cudaStreamNonBlocking));
    CUDA_TRY(cudaEventCreateWithFlags(&cx->ll_join[i], cudaEventDisableTiming));
  }
  cx->ev_ready = true;
  cx->device = device;
  return set_kernel_attrs();
}

void shutdown_device(Ctx *cx) {   // g_reg_mu held
  Enter en(cx);
  if (cx->device < 0) return;
  cudaStreamSynchronize(cx->stream);
  // handles that are still alive lose their device buffers; later calls on them fail with BOSS_ERR_STATE and
  // boss_gp_free only releases the host structure
  for (boss_gp *h : cx->live) {
    h->free_dev();
    h->dev = -1;
  }
  cx->live.clear();
  for (DevBuf *b : {&cx->ks, &cx->muv, &cx->sumsq, &cx->xs_stage, &cx->pm_stage, &cx->acq_stage, &cx->mu_stage,
                    &cx->blk_val, &cx->blk_idx, &cx->small, &cx->chol_L, &cx->chol_Winv, &cx->chol_misc, &cx->tt, &cx->vt,
                    &cx->ut, &cx->dmu, &cx->dvar, &cx->part_mu, &cx->part_ss, &cx->part_gm, &cx->part_gv, &cx->cov_p,
                    &cx->cov_stage, &cx->chol_W, &cx->chol_WT, &cx->ll_vec, &cx->ll_part, &cx->ms_buf})
    b->release();
  pool_release_all();
  if (cx->pinned) cudaFreeHost(cx->pinned);
  cx->pinned = nullptr;
  cx->pinned_cap = 0;
  if (cx->ev_ready) {
    for (int i = 0; i < EV_POOL; ++i) {
      cudaEventDestroy(cx->ev_a[i]);
      cudaEventDestroy(cx->ev_b[i]);
    }
    cudaEventDestroy(cx->call_a);
    cudaEventDestroy(cx->call_b);
    cudaEventDestroy(cx->caller_ev);
    cudaEventDestroy(cx->ll_fork);
    for (int i = 0; i < 2; ++i) cudaEventDestroy(cx->pin_ev[i]);
    for (int i = 0; i < LL_GROUPS; ++i) {
      cudaStreamDestroy(cx->ll_stream[i]);
      cudaEventDestroy(cx->ll_join[i]);
    }
    cx->ev_ready = false;
  }
  cudaStreamSynchronize(cx->side);
  cudaStreamDestroy(cx->side);
  cudaEventDestroy(cx->side_fork);
  cudaEventDestroy(cx->side_join);
  cx->side = nullptr;
  cx->side_fork = cx->side_join = nullptr;
  cudaStreamDestroy(cx->stream);
  cx->stream = nullptr;
  cx->attrs_done = false;
  cx->device = -1;
}

// Run fn(k, context of device k) for the ndev devices of a multi-device call on one host thread each and return the
// first non-zero status in device order.  Each worker enters its own context, so the calls below it are exactly the
// single-device code paths.
int for_each_device(int ndev, const std::function<int(int, Ctx *)> &fn) {
  std::vector<int> rc(ndev, 0);
  std::vector<std::string> err(ndev);
  std::vector<std::thread> th;
  for (int k = 0; k < ndev; ++k)
    th.emplace_back([&, k]() {
      Ctx *cx = ctx_of(k);
      if (!cx) {
        rc[k] = BOSS_ERR_STATE;
        err[k] = "multi-device call: device not initialised";
        return;
      }
      Enter en(cx);
      rc[k] = fn(k, cx);
      if (rc[k]) err[k] = tl_err;
    });
  for (auto &t : th) t.join();
  for (int k = 0; k < ndev; ++k)
    if (rc[k] < 0) return fail(rc[k], err[k]);
  for (int k = 0; k < ndev; ++k)
    if (rc[k]) {
      tl_err = err[k];
      return rc[k];
    }
  return 0;
}

// Kernel ids: 0-3 name a covariance function directly; 256 + slot names RationalQuadratic with the rq_a registered in
// that slot (boss_kernel_rational_quadratic).  The table lives for the process and holds no device state; a slot is
// written once, under the mutex, before its id is handed out.
constexpr int RQ_ID0 = 256;
std::mutex g_rq_mu;
uint64_t g_rq_bits[BOSS_RQ_SLOTS];
int g_rq_n = 0;

struct KernelSpec {
  int kid = 0;        // template KID of the device kernels (tk_params.cuh)
  double rq_a = 0.0;  // RationalQuadratic shape parameter (kid 4)
};

// kernel_id -> (KID, rq_a); false for an unknown id
bool decode_kernel(int kernel_id, KernelSpec *ks) {
  if (kernel_id >= 0 && kernel_id <= BOSS_KERNEL_MATERN12) {
    *ks = KernelSpec{kernel_id, 0.0};
    return true;
  }
  if (kernel_id < RQ_ID0 || kernel_id >= RQ_ID0 + BOSS_RQ_SLOTS) return false;
  std::lock_guard<std::mutex> lk(g_rq_mu);
  const int slot = kernel_id - RQ_ID0;
  if (slot >= g_rq_n) return false;
  double a;
  std::memcpy(&a, &g_rq_bits[slot], 8);
  *ks = KernelSpec{4, a};
  return true;
}

// boss_dbg_kernel_fn_id: the four covariance-function variants of one KID at n squared distances
template <int KID>
__global__ void dbg_kernel_fn_id_kernel(int which, double rq_a, const double *d2, double *out, int n) {
  __shared__ double tab[EXPTAB_N];
  exptab_init(tab);
  __syncthreads();
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const double x = d2[i];
    out[i] = which == 0 ? kappa_fast<KID>(x, tab, rq_a)
             : which == 1 ? kappa_dr_over_r_fast<KID>(x, tab, rq_a)
             : which == 2 ? kappa<KID>(x, rq_a)
                          : kappa_dr_over_r<KID>(x, rq_a);
  }
}

}  // namespace

extern "C" {

int boss_kernel_rational_quadratic(double rq_a, int *kernel_id) {
  if (!kernel_id) return fail(BOSS_ERR_ARG, "boss_kernel_rational_quadratic: kernel_id is NULL");
  if (!std::isfinite(rq_a) || !(rq_a > 0.0))
    return fail(BOSS_ERR_ARG, "boss_kernel_rational_quadratic: rq_a must be finite and > 0");
  uint64_t bits;
  std::memcpy(&bits, &rq_a, 8);
  std::lock_guard<std::mutex> lk(g_rq_mu);
  for (int i = 0; i < g_rq_n; ++i)
    if (g_rq_bits[i] == bits) {
      *kernel_id = RQ_ID0 + i;
      return 0;
    }
  if (g_rq_n >= BOSS_RQ_SLOTS)
    return fail(BOSS_ERR_ARG, "boss_kernel_rational_quadratic: all " + std::to_string(BOSS_RQ_SLOTS) +
                                  " rational-quadratic slots are in use");
  g_rq_bits[g_rq_n] = bits;
  *kernel_id = RQ_ID0 + g_rq_n++;
  return 0;
}

int boss_version(void) { return 200; }
int boss_device(void) {
  Ctx *cx = ctx_current();
  return cx ? cx->device : -1;
}
int boss_n_devices(void) { return g_ndev; }
void *boss_stream(void) {
  Ctx *cx = ctx_current();
  return cx ? (void *)cx->stream : nullptr;
}
const char *boss_last_error(void) { return tl_err.c_str(); }
int64_t boss_launch_count(void) {
  int64_t t = 0;
  for (int k = 0; k < MAX_DEV; ++k)
    if (g_ctx[k]) t += g_ctx[k]->launches;
  return t;
}
double boss_last_kernel_ms(int which) {
  Ctx *cx = ctx_current();
  return (cx && which >= 0 && which < N_TIMERS) ? cx->last_ms[which] : 0.0;
}
int boss_last_kernel_count(int which) {
  Ctx *cx = ctx_current();
  return (cx && which >= 0 && which < N_TIMERS) ? cx->last_cnt[which] : 0;
}
void boss_set_timing(int on) {
  for (int k = 0; k < MAX_DEV; ++k)
    if (g_ctx[k]) g_ctx[k]->timing = on != 0;
}

int boss_init(int device) {
  std::lock_guard<std::mutex> lk(g_reg_mu);
  if (g_primary >= 0 && g_primary != device && g_ndev <= 1)
    return fail(BOSS_ERR_STATE, "boss_init: already initialised on another device (use boss_init_multi to drive several)");
  int rc = init_device(device);
  if (rc) return rc;
  if (g_primary < 0) {
    g_primary = device;
    g_ndev = 1;
  }
  return 0;
}

int boss_init_multi(int n_gpus) {
  std::lock_guard<std::mutex> lk(g_reg_mu);
  int count = 0;
  CUDA_TRY(cudaGetDeviceCount(&count));
  if (n_gpus < 1 || n_gpus > count || n_gpus > MAX_DEV) return fail(BOSS_ERR_ARG, "boss_init_multi: bad device count");
  if (g_primary > 0) return fail(BOSS_ERR_STATE, "boss_init_multi: already initialised on a device other than 0");
  for (int k = 0; k < n_gpus; ++k) {
    int rc = init_device(k);
    if (rc) return rc;
  }
  g_primary = 0;
  g_ndev = std::max(g_ndev, n_gpus);
  return 0;
}

int boss_set_device(int device) {
  if (device < 0) {
    tl_dev = -1;
    return 0;
  }
  if (!ctx_of(device)) return fail(BOSS_ERR_STATE, "boss_set_device: device not initialised");
  tl_dev = device;
  return 0;
}

void boss_shutdown(void) {
  std::lock_guard<std::mutex> lk(g_reg_mu);
  for (int k = 0; k < MAX_DEV; ++k)
    if (g_ctx[k]) shutdown_device(g_ctx[k]);
  g_primary = -1;
  g_ndev = 0;
  tl_dev = -1;
}

// pick the calling thread's context, lock it and make it current; `cx` is visible to the rest of the function
#define REQUIRE_INIT()                                                                    \
  Ctx *cx = ctx_current();                                                                \
  if (!cx) return fail(BOSS_ERR_STATE, "boss_init() has not been called");                \
  Enter _enter(cx)
// the same for calls that work on a fitted handle: the context is the one the handle lives in
#define REQUIRE_HANDLE_CTX(h)                                                                              \
  Ctx *cx = (h) ? ctx_of((h)->dev) : ctx_current();                                                        \
  if (!cx) return fail(BOSS_ERR_STATE, (h) ? "handle is not valid any more (boss_shutdown was called)"     \
                                           : "boss_init() has not been called");                           \
  Enter _enter(cx)

// ---------------------------------------------------------------------------------------------
// fit
// ---------------------------------------------------------------------------------------------
// one posterior fit inside the current context
static int fit_single(const double *X, int d, int n, const double *y_minus_mean, const double *lengthscales,
                      double amplitude, double noise_std, KernelSpec ks, const uint8_t *discrete_mask, boss_gp **out,
                      double *loglik_out) {
  if (!out) return fail(BOSS_ERR_ARG, "boss_gp_fit: out is NULL");
  *out = nullptr;
  if (!X || !y_minus_mean || !lengthscales || d < 1 || n < 1) return fail(BOSS_ERR_ARG, "boss_gp_fit: bad arguments");
  const int kernel_id = ks.kid;
  const int dp = pick_dp(d);
  if (dp < 0) return fail(BOSS_ERR_ARG, "boss_gp_fit: x_dim > 32 is not supported");
  // reference asserts (src/models/gaussian_process.jl:227-229)
  for (int i = 0; i < d; ++i)
    if (!(lengthscales[i] >= 0)) return fail(BOSS_ERR_ARG, "boss_gp_fit: negative lengthscale");
  if (!(amplitude >= 0) || !(noise_std >= 0)) return fail(BOSS_ERR_ARG, "boss_gp_fit: negative amplitude / noise_std");

  boss_gp *h = new boss_gp();
  h->n = n;
  h->d = d;
  h->n_pad = round_up(n, TM);
  h->nblk = h->n_pad / TM;
  h->ktiles = h->n_pad / TK;
  h->kernel_id = kernel_id;
  h->rq_a = ks.rq_a;
  h->dp = dp;
  h->disc = mask_bits(discrete_mask, d);
  h->amp = amplitude + MIN_PARAM_VALUE;
  h->noise = noise_std + MIN_PARAM_VALUE;
  h->a2 = h->amp * h->amp;
  const size_t npad = h->n_pad, mat = npad * npad;
  const int nblk = h->nblk;

  auto bail = [&](int code) {
    h->free_dev();
    delete h;
    return code;
  };
#define FIT_TRY(expr)                                                                                         \
  do {                                                                                                        \
    cudaError_t _e = (expr);                                                                                  \
    if (_e != cudaSuccess)                                                                                    \
      return bail(fail(BOSS_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e) + " (line " +       \
                                          std::to_string(__LINE__) + ")"));                                   \
  } while (0)

  FIT_TRY(pool_alloc(&h->L, mat * 8));
  FIT_TRY(pool_alloc(&h->W, mat * 8));
  FIT_TRY(pool_alloc(&h->WT, mat * 8));
  FIT_TRY(pool_alloc(&h->alpha, npad * 8));
  FIT_TRY(pool_alloc(&h->Xt, npad * dp * 8));
  FIT_TRY(pool_alloc(&h->invl, dp * 8));
  FIT_TRY(pool_alloc(&h->wvec, npad * 8));
  FIT_TRY(pool_alloc(&h->ymm, npad * 8));
  FIT_TRY(cudaMemsetAsync(h->L, 0, mat * 8, C().stream));
  FIT_TRY(cudaMemsetAsync(h->W, 0, mat * 8, C().stream));
  FIT_TRY(cudaMemsetAsync(h->WT, 0, mat * 8, C().stream));

  // misc device scratch: X | ymm_pad | ls | amp | noise | invl(host computed) | logdet_blk | w | status
  const size_t off_X = 0, off_y = off_X + (size_t)n * d, off_ls = off_y + npad, off_amp = off_ls + d,
               off_noise = off_amp + 1, off_ld = off_noise + 1, off_w = off_ld + nblk, off_st = off_w + npad,
               total = off_st + 2;
  FIT_TRY(C().chol_misc.ensure(total * 8));
  double *misc = C().chol_misc.as<double>();
  FIT_TRY(cudaMemsetAsync(misc, 0, total * 8, C().stream));
  FIT_TRY(cudaMemcpyAsync(misc + off_X, X, (size_t)n * d * 8, cudaMemcpyHostToDevice, C().stream));
  FIT_TRY(cudaMemcpyAsync(misc + off_y, y_minus_mean, (size_t)n * 8, cudaMemcpyHostToDevice, C().stream));
  FIT_TRY(cudaMemcpyAsync(misc + off_ls, lengthscales, (size_t)d * 8, cudaMemcpyHostToDevice, C().stream));
  FIT_TRY(cudaMemcpyAsync(misc + off_amp, &amplitude, 8, cudaMemcpyHostToDevice, C().stream));
  FIT_TRY(cudaMemcpyAsync(misc + off_noise, &noise_std, 8, cudaMemcpyHostToDevice, C().stream));
  std::vector<double> invl(dp, 0.0);
  for (int i = 0; i < d; ++i) invl[i] = 1.0 / (lengthscales[i] + MIN_PARAM_VALUE);
  FIT_TRY(cudaMemcpyAsync(h->invl, invl.data(), dp * 8, cudaMemcpyHostToDevice, C().stream));
  int *status = reinterpret_cast<int *>(misc + off_st);

  FIT_TRY(C().chol_Winv.ensure((size_t)nblk * TM * TM * 8));

  timing_begin();
  BuildKParams bk{};
  bk.X = misc + off_X;
  bk.d = d;
  bk.n = n;
  bk.nblk = nblk;
  bk.ktiles = h->ktiles;
  bk.ls = misc + off_ls;
  bk.amp = misc + off_amp;
  bk.noise = misc + off_noise;
  bk.disc_bits = h->disc;
  bk.K = h->L;
  bk.K_stride = mat;
  bk.status = status;
  bk.rq_a = ks.rq_a;
  {
    Timed t(1);
    launch_build_k(kernel_id, dp, bk, dim3(nblk * (nblk + 1) / 2, 1), C().stream);
    ++C().launches;
  }
  int rc = run_cholesky(h->L, mat, C().chol_Winv.as<double>(), (size_t)nblk * TM * TM, nblk, h->ktiles, 1,
                        misc + off_ld, status, h->W, h->WT, nullptr, 0, 0, true);
  if (rc) return bail(rc);
  // w = W delta ; alpha = W^T w
  matvec_p_kernel<<<h->n_pad / 64, 256, 0, C().stream>>>(h->W, misc + off_y, misc + off_w, h->ktiles);
  matvec_p_kernel<<<h->n_pad / 64, 256, 0, C().stream>>>(h->WT, misc + off_w, h->alpha, h->ktiles);
  {
    const int tot = h->n_pad * dp;
    scale_train_kernel<<<(tot + 255) / 256, 256, 0, C().stream>>>(misc + off_X, d, n, h->n_pad, dp, h->invl, h->disc, h->Xt);
  }
  C().launches += 3;
  FIT_TRY(cudaGetLastError());
  FIT_TRY(cudaMemcpyAsync(h->wvec, misc + off_w, npad * 8, cudaMemcpyDeviceToDevice, C().stream));
  FIT_TRY(cudaMemcpyAsync(h->ymm, misc + off_y, npad * 8, cudaMemcpyDeviceToDevice, C().stream));
  std::vector<double> host(nblk + npad + 2);
  FIT_TRY(cudaMemcpyAsync(host.data(), misc + off_ld, (nblk + npad + 2) * 8, cudaMemcpyDeviceToHost, C().stream));
  FIT_TRY(cudaStreamSynchronize(C().stream));
  timing_end();
  int st;
  std::memcpy(&st, &host[nblk + npad], sizeof(int));
  if (st != 0) {
    bail(0);
    if (loglik_out) *loglik_out = -std::numeric_limits<double>::infinity();
    tl_err = "boss_gp_fit: kernel matrix is not positive definite";
    return BOSS_NOT_POSDEF;
  }
  double ld = 0.0, mahal = 0.0;
  for (int b = 0; b < nblk; ++b) ld += host[b];
  for (size_t k = 0; k < npad; ++k) mahal = std::fma(host[nblk + k], host[nblk + k], mahal);
  h->loglik = -((double)n * 1.8378770664093453 + 2.0 * ld + mahal) * 0.5;
  if (loglik_out) *loglik_out = h->loglik;
  h->dev = C().device;
  h->rep[h->dev] = h;
  C().live.insert(h);
  *out = h;
  return 0;
#undef FIT_TRY
}

// release one replica (its own context is entered here)
static void free_replica(boss_gp *r) {
  if (!r) return;
  Ctx *cx = ctx_of(r->dev);
  if (cx) {
    Enter en(cx);
    cx->live.erase(r);
    r->free_dev();
  }
  delete r;
}

// Tie the per-device fits of one posterior together: reps[k] is the fit on device k (all non-null, bit-identical
// because every device runs the same deterministic kernels on the same inputs).
static boss_gp *link_replicas(const std::vector<boss_gp *> &reps) {
  boss_gp *prim = reps[0];
  for (size_t k = 0; k < reps.size(); ++k) prim->rep[reps[k]->dev] = reps[k];
  return prim;
}

int boss_gp_fit(const double *X, int d, int n, const double *y_minus_mean, const double *lengthscales,
                double amplitude, double noise_std, int kernel_id, const uint8_t *discrete_mask, boss_gp **out,
                double *loglik_out) {
  if (!out) return fail(BOSS_ERR_ARG, "boss_gp_fit: out is NULL");
  *out = nullptr;
  KernelSpec ks;
  if (!decode_kernel(kernel_id, &ks)) return fail(BOSS_ERR_ARG, "boss_gp_fit: unknown kernel_id");
  if (g_ndev > 1 && tl_dev < 0) {
    // multi-device mode: the same deterministic fit on every device (2.9 GF at n = 2048 - cheaper than shipping
    // 3 x 32 MB of factors over NVLink, and it needs no peer access)
    const int nd = g_ndev;
    std::vector<boss_gp *> reps(nd, nullptr);
    std::vector<double> ll(nd, 0.0);
    int rc = for_each_device(nd, [&](int k, Ctx *) {
      return fit_single(X, d, n, y_minus_mean, lengthscales, amplitude, noise_std, ks, discrete_mask, &reps[k], &ll[k]);
    });
    if (loglik_out) *loglik_out = ll[0];
    if (rc) {
      const std::string keep = tl_err;
      for (boss_gp *r : reps) free_replica(r);
      tl_err = keep;
      return rc;
    }
    *out = link_replicas(reps);
    return 0;
  }
  REQUIRE_INIT();
  return fit_single(X, d, n, y_minus_mean, lengthscales, amplitude, noise_std, ks, discrete_mask, out, loglik_out);
}

void boss_gp_free(boss_gp *gp) {
  if (!gp) return;
  for (int k = 0; k < MAX_DEV; ++k)
    if (gp->rep[k] && gp->rep[k] != gp) free_replica(gp->rep[k]);
  free_replica(gp);
}
// Grow a handle's capacity by one 128-block (P-layout stride changes -> repack on the device).
static int grow_handle(boss_gp *h) {
  const int npad_new = h->n_pad + TM, kt_new = npad_new / TK;
  const size_t mat_new = (size_t)npad_new * npad_new;
  double *nL = nullptr, *nW = nullptr, *nWT = nullptr, *nal = nullptr, *nXt = nullptr, *nw = nullptr, *ny = nullptr;
  auto cleanup = [&]() {
    for (double *q : {nL, nW, nWT, nal, nXt, nw, ny})
      if (q) pool_free(q);
  };
#define GROW_TRY(expr)                                                                                       \
  do {                                                                                                       \
    cudaError_t _e = (expr);                                                                                 \
    if (_e != cudaSuccess) {                                                                                 \
      cleanup();                                                                                             \
      return fail(BOSS_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));                        \
    }                                                                                                        \
  } while (0)
  GROW_TRY(pool_alloc(&nL, mat_new * 8));
  GROW_TRY(pool_alloc(&nW, mat_new * 8));
  GROW_TRY(pool_alloc(&nWT, mat_new * 8));
  GROW_TRY(pool_alloc(&nal, (size_t)npad_new * 8));
  GROW_TRY(pool_alloc(&nXt, (size_t)npad_new * h->dp * 8));
  GROW_TRY(pool_alloc(&nw, (size_t)npad_new * 8));
  GROW_TRY(pool_alloc(&ny, (size_t)npad_new * 8));
  const unsigned nb = (unsigned)((mat_new + 255) / 256);
  repack_grow_kernel<<<nb, 256, 0, C().stream>>>(h->L, h->ktiles, h->n_pad, nL, kt_new, npad_new);
  repack_grow_kernel<<<nb, 256, 0, C().stream>>>(h->W, h->ktiles, h->n_pad, nW, kt_new, npad_new);
  repack_grow_kernel<<<nb, 256, 0, C().stream>>>(h->WT, h->ktiles, h->n_pad, nWT, kt_new, npad_new);
  C().launches += 3;
  struct {
    double *dst, *src;
    size_t n_new, n_old;
  } vecs[4] = {{nal, h->alpha, (size_t)npad_new, (size_t)h->n_pad},
               {nXt, h->Xt, (size_t)npad_new * h->dp, (size_t)h->n_pad * h->dp},
               {nw, h->wvec, (size_t)npad_new, (size_t)h->n_pad},
               {ny, h->ymm, (size_t)npad_new, (size_t)h->n_pad}};
  for (auto &v : vecs) {
    GROW_TRY(cudaMemsetAsync(v.dst, 0, v.n_new * 8, C().stream));
    GROW_TRY(cudaMemcpyAsync(v.dst, v.src, v.n_old * 8, cudaMemcpyDeviceToDevice, C().stream));
  }
  GROW_TRY(cudaGetLastError());
  GROW_TRY(cudaStreamSynchronize(C().stream));
#undef GROW_TRY
  for (double *q : {h->L, h->W, h->WT, h->alpha, h->Xt, h->wvec, h->ymm}) pool_free(q);
  h->L = nL; h->W = nW; h->WT = nWT; h->alpha = nal; h->Xt = nXt; h->wvec = nw; h->ymm = ny;
  h->n_pad = npad_new;
  h->nblk = npad_new / TM;
  h->ktiles = kt_new;
  return 0;
}

static int append_single(boss_gp *h, const double *x_new, double y_minus_mean_new, double *loglik_out) {
  if (!h || !x_new) return fail(BOSS_ERR_ARG, "boss_gp_append: bad arguments");
  if (h->n == h->n_pad) {
    int rc = grow_handle(h);
    if (rc) return rc;
  }
  const int n = h->n, npad = h->n_pad, d = h->d;
  // workspace: xnew[32] | kvec[npad] | l[npad] | u[npad] | sc[4] | status
  const size_t o_k = 32, o_l = o_k + npad, o_u = o_l + npad, o_sc = o_u + npad, o_st = o_sc + 4, total = o_st + 1;
  CUDA_TRY(C().chol_misc.ensure(total * 8));
  double *ws = C().chol_misc.as<double>();
  int *status = reinterpret_cast<int *>(ws + o_st);
  CUDA_TRY(cudaMemsetAsync(status, 0, 8, C().stream));
  CUDA_TRY(cudaMemcpyAsync(ws, x_new, (size_t)d * 8, cudaMemcpyHostToDevice, C().stream));
  launch_append_kvec(h->kernel_id, h->dp, ws, d, n, npad, h->invl, h->disc, h->a2, h->rq_a, h->Xt, ws + o_k, C().stream);
  matvec_p_kernel<<<npad / 64, 256, 0, C().stream>>>(h->W, ws + o_k, ws + o_l, h->ktiles);
  append_scalars_kernel<<<1, 256, 0, C().stream>>>(ws + o_l, h->wvec, n, h->a2 + h->noise * h->noise, y_minus_mean_new,
                                                 ws + o_sc, status);
  matvec_p_kernel<<<npad / 64, 256, 0, C().stream>>>(h->WT, ws + o_l, ws + o_u, h->ktiles);
  append_scatter_kernel<<<(n + 256) / 256, 256, 0, C().stream>>>(h->L, h->W, h->WT, n, h->ktiles, ws + o_l, ws + o_u,
                                                              ws + o_sc, status, h->wvec, h->ymm, y_minus_mean_new);
  C().launches += 5;
  CUDA_TRY(cudaGetLastError());
  double hs[5];
  CUDA_TRY(cudaMemcpyAsync(hs, ws + o_sc, 40, cudaMemcpyDeviceToHost, C().stream));
  CUDA_TRY(cudaStreamSynchronize(C().stream));
  int st;
  std::memcpy(&st, &hs[4], sizeof(int));
  if (st != 0) {
    if (loglik_out) *loglik_out = -std::numeric_limits<double>::infinity();
    tl_err = "boss_gp_append: the extended kernel matrix is not positive definite (handle left unchanged)";
    return BOSS_NOT_POSDEF;
  }
  h->n = n + 1;
  matvec_p_kernel<<<npad / 64, 256, 0, C().stream>>>(h->WT, h->wvec, h->alpha, h->ktiles);   // alpha = W^T w
  ++C().launches;
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaStreamSynchronize(C().stream));
  h->loglik += -0.5 * 1.8378770664093453 - std::log(hs[0]) - 0.5 * hs[1] * hs[1];
  if (loglik_out) *loglik_out = h->loglik;
  return 0;
}

int boss_gp_append(boss_gp *h, const double *x_new, double y_minus_mean_new, double *loglik_out) {
  if (!h || !x_new) return fail(BOSS_ERR_ARG, "boss_gp_append: bad arguments");
  int nrep = 0;
  for (int k = 0; k < MAX_DEV; ++k) nrep += h->rep[k] != nullptr;
  if (nrep > 1) {
    // every replica takes the same O(n^2) update; a non-positive-definite extension is detected identically on all
    // of them (same arithmetic), so the replicas stay in step
    std::vector<boss_gp *> reps;
    for (int k = 0; k < MAX_DEV; ++k)
      if (h->rep[k]) reps.push_back(h->rep[k]);
    std::vector<int> rc(reps.size(), 0);
    std::vector<std::string> err(reps.size());
    std::vector<double> ll(reps.size(), 0.0);
    std::vector<std::thread> th;
    for (size_t q = 0; q < reps.size(); ++q)
      th.emplace_back([&, q]() {
        Ctx *cx = ctx_of(reps[q]->dev);
        if (!cx) {
          rc[q] = BOSS_ERR_STATE;
          err[q] = "boss_gp_append: handle is not valid any more";
          return;
        }
        Enter en(cx);
        rc[q] = append_single(reps[q], x_new, y_minus_mean_new, &ll[q]);
        if (rc[q]) err[q] = tl_err;
      });
    for (auto &t : th) t.join();
    for (size_t q = 0; q < reps.size(); ++q)
      if (reps[q] == h && loglik_out) *loglik_out = ll[q];
    for (size_t q = 0; q < reps.size(); ++q)
      if (rc[q]) return fail(rc[q], err[q]);
    return 0;
  }
  REQUIRE_HANDLE_CTX(h);
  return append_single(h, x_new, y_minus_mean_new, loglik_out);
}

int boss_gp_n(const boss_gp *gp) { return gp ? gp->n : -1; }
int boss_gp_d(const boss_gp *gp) { return gp ? gp->d : -1; }

// ---------------------------------------------------------------------------------------------
// scoring core (shared by predict / ei_score, host- and device-pointer variants)
// ---------------------------------------------------------------------------------------------
namespace {

struct ScoreArgs {
  const boss_gp *const *slices;
  int y_dim, n_samples;
  const double *Xs;  // host or device
  long long M;
  const double *prior_mean;  // y_dim x M, host or device
  const double *coefs, *best, *y_max, *lb, *ub;  // host
  const uint8_t *cons_mask;                      // host or device
  double *acq, *grad;                            // host or device
  const double *prior_mean_grad;                 // y_dim x d x M (host or device) or null
  double *mu_out, *var_out;                      // predict mode, host or device: P x M (P = n_samples*y_dim)
  int32_t *status_out;
  double *dmu_out = nullptr, *dvar_out = nullptr; // predict mode with x-gradients (boss_gp_predict_grad): P x d x M
  double *best_val;  // host
  int64_t *best_idx; // host
  bool dev;          // arrays are device pointers
  bool want_argmax;
  int any_fail;      // out
  const CandGen *gen = nullptr;   // candidates generated on the device (Xs == NULL); other arrays are host pointers
  void *caller_stream = nullptr;  // dev == true: the stream the caller produced its device arrays on (NULL = legacy default stream)
  bool internal = false;          // dev == true from inside the library (arrays were produced on the library stream)
  const MixParams *mix = nullptr; // MC-EI for NonlinFitness expression sets (score.cuh); null = LinFitness closed form
  long long topk = 0;             // > 0: the topk best (value, index) pairs in isless order go to top_val / top_idx (host)
  double *top_val = nullptr;
  int64_t *top_idx = nullptr;
  const long long *topk_map = nullptr;   // device, or null: returned indices are topk_map[i] (the screened pool's origins)

  // boss_gp_predict_grad: the posterior gradients themselves are the output (predict_grad_kernel)
  bool pgrad() const { return dmu_out || dvar_out; }
  // the x-gradient pipeline runs (V^T store, wtv, grad, grad_reduce): for the acquisition or for the posteriors
  bool xgrad() const { return grad || pgrad(); }
};

// Julia's isless order on (value, index): NaN maximal, -0.0 < +0.0, ties -> lowest index (host twin of acq_better)
bool acq_better_host(double va, long long ia, double vb, long long ib) {
  const bool na = va != va, nb = vb != vb;
  if (na || nb) {
    if (na && nb) return ia < ib;
    return na;
  }
  if (va > vb) return true;
  if (va < vb) return false;
  long long ba, bb;
  std::memcpy(&ba, &va, 8);
  std::memcpy(&bb, &vb, 8);
  if (ba != bb) return ba >= 0 && bb < 0;
  return ia < ib;
}

// order the library stream after whatever the caller enqueued on `caller_stream` (its device inputs)
int wait_for_caller(void *caller_stream) {
  cudaStream_t cs = caller_stream ? (cudaStream_t)caller_stream : cudaStreamLegacy;
  CUDA_TRY(cudaEventRecord(C().caller_ev, cs));
  CUDA_TRY(cudaStreamWaitEvent(C().stream, C().caller_ev, 0));
  return 0;
}

bool is_pinned_host(const void *p) {
  if (!p) return false;
  cudaPointerAttributes at{};
  if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return at.type == cudaMemoryTypeHost;
}

// offset of the next `bytes` in a buffer carved in 256-byte aligned pieces, `tot` bytes so far
size_t take(size_t &tot, size_t bytes) {
  const size_t o = tot;
  tot += (bytes + 255) / 256 * 256;
  return o;
}

// the one place an XcovParams is filled: slice h against the candidates xs (candidate m in column m - in_off), the
// partials of the chunk that starts at m0 with leading dimension ld
XcovParams xcov_params(const boss_gp *h, const double *xs, long long M, long long m0, long long in_off, int d, int ld) {
  XcovParams xp{};
  xp.Xs = xs;
  xp.M = M;
  xp.m0 = m0;
  xp.in_off = in_off;
  xp.d = d;
  xp.n = h->n;
  xp.n_pad = h->n_pad;
  xp.ktiles = h->ktiles;
  xp.Xt = h->Xt;
  xp.invl = h->invl;
  xp.disc_bits = h->disc;
  xp.alpha = h->alpha;
  xp.a2 = h->a2;
  xp.Ks = C().ks.as<double>();
  xp.mu_part = C().part_mu.as<double>();
  xp.ld = ld;
  xp.rq_a = h->rq_a;
  return xp;
}

// device arrays of one chunk: candidate m of the call is at position m - off of each
struct ChunkIO {
  const double *xs = nullptr, *pm = nullptr, *pmg = nullptr;
  const unsigned char *cm = nullptr;
  double *acq = nullptr, *mu = nullptr, *var = nullptr, *grad = nullptr;
  int *st = nullptr;
  long long off = 0;
  double *dmu = nullptr, *dvar = nullptr;
};

// Host <-> device staging of a chunked call with HOST arrays.  The caller's arrays are ordinary pageable memory in
// the drop-in case (a Julia Matrix{Float64}); a cudaMemcpyAsync from pageable memory first drains the stream and then
// copies synchronously, so the GPU would idle during every chunk's transfer.  Instead each chunk's inputs go through
// one of two pinned slots (host memcpy -> DMA on a copy stream) into one of two device slots while the previous chunk
// computes, and the outputs of chunk c are copied out of their pinned slot while chunk c+1 runs.
struct HostStaging {
  const ScoreArgs *a = nullptr;   // null: the call has no host arrays
  int d = 0, CH = 0;
  bool has_pmg = false;
  bool xs_direct = false;   // the caller's candidate matrix is pinned already: DMA straight from it
  // byte offsets of every array inside a slot
  size_t in_xs = 0, in_pm = 0, in_cm = 0, in_pmg = 0, in_total = 0;
  size_t out_acq = 0, out_mu = 0, out_var = 0, out_st = 0, out_gr = 0, out_dmu = 0, out_dvar = 0, out_total = 0;
  int P = 1;   // posteriors per candidate in the predict outputs (1 for boss_gp_predict)
  unsigned char *pin_in[2] = {}, *pin_out[2] = {}, *dev_in[2] = {}, *dev_out[2] = {};
  cudaStream_t cp = C().ll_stream[LL_GROUPS - 1];   // copy stream (the last log-likelihood group stream is idle here)
  cudaEvent_t ev_in[2] = {C().ll_join[LL_GROUPS - 1], C().ll_join[LL_GROUPS - 2]};     // H2D of the slot done
  cudaEvent_t ev_free[2] = {C().ll_join[LL_GROUPS - 3], C().ll_join[LL_GROUPS - 4]};   // compute done with the device slot
  cudaEvent_t ev_out[2] = {C().pin_ev[0], C().pin_ev[1]};                              // outputs of the slot are in pinned memory
  bool in_used[2] = {false, false}, free_rec[2] = {false, false};
  long long prev_m0 = -1;      // the chunk whose outputs wait in their pinned slot
  int prev_ch = 0, prev_slot = 0;

  int plan(const ScoreArgs &args, int ch_cap, int dim) {
    a = &args;
    CH = ch_cap;
    d = dim;
    P = a->y_dim * a->n_samples;
    has_pmg = a->xgrad() && a->prior_mean_grad;
    xs_direct = !a->gen && is_pinned_host(a->Xs);
    in_xs = take(in_total, (size_t)CH * d * 8);   // device slot always holds the candidates
    if (a->prior_mean) in_pm = take(in_total, (size_t)CH * a->y_dim * 8);
    if (a->cons_mask) in_cm = take(in_total, (size_t)CH);
    if (has_pmg) in_pmg = take(in_total, (size_t)CH * d * a->y_dim * 8);
    if (a->acq) out_acq = take(out_total, (size_t)CH * 8);
    if (a->mu_out) out_mu = take(out_total, (size_t)P * CH * 8);
    if (a->var_out) out_var = take(out_total, (size_t)P * CH * 8);
    if (a->status_out) out_st = take(out_total, (size_t)P * CH * 4);
    if (a->grad) out_gr = take(out_total, (size_t)CH * d * 8);
    if (a->dmu_out) out_dmu = take(out_total, (size_t)P * d * CH * 8);
    if (a->dvar_out) out_dvar = take(out_total, (size_t)P * d * CH * 8);
    const size_t out_slot = std::max<size_t>(out_total, 256);
    CUDA_TRY(C().xs_stage.ensure(2 * in_total));    // both device input slots
    CUDA_TRY(C().acq_stage.ensure(2 * out_slot));   // both device output slots
    const size_t need = 2 * (in_total + out_total) + 256;   // both pinned input and output slots
    if (need > C().pinned_cap) {
      if (C().pinned) cudaFreeHost(C().pinned);
      C().pinned = nullptr;
      C().pinned_cap = 0;
      CUDA_TRY(cudaHostAlloc(&C().pinned, need + need / 4, cudaHostAllocDefault));
      C().pinned_cap = need + need / 4;
    }
    unsigned char *pin = reinterpret_cast<unsigned char *>(C().pinned);
    pin_in[0] = pin;
    pin_in[1] = pin + in_total;
    pin_out[0] = pin + 2 * in_total;
    pin_out[1] = pin + 2 * in_total + out_total;
    dev_in[0] = C().xs_stage.as<unsigned char>();
    dev_in[1] = dev_in[0] + in_total;
    dev_out[0] = C().acq_stage.as<unsigned char>();
    dev_out[1] = dev_out[0] + out_slot;
    return 0;
  }

  // device arrays of chunk [m0, m0 + ch) in `slot`: its inputs were staged while the previous chunk was being launched
  // (the first chunk's are staged here), generated candidates are written into the slot now
  int chunk_inputs(long long m0, int ch, int slot, ChunkIO &io) {
    if (m0 == 0) {
      CUDA_TRY(cudaEventRecord(ev_free[0], C().stream));   // nothing enqueued before this point reads the slots
      int rc = stage_in(0, ch, 0);
      if (rc) return rc;
    }
    CUDA_TRY(cudaStreamWaitEvent(C().stream, ev_in[slot], 0));
    io.xs = reinterpret_cast<const double *>(dev_in[slot] + in_xs);
    if (a->gen) {
      gen_candidates_kernel<<<(ch * d + 255) / 256, 256, 0, C().stream>>>(*a->gen, m0, ch, const_cast<double *>(io.xs));
      ++C().launches;
    }
    if (a->prior_mean) io.pm = reinterpret_cast<const double *>(dev_in[slot] + in_pm);
    if (a->cons_mask) io.cm = dev_in[slot] + in_cm;
    if (has_pmg) io.pmg = reinterpret_cast<const double *>(dev_in[slot] + in_pmg);
    io.off = m0;   // the slot arrays start at the chunk's first candidate
    if (a->acq) io.acq = reinterpret_cast<double *>(dev_out[slot] + out_acq);
    if (a->mu_out) io.mu = reinterpret_cast<double *>(dev_out[slot] + out_mu);
    if (a->var_out) io.var = reinterpret_cast<double *>(dev_out[slot] + out_var);
    if (a->status_out) io.st = reinterpret_cast<int *>(dev_out[slot] + out_st);
    if (a->grad) io.grad = reinterpret_cast<double *>(dev_out[slot] + out_gr);
    if (a->dmu_out) io.dmu = reinterpret_cast<double *>(dev_out[slot] + out_dmu);
    if (a->dvar_out) io.dvar = reinterpret_cast<double *>(dev_out[slot] + out_dvar);
    return 0;
  }

  // after the chunk's kernels have been enqueued: its outputs go to their pinned slot, and while the chunk runs the next
  // chunk's inputs are staged and the previous chunk's outputs are handed to the caller
  int end_chunk(long long m0, int ch, int slot) {
    CUDA_TRY(cudaEventRecord(ev_free[slot], C().stream));   // the kernels above were the last readers of the input slot
    free_rec[slot] = true;
    if (out_total) {
      CUDA_TRY(cudaMemcpyAsync(pin_out[slot], dev_out[slot], out_total, cudaMemcpyDeviceToHost, C().stream));
      CUDA_TRY(cudaEventRecord(ev_out[slot], C().stream));
    }
    if (m0 + CH < a->M) {
      int rc = stage_in(m0 + CH, (int)std::min<long long>(CH, a->M - m0 - CH), slot ^ 1);
      if (rc) return rc;
    }
    if (prev_m0 >= 0) {
      int rc = drain_out(prev_m0, prev_ch, prev_slot);
      if (rc) return rc;
    }
    prev_m0 = m0;
    prev_ch = ch;
    prev_slot = slot;
    return 0;
  }

  // once the stream has drained: the copy stream is idle and the last chunk's outputs (their event has completed by
  // then) go to the caller.  Nothing to do for device arrays.
  int drain_last() {
    if (!a) return 0;
    CUDA_TRY(cudaStreamSynchronize(cp));
    return prev_m0 >= 0 ? drain_out(prev_m0, prev_ch, prev_slot) : 0;
  }

 private:
  // inputs of chunk [m0, m0 + ch) -> device slot; returns after the copies have been ENQUEUED on the copy stream
  int stage_in(long long m0, int ch, int slot) {
    if (in_used[slot]) CUDA_TRY(cudaEventSynchronize(ev_in[slot]));   // the pinned slot's previous DMA has completed
    if (free_rec[slot]) CUDA_TRY(cudaStreamWaitEvent(cp, ev_free[slot], 0));   // kernels of chunk c-2 are done with the device slot
    unsigned char *pin = pin_in[slot], *dv = dev_in[slot];
    auto put = [&](size_t off, const void *src, size_t bytes) {   // host array -> pinned slot -> device slot
      std::memcpy(pin + off, src, bytes);
      return cudaMemcpyAsync(dv + off, pin + off, bytes, cudaMemcpyHostToDevice, cp);
    };
    if (!a->gen) {
      const double *src = a->Xs + (size_t)m0 * d;
      if (xs_direct)
        CUDA_TRY(cudaMemcpyAsync(dv + in_xs, src, (size_t)ch * d * 8, cudaMemcpyHostToDevice, cp));
      else
        CUDA_TRY(put(in_xs, src, (size_t)ch * d * 8));
    }
    if (a->prior_mean) CUDA_TRY(put(in_pm, a->prior_mean + (size_t)m0 * a->y_dim, (size_t)ch * a->y_dim * 8));
    if (a->cons_mask) CUDA_TRY(put(in_cm, a->cons_mask + m0, (size_t)ch));
    if (has_pmg) CUDA_TRY(put(in_pmg, a->prior_mean_grad + (size_t)m0 * d * a->y_dim, (size_t)ch * d * a->y_dim * 8));
    CUDA_TRY(cudaEventRecord(ev_in[slot], cp));
    in_used[slot] = true;
    return 0;
  }
  // outputs of chunk [m0, m0 + ch): pinned slot -> the caller's arrays (after the chunk's D2H has completed)
  int drain_out(long long m0, int ch, int slot) {
    if (out_total == 0) return 0;
    CUDA_TRY(cudaEventSynchronize(ev_out[slot]));
    const unsigned char *pin = pin_out[slot];
    if (a->acq) std::memcpy(a->acq + m0, pin + out_acq, (size_t)ch * 8);
    if (a->mu_out) std::memcpy(a->mu_out + (size_t)m0 * P, pin + out_mu, (size_t)ch * P * 8);
    if (a->var_out) std::memcpy(a->var_out + (size_t)m0 * P, pin + out_var, (size_t)ch * P * 8);
    if (a->status_out) std::memcpy(a->status_out + (size_t)m0 * P, pin + out_st, (size_t)ch * P * 4);
    if (a->grad) std::memcpy(a->grad + (size_t)m0 * d, pin + out_gr, (size_t)ch * d * 8);
    if (a->dmu_out) std::memcpy(a->dmu_out + (size_t)m0 * d * P, pin + out_dmu, (size_t)ch * d * P * 8);
    if (a->dvar_out) std::memcpy(a->dvar_out + (size_t)m0 * d * P, pin + out_dvar, (size_t)ch * d * P * 8);
    return 0;
  }
};

// boss_gp_predict_grad: the chunk is capped so that one output slot (P x M values, P x d x M gradients, pinned and on
// the device, two of each) stays within this budget; at P = 16, d = 32 that is 246 candidate blocks instead of 296
constexpr size_t PGRAD_SLOT_BYTES = (size_t)256 << 20;

// What every stage of one scoring call reads: its arguments, the slices' replicas on this device, the chunk capacity
// and the small block of per-call device scalars.
struct ScoreCall {
  ScoreArgs &a;
  std::vector<const boss_gp *> sl;
  int nsl = 0, d = 0, CH = 0;
  bool have_vt = false;
  // small: a2[nsl] | lb[d] | ub[d] | best(1) | bidx(1 as int64) | any_fail(int) | finished-CTA counter (fused epilogue)
  std::vector<double> hs;   // host image of the small block
  double *small = nullptr, *d_best = nullptr;
  long long *d_bidx = nullptr;
  int *d_anyfail = nullptr;
  unsigned int *d_counter = nullptr;
  MixParams mixp{};

  explicit ScoreCall(ScoreArgs &args) : a(args) {}

  // the replicas of the slices on this context's device
  int bind() {
    nsl = a.y_dim * a.n_samples;
    if (nsl < 1 || a.y_dim > MAX_YDIM) return fail(BOSS_ERR_ARG, "score: y_dim must be in 1..16");
    sl.resize(nsl);
    for (int q = 0; q < nsl; ++q) {
      if (!a.slices[q]) return fail(BOSS_ERR_ARG, "score: NULL slice handle");
      sl[q] = replica_on(a.slices[q], C().device);
      if (!sl[q]) return fail(BOSS_ERR_STATE, "score: a slice handle has no replica on this device (or was invalidated by boss_shutdown)");
      if (sl[q]->d != sl[0]->d) return fail(BOSS_ERR_ARG, "score: slices disagree on x_dim");
    }
    d = sl[0]->d;
    return 0;
  }

  // chunk size, workspaces, the small block and the MC-EI eps matrix on the device
  int setup() {
    int max_npad = 0;
    for (int q = 0; q < nsl; ++q) max_npad = std::max(max_npad, sl[q]->n_pad);
    // chunk size: K*^T scratch budget 4 GiB, at most 4 waves of 148 CTAs
    long long ncb_max = (4ll << 30) / (1024ll * max_npad);
    ncb_max = std::min<long long>(ncb_max, 592);
    if (ncb_max >= 148) ncb_max = ncb_max / 148 * 148;
    if (ncb_max < 1) return fail(BOSS_ERR_ARG, "score: n too large for the scratch budget");
    if (a.xgrad()) ncb_max = std::max<long long>(1, std::min<long long>(ncb_max, ncb_max >= 296 ? 296 : ncb_max));
    if (a.pgrad()) {   // one output slot (pinned and device) within PGRAD_SLOT_BYTES (DESIGN.md 2.12)
      const long long per_block = 128ll * nsl * (20 + 16ll * d);   // mu, var, status, dmu, dvar of 128 candidates
      ncb_max = std::max<long long>(1, std::min<long long>(ncb_max, (long long)(PGRAD_SLOT_BYTES / per_block)));
    }
    const long long need_cb = (a.M + 127) / 128;
    const int ncb_cap = (int)std::min<long long>(ncb_max, need_cb);
    CH = ncb_cap * 128;

    CUDA_TRY(C().ks.ensure((size_t)CH * max_npad * 8));
    CUDA_TRY(C().muv.ensure((size_t)nsl * CH * 8));
    CUDA_TRY(C().sumsq.ensure((size_t)nsl * CH * 8));
    const int max_nblk = max_npad / TM;
    CUDA_TRY(C().part_mu.ensure((size_t)2 * max_nblk * CH * 8));
    CUDA_TRY(C().part_ss.ensure((size_t)2 * max_nblk * CH * 8));
    // batches up to 8192 candidates keep V^T even without gradients: the quarter-row kernels (10 % faster than the
    // row-split wide kernels up to there) reduce the variance from the stored tile
    have_vt = a.xgrad() || CH <= 8192;
    if (have_vt && !a.xgrad()) CUDA_TRY(C().vt.ensure((size_t)CH * max_npad * 8));
    if (a.xgrad()) {
      if (d > 32) return fail(BOSS_ERR_ARG, "score: gradients need x_dim <= 32");
      CUDA_TRY(C().vt.ensure((size_t)CH * max_npad * 8));
      CUDA_TRY(C().ut.ensure((size_t)CH * max_npad * 8));
      CUDA_TRY(C().dmu.ensure((size_t)nsl * d * CH * 8));
      CUDA_TRY(C().dvar.ensure((size_t)nsl * d * CH * 8));
      CUDA_TRY(C().part_gm.ensure((size_t)2 * max_nblk * d * CH * 8));
      CUDA_TRY(C().part_gv.ensure((size_t)2 * max_nblk * d * CH * 8));
    }
    const int nblk_acq_max = (CH + 127) / 128;     // block winners: per 256 candidates (acq_kernel) or per 128 (fused epilogue)
    CUDA_TRY(C().blk_val.ensure((size_t)nblk_acq_max * 8));
    CUDA_TRY(C().blk_idx.ensure((size_t)nblk_acq_max * 8));
    const size_t sm_n = (size_t)nsl + 2 * d + 5;
    CUDA_TRY(C().small.ensure(sm_n * 8));
    small = C().small.as<double>();
    hs.assign(sm_n, 0.0);
    for (int q = 0; q < nsl; ++q) hs[q] = sl[q]->a2;
    if (a.lb && a.ub) {
      for (int i = 0; i < d; ++i) {
        hs[nsl + i] = a.lb[i];
        hs[nsl + d + i] = a.ub[i];
      }
    }
    long long neg1 = -1;
    std::memcpy(&hs[nsl + 2 * d + 1], &neg1, 8);
    int rc = upload_small();
    if (rc) return rc;
    d_best = small + nsl + 2 * d;
    d_bidx = reinterpret_cast<long long *>(small + nsl + 2 * d + 1);
    d_anyfail = reinterpret_cast<int *>(small + nsl + 2 * d + 2);
    d_counter = reinterpret_cast<unsigned int *>(small + nsl + 2 * d + 3);
    if (a.mix) {   // MC-EI: the eps matrix (y_dim x n_eps) goes to the device once per call
      mixp = *a.mix;
      if (!mixp.eps) {   // already on the device: the multi-start driver uploads it once per solve
        const size_t eb = (size_t)a.y_dim * mixp.n_eps * 8;
        CUDA_TRY(C().tt.ensure(eb));
        CUDA_TRY(cudaMemcpyAsync(C().tt.p, mixp.eps_host, eb, cudaMemcpyHostToDevice, C().stream));
        CUDA_TRY(cudaStreamSynchronize(C().stream));
        mixp.eps = C().tt.as<double>();
      }
    }
    return 0;
  }

  // hs is pageable: the runtime has copied these few bytes to its staging memory when the call returns (CUDA's
  // documented behaviour for pageable-to-device cudaMemcpyAsync), and hs lives until the end of the call: no stream
  // round trip is needed here
  int upload_small() const {
    CUDA_TRY(cudaMemcpyAsync(small, hs.data(), hs.size() * 8, cudaMemcpyHostToDevice, C().stream));
    return 0;
  }

  AcqParams acq_params(long long m0, int ch, const ChunkIO &io) const {
    AcqParams ap{};
    ap.y_dim = a.y_dim;
    ap.n_samples = a.n_samples;
    ap.d = d;
    ap.M = a.M;
    ap.m0 = m0;
    ap.in_off = io.off;
    ap.out_off = io.off;
    ap.chunk = ch;
    ap.chunk_ld = CH;
    ap.mu = C().muv.as<double>();
    ap.sumsq = C().sumsq.as<double>();
    ap.a2 = small;
    ap.prior_mean = io.pm;
    for (int i = 0; i < a.y_dim; ++i) {
      ap.coefs[i] = a.coefs ? a.coefs[i] : (i == 0 ? 1.0 : 0.0);
      ap.y_max[i] = a.y_max ? a.y_max[i] : INFINITY;
    }
    ap.has_best = a.best != nullptr;
    ap.best = a.best ? *a.best : 0.0;
    ap.has_ymax = a.y_max != nullptr;
    ap.Xs = io.xs;
    ap.lb = (a.lb && a.ub) ? small + nsl : nullptr;
    ap.ub = (a.lb && a.ub) ? small + nsl + d : nullptr;
    ap.cons_mask = io.cm;
    ap.acq = io.acq;
    if (!a.pgrad()) {   // predict_grad_kernel writes boss_gp_predict_grad's P x M layout
      ap.mu_out = io.mu;
      ap.var_out = io.var;
      ap.status_out = io.st;
    }
    ap.any_fail = d_anyfail;
    ap.blk_val = a.want_argmax ? C().blk_val.as<double>() : nullptr;
    ap.blk_idx = a.want_argmax ? C().blk_idx.as<long long>() : nullptr;
    ap.mix = mixp;
    return ap;
  }
};

// Slice q of one chunk on the full path: mean partials and K*^T (xcov), the triangular product, the reductions and,
// with gradients, the gradient launches.  Returns whether the scoring kernel finished the chunk itself (fused epilogue).
bool score_slice(const ScoreCall &c, int q, const AcqParams &ap, const ChunkIO &io) {
  const ScoreArgs &a = c.a;
  const boss_gp *h = c.sl[q];
  const int CH = c.CH, d = c.d, ch = ap.chunk, ncb = (ch + 127) / 128;
  // Small candidate batches (multi-start optimiser iterations, single-point calls) cannot fill 148 SMs
  // with one CTA per 128 candidates: deal the training chunks / W row blocks of a candidate block to
  // several CTAs.  Partial sums are kept per chunk / per row block, so results do not depend on the split.
  const int want = (16 * 148 + ncb - 1) / ncb;   // >= 16 CTAs per SM in flight over the launch (4 waves of 4)
  const int nks = std::max(1, std::min(h->nblk, want));            // xcov / grad: splits over training chunks
  double cost_w = 0.0, cost_n = 0.0;
  const int nsp = pick_row_splits(ncb, h->nblk, &cost_w);          // trmm / wtv: zig-zag row-block splits
  // Small batches: 32-candidate CTAs (score_narrow.cuh) do a quarter of the tensor work per stage of W; worth it
  // when the wide launch cannot fill the GPU (cost = waves x longest per-CTA share, in block-steps; a narrow stage
  // takes ~0.3 of a wide one).  Same bits either way.
  const int ncb32 = (ch + NW_NB - 1) / NW_NB;
  const int nsp32 = pick_row_splits(ncb32, h->nblk, &cost_n);
  bool narrow = 0.32 * cost_n < cost_w;
  // Tiny batches: quarter-row-block CTAs (4 nblk per 32 candidates, 4 to an SM).  Cost in the same unit: the
  // longest CTA's latency-bound walk over 8 nblk short stages, or the launch's tensor work spread over the SMs.
  const double cost_q = std::max(NQ_COST_CHAIN * h->nblk, NQ_COST_WORK * ncb32 * (h->nblk * (h->nblk + 1) / 2)) + NQ_COST_FIXED;
  bool quarter = c.have_vt && cost_q < std::min(cost_w, narrow ? 0.32 * cost_n : cost_w) && h->nblk >= 2;
  if (const char *e = getenv("BOSS_SCORE_PATH")) {   // A/B switch: wide | narrow | quarter
    if (!strcmp(e, "wide")) narrow = quarter = false;
    if (!strcmp(e, "narrow")) narrow = true, quarter = false;
    if (!strcmp(e, "quarter") && c.have_vt) quarter = true;
  }
  if (quarter) narrow = false;
  const int cnt = ncb * 128;
  {
    Timed t(1);
    launch_xcov(h->kernel_id, h->dp, xcov_params(h, io.xs, a.M, ap.m0, io.off, d, CH), dim3(ncb, nks), C().stream);
  }
  // One CTA per candidate block walks all of W (large batches) and this is the chunk's last slice: the scoring
  // kernel finishes the candidates itself (fused epilogue) -- no reduce / acquisition / argmax launches.
  const bool fuse = nsp == 1 && !narrow && !quarter && q == c.nsl - 1 && getenv("BOSS_UNFUSED_SCORE") == nullptr;
  ++C().score_paths[quarter ? 3 : narrow ? 2 : fuse ? 0 : 1];
  if (a.xgrad()) ++C().score_paths[4];
  if (!fuse && !quarter)
    reduce_rows_kernel<<<(cnt + 255) / 256, 256, 0, C().stream>>>(C().part_mu.as<double>(), 2 * h->nblk, (size_t)CH,
                                                               C().muv.as<double>() + (size_t)q * CH, cnt);
  ScoreParams sp{};
  sp.W = h->W;
  sp.Ks = C().ks.as<double>();
  sp.nblk = h->nblk;
  sp.ktiles = h->ktiles;
  sp.ss_part = C().part_ss.as<double>();
  sp.ld = CH;
  sp.VT = a.xgrad() ? C().vt.as<double>() : nullptr;
  if (fuse) {
    sp.fused = 1;
    sp.ap = ap;
    sp.mu_part = C().part_mu.as<double>();
    sp.P = 2 * h->nblk;
    sp.mu_row = C().muv.as<double>() + (size_t)q * CH;
    sp.ss_row = C().sumsq.as<double>() + (size_t)q * CH;
    sp.best = c.d_best;
    sp.bidx = c.d_bidx;
    sp.counter = c.d_counter;
  }
  if (quarter) {
    NarrowParams np{h->W, C().ks.as<double>(), h->nblk, h->ktiles, nullptr, CH, C().vt.as<double>()};
    Timed t(0);
    score_quarter_kernel<0, 4, 1><<<dim3(ncb32, 4 * h->nblk), NQ_THREADS, NQ_SMEM_BYTES, C().stream>>>(np);
    quarter_sumsq_kernel<<<dim3(ncb32, h->nblk), 256, 0, C().stream>>>(C().vt.as<double>(), h->ktiles,
                                                                     C().part_ss.as<double>(), CH);
  } else if (narrow) {
    NarrowParams np{h->W, C().ks.as<double>(), h->nblk, h->ktiles, C().part_ss.as<double>(), CH,
                    a.xgrad() ? C().vt.as<double>() : nullptr};
    Timed t(0);
    score_narrow_kernel<0><<<dim3(ncb32, nsp32), 256, NW_SMEM_BYTES, C().stream>>>(np);
  } else {
    Timed t(0);
    score_trmm_kernel<<<dim3(ncb, nsp), GEMM_THREADS, GEMM_SMEM_BYTES, C().stream>>>(sp);
  }
  if (quarter)   // mu partials (xcov) and sums of squares (quarter_sumsq) of this slice in one launch
    reduce_rows_pair_kernel<<<dim3((cnt + 255) / 256, 2), 256, 0, C().stream>>>(
        C().part_mu.as<double>(), C().part_ss.as<double>(), 2 * h->nblk, (size_t)CH, C().muv.as<double>() + (size_t)q * CH,
        C().sumsq.as<double>() + (size_t)q * CH, cnt);
  else if (!fuse)
    reduce_rows2_kernel<<<(cnt + 255) / 256, 256, 0, C().stream>>>(C().part_ss.as<double>(), 2 * h->nblk, (size_t)CH,
                                                                C().sumsq.as<double>() + (size_t)q * CH, cnt);
  C().launches += fuse ? 2 : 4;
  if (a.xgrad()) {
    WtvParams wp{h->WT, C().vt.as<double>(), C().ut.as<double>(), h->nblk, h->ktiles};
    NarrowParams np{h->WT, C().vt.as<double>(), h->nblk, h->ktiles, nullptr, CH, C().ut.as<double>()};
    if (quarter) {
      Timed t(0);
      score_quarter_kernel<1, 4, 1><<<dim3(ncb32, 4 * h->nblk), NQ_THREADS, NQ_SMEM_BYTES, C().stream>>>(np);
    } else if (narrow) {
      Timed t(0);
      score_narrow_kernel<1><<<dim3(ncb32, nsp32), 256, NW_SMEM_BYTES, C().stream>>>(np);
    } else {
      Timed t(0);
      wtv_kernel<<<dim3(ncb, nsp), GEMM_THREADS, GEMM_SMEM_BYTES, C().stream>>>(wp);
    }
    GradParams gq{};
    gq.Xs = io.xs;
    gq.M = a.M;
    gq.m0 = ap.m0;
    gq.in_off = io.off;
    gq.d = d;
    gq.n = h->n;
    gq.n_pad = h->n_pad;
    gq.ktiles = h->ktiles;
    gq.chunk_ld = CH;
    gq.Xt = h->Xt;
    gq.invl = h->invl;
    gq.alpha = h->alpha;
    gq.disc_bits = h->disc;
    gq.a2 = h->a2;
    gq.UT = C().ut.as<double>();
    gq.gm_part = C().part_gm.as<double>();
    gq.gv_part = C().part_gv.as<double>();
    gq.rq_a = h->rq_a;
    {
      Timed t(1);
      launch_grad(h->kernel_id, h->dp, gq, dim3(ncb, nks), C().stream);
    }
    GradReduceParams gr{C().part_gm.as<double>(), C().part_gv.as<double>(), 2 * h->nblk, d, CH, cnt, h->invl, h->disc,
                        C().dmu.as<double>() + (size_t)q * d * CH, C().dvar.as<double>() + (size_t)q * d * CH};
    grad_reduce_kernel<<<dim3((cnt + 255) / 256, d), 256, 0, C().stream>>>(gr);
    C().launches += 3;
  }
  return fuse;
}

// seed batch of a screened top-k call: the S_k highest bounds of the first chunk, S_k = 2k rounded up to 128, at least
// SEED_N and at most the chunk (DESIGN.md 2.10)
int topk_seed_n(long long k, int ch) {
  return (int)std::min<long long>(ch, std::max<long long>(SEED_N, (2 * k + 127) / 128 * 128));
}

// device buffers of a top-k call (topk.cuh): two running sets of `cap` pairs, the chunk's scores, the selection state
// and per-256 counts, the sorted result.  Sized by the outermost call; score_subset checks that the nested seed and pool
// calls fit inside.
struct TopkBufs {
  double *run_val[2] = {}, *scores = nullptr, *out_val = nullptr;
  long long *run_idx[2] = {}, *out_idx = nullptr;
  SelectState *st = nullptr;
  int2 *cnt = nullptr;
  long long k = 0;
  int r = 0, par = 0;   // the running set: r pairs in run_*[par]
  int setup(long long k_, int CH, int ch0) {
    k = k_;
    const int cap = (int)std::max<long long>(k, topk_seed_n(k, ch0));
    size_t tot = 0;
    const size_t o_rv0 = take(tot, (size_t)cap * 8), o_rv1 = take(tot, (size_t)cap * 8), o_ri0 = take(tot, (size_t)cap * 8),
                 o_ri1 = take(tot, (size_t)cap * 8), o_sc = take(tot, (size_t)CH * 8), o_st = take(tot, sizeof(SelectState)),
                 o_cnt = take(tot, ((size_t)cap + CH + 255) / 256 * sizeof(int2)), o_ov = take(tot, (size_t)k * 8),
                 o_oi = take(tot, (size_t)k * 8);
    CUDA_TRY(C().topk.ensure(tot));
    unsigned char *b = C().topk.as<unsigned char>();
    run_val[0] = reinterpret_cast<double *>(b + o_rv0);
    run_val[1] = reinterpret_cast<double *>(b + o_rv1);
    run_idx[0] = reinterpret_cast<long long *>(b + o_ri0);
    run_idx[1] = reinterpret_cast<long long *>(b + o_ri1);
    scores = reinterpret_cast<double *>(b + o_sc);
    st = reinterpret_cast<SelectState *>(b + o_st);
    cnt = reinterpret_cast<int2 *>(b + o_cnt);
    out_val = reinterpret_cast<double *>(b + o_ov);
    out_idx = reinterpret_cast<long long *>(b + o_oi);
    return 0;
  }
  // the `target` best of (in's running set, in's new values) -> out, in ascending index order (topk.cuh)
  int select(const SelectIn &in, int target, double *out_val_, long long *out_idx_) {
    const int N = in.r + in.n;
    if (N < 1 || target < 1) return 0;
    select_init_kernel<<<1, 256, 0, C().stream>>>(st, target >= N ? N : target);
    ++C().launches;
    if (target < N) {
      const int gh = std::min((N + 255) / 256, 8 * 148);
      for (int shift = 56; shift >= 0; shift -= 8) {
        select_hist_kernel<<<gh, 256, 0, C().stream>>>(in, st, shift);
        select_scan_kernel<<<1, 256, 0, C().stream>>>(st, shift);
      }
      C().launches += 16;
    }
    const int nb = (N + 255) / 256;
    select_count_kernel<<<nb, 256, 0, C().stream>>>(in, st, cnt);
    select_compact_kernel<<<nb, 256, 0, C().stream>>>(in, st, cnt, out_val_, out_idx_);
    C().launches += 2;
    return 0;
  }
  // the running set becomes the best min(k, seen) of (running set, the chunk's scores)
  int absorb(long long m0, int ch) {
    const int tgt = (int)std::min<long long>(k, (long long)r + ch);
    SelectIn in{run_val[par], run_idx[par], r, scores, m0, ch, 0};
    int rc = select(in, tgt, run_val[par ^ 1], run_idx[par ^ 1]);
    if (rc) return rc;
    par ^= 1;
    r = tgt;
    return 0;
  }
  // the running set, sorted in one CTA, to the caller: k pairs (indices through `map` unless null), no M-sized output
  // and no host sort.  The copies are enqueued; the caller synchronises.
  int finish(const long long *map, double *top_val, int64_t *top_idx) {
    if (r != k) return fail(BOSS_ERR_STATE, "score: top-k set incomplete");
    int P = 2;
    while (P < r) P <<= 1;
    topk_sort_kernel<<<1, 1024, (size_t)P * 12, C().stream>>>(run_val[par], run_idx[par], r, P, map, out_val, out_idx);
    ++C().launches;
    CUDA_TRY(cudaMemcpyAsync(top_val, out_val, (size_t)r * 8, cudaMemcpyDeviceToHost, C().stream));
    CUDA_TRY(cudaMemcpyAsync(top_idx, out_idx, (size_t)r * 8, cudaMemcpyDeviceToHost, C().stream));
    return 0;
  }
};

int score_core(ScoreArgs &a);

// what a nested call returns besides the top-k pairs
struct SubsetResult {
  double best_val = 0.0;
  int64_t best_idx = -1;
  int any_fail = 0;
};

// Every nested call of a screened call: scores M candidates that the library wrote to device memory on its stream (the
// seed batch or the survivor pool) with the model and acquisition of c's call, top-k pairs to top_val / top_idx with
// indices through topk_map.  The nested call rewrites the small block, so restore_small puts c's back when the outer
// call goes on using it.  The outer call holds raw pointers into the small block, the top-k buffers and the screening
// buffers: a nested call that grew one of them would leave those pointers dangling, so that is an error.
int score_subset(const ScoreCall &c, const double *x, const double *pm, const unsigned char *cm, long long M,
                 double *top_val, int64_t *top_idx, const long long *topk_map, bool restore_small, SubsetResult &r) {
  const size_t held[4] = {C().small.cap, C().topk.cap, C().scr_misc.cap, C().scr_pool.cap};
  ScoreArgs s = c.a;
  s.Xs = x;
  s.M = M;
  s.prior_mean = pm;
  s.cons_mask = cm;
  s.gen = nullptr;
  s.dev = true;
  s.internal = true;
  s.best_val = &r.best_val;
  s.best_idx = &r.best_idx;
  s.top_val = top_val;
  s.top_idx = top_idx;
  s.topk_map = topk_map;
  int rc = score_core(s);
  if (rc) return rc;
  if (held[0] != C().small.cap || held[1] != C().topk.cap || held[2] != C().scr_misc.cap || held[3] != C().scr_pool.cap)
    return fail(BOSS_ERR_STATE, "score: a nested scoring call grew a buffer of the outer call");
  r.any_fail = s.any_fail;
  return restore_small ? c.upload_small() : 0;
}

// Argmax screening (DESIGN.md 2.9) runs for calls of at least this many candidates (BOSS_SCREEN_MIN_M overrides, read
// per call): below it the bounds, the seed batch and the two waits of the first chunk are a visible share of the call.
constexpr long long SCREEN_MIN_M = 65536;
constexpr size_t SCREEN_POOL_BYTES = (size_t)1 << 30;   // pool for every candidate of the call; larger calls are not screened
constexpr double SCREEN_MIN_T = 0x1p-960;   // below it the EI evaluations lose relative precision (DESIGN.md 2.9)
long long screen_min_m() {
  const char *e = getenv("BOSS_SCREEN_MIN_M");
  return e ? atoll(e) : SCREEN_MIN_M;
}

// Argmax screening (DESIGN.md 2.9): a call that wants only the argmax of the closed-form EI over many candidates bounds
// every candidate from its mean alone and scores exactly only those that can still win.  Top-k calls (DESIGN.md 2.10)
// use the same bound against the k-th best score of a larger seed batch.
struct Screen {
  enum State { OFF, SCREENING, FELL_BACK } state = OFF;   // scr_stats[0]: 1 once a screened call finished, 2 fell back
  double thr = -INFINITY;   // survivors: bound >= thr or NaN
  double T = 0.0;           // the seed batch's best (argmax) or k-th best (top-k) score
  // FP32 mean tier from the second chunk on (BOSS_SCREEN_F64=1: the FP64 tier throughout); the threshold re-seeded
  // from the whole pool before it is scored (BOSS_SCREEN_NO_RESEED=1: not)
  bool f32 = false, reseed = false;
  // device-resident FP32 tier: one launch over every candidate after the first chunk, on the context's side stream
  // beside the first chunk's chain; `pending` until the library stream waits for it
  bool side = false, pending = false;
  long long n0 = 0, n_amb = 0;   // pool rows of the first chunk; ambiguous candidates of the call
  // device buffers: the bounds of one chunk (hi in the FP32 tier) and lo, per-256 survivor counts, the pool sizes (two
  // slots for the chunks, two for the re-compaction), the seed selection (two ping-pong rounds), the seed batch, the
  // refinement batch, the survivor pool with each row's bound and verdict, and the re-compacted pool
  double *bound = nullptr, *lo = nullptr, *seed_x = nullptr, *seed_pm = nullptr, *pool_x = nullptr, *pool_pm = nullptr;
  double *pool_bound = nullptr, *ref_x = nullptr, *ref_pm = nullptr, *consts = nullptr, *a2s = nullptr;
  int *fail_flag = nullptr;   // [2]: the side pass's and the variance tier's failed-variance flags
  int *ti[2] = {}, *ref_row = nullptr, *ref_cnt = nullptr;
  unsigned long long *tk[2] = {};
  long long *cnt = nullptr, *base = nullptr, *pool_idx = nullptr;   // cnt: survivors per 128 candidates, then offsets
  unsigned char *seed_cm = nullptr, *pool_cm = nullptr, *pool_ver = nullptr;
  std::vector<float *> xt32, al32;   // per slice: the MMA tier's B fragments of the centred training inputs, |t~|^2 and alpha

  bool on() const { return state == SCREENING; }

  // every exit of the call orders the library stream after the side stream's pass (it reads the caller's candidates)
  ~Screen() { join(); }
  void join() {
    if (pending) cudaStreamWaitEvent(C().stream, C().side_join, 0);
    pending = false;
  }

  // bytes of one pool row: candidate, index, bound, verdict, prior means, constraint-mask entry
  static size_t pool_row(const ScoreArgs &a, int d) {
    return (size_t)d * 8 + 8 + 8 + 1 + (a.prior_mean ? (size_t)a.y_dim * 8 : 0) + (a.cons_mask ? 1 : 0);
  }

  // ch0: the first chunk, which the seed batch is drawn from
  static bool eligible(const ScoreArgs &a, int ch0, int d) {
    return (a.want_argmax || a.topk) && a.best && !a.internal && !a.acq && !a.xgrad() && !a.mu_out && !a.var_out &&
           !a.status_out && !a.mix && a.M >= screen_min_m() && (size_t)a.M * pool_row(a, d) <= SCREEN_POOL_BYTES &&
           a.topk <= ch0 && getenv("BOSS_NO_SCREEN") == nullptr;
  }

  int begin(const ScoreCall &c, int ch0) {
    const ScoreArgs &a = c.a;
    const long long M = a.M;
    const int CH = c.CH, d = c.d, y_dim = a.y_dim, ns_max = a.topk ? topk_seed_n(a.topk, ch0) : SEED_N;
    const bool pm = a.prior_mean != nullptr, cm = a.cons_mask != nullptr;
    // the FP32 tier's error bound is proven for KIDs 0-2 only, and its kernel takes up to SCREEN_F32_MAX_SL slices of one
    // covariance function: any other call keeps FP64 means throughout
    const int kid0 = c.sl[0]->kernel_id;
    f32 = getenv("BOSS_SCREEN_F64") == nullptr && kid_has_f32_tier(kid0) && c.nsl <= SCREEN_F32_MAX_SL &&
          std::all_of(c.sl.begin(), c.sl.begin() + c.nsl, [&](const boss_gp *h) { return h->kernel_id == kid0; });
    reseed = getenv("BOSS_SCREEN_NO_RESEED") == nullptr;
    size_t tot = 0;
    const size_t ntk = (size_t)(CH + TOPK_IN - 1) / TOPK_IN * SEED_N;
    // bounds and counts for one chunk, or for all candidates after the first when they are on the device (FP32 tier)
    const size_t span = a.dev && f32 ? std::max<long long>(CH, M) : CH;
    const size_t o_bound = take(tot, span * 8), o_lo = take(tot, span * 8);
    const size_t o_cnt = take(tot, (span + 127) / 128 * 8), o_base = take(tot, 48);
    const size_t o_tk0 = take(tot, ntk * 8), o_tk1 = take(tot, ntk * 8), o_ti0 = take(tot, ntk * 4), o_ti1 = take(tot, ntk * 4);
    const size_t o_sx = take(tot, (size_t)ns_max * d * 8), o_spm = take(tot, (size_t)ns_max * y_dim * 8), o_scm = take(tot, ns_max);
    const size_t o_rx = take(tot, (size_t)CH * d * 8), o_rpm = take(tot, pm ? (size_t)CH * y_dim * 8 : 0);
    const size_t o_rrow = take(tot, (size_t)CH * 4), o_rcnt = take(tot, 8);
    const size_t o_consts = take(tot, (size_t)c.nsl * SCREEN_NCONST * 8), o_a2s = take(tot, (size_t)c.nsl * 8),
                 o_fail = take(tot, 8);
    std::vector<size_t> o_xt(c.nsl), o_al(c.nsl);
    for (int q = 0; q < c.nsl; ++q) {
      o_xt[q] = take(tot, f32 ? (size_t)c.sl[q]->n_pad * ((c.sl[q]->dp + 7) / 8 * 8) * 8 : 0);
      o_al[q] = take(tot, f32 ? (size_t)c.sl[q]->n_pad * 8 : 0);
    }
    CUDA_TRY(C().scr_misc.ensure(tot));
    unsigned char *b = C().scr_misc.as<unsigned char>();
    bound = reinterpret_cast<double *>(b + o_bound);
    lo = reinterpret_cast<double *>(b + o_lo);
    cnt = reinterpret_cast<long long *>(b + o_cnt);
    base = reinterpret_cast<long long *>(b + o_base);
    tk[0] = reinterpret_cast<unsigned long long *>(b + o_tk0);
    tk[1] = reinterpret_cast<unsigned long long *>(b + o_tk1);
    ti[0] = reinterpret_cast<int *>(b + o_ti0);
    ti[1] = reinterpret_cast<int *>(b + o_ti1);
    seed_x = reinterpret_cast<double *>(b + o_sx);
    seed_pm = reinterpret_cast<double *>(b + o_spm);
    seed_cm = b + o_scm;
    ref_x = reinterpret_cast<double *>(b + o_rx);
    ref_pm = pm ? reinterpret_cast<double *>(b + o_rpm) : nullptr;
    ref_row = reinterpret_cast<int *>(b + o_rrow);
    ref_cnt = reinterpret_cast<int *>(b + o_rcnt);
    consts = reinterpret_cast<double *>(b + o_consts);
    a2s = reinterpret_cast<double *>(b + o_a2s);
    fail_flag = reinterpret_cast<int *>(b + o_fail);
    xt32.assign(c.nsl, nullptr);
    al32.assign(c.nsl, nullptr);
    // Device-resident candidates: the constants and the FP32 pass over [ch0, M) go to the side stream, forked here
    // (after the wait for the caller's stream).  Nested calls of the first chunk rewrite the small block, so the pass
    // reads its own copy of the prior variances.
    side = f32 && a.dev && M > ch0;
    cudaStream_t cs = C().stream;
    if (side) {
      CUDA_TRY(cudaMemcpyAsync(a2s, c.small, (size_t)c.nsl * 8, cudaMemcpyDeviceToDevice, C().stream));
      CUDA_TRY(cudaEventRecord(C().side_fork, C().stream));
      CUDA_TRY(cudaStreamWaitEvent(C().side, C().side_fork, 0));
      cs = C().side;
      pending = true;
    }
    for (int q = 0; q < c.nsl && f32; ++q) {   // per call, so that an appended point or a refit is never missed
      const boss_gp *h = c.sl[q];
      xt32[q] = reinterpret_cast<float *>(b + o_xt[q]);
      al32[q] = reinterpret_cast<float *>(b + o_al[q]);
      screen_consts_kernel<<<1, 1024, 0, cs>>>(h->Xt, h->alpha, h->n, h->n_pad, h->dp, xt32[q], al32[q],
                                               consts + (size_t)SCREEN_NCONST * q);
      ++C().launches;
    }
    tot = 0;
    const size_t o_px = take(tot, (size_t)M * d * 8), o_pidx = take(tot, (size_t)M * 8);
    const size_t o_pb = take(tot, (size_t)M * 8), o_pv = take(tot, (size_t)M);
    const size_t o_ppm = pm ? take(tot, (size_t)M * y_dim * 8) : 0, o_pcm = cm ? take(tot, (size_t)M) : 0;
    CUDA_TRY(C().scr_pool.ensure(tot));
    b = C().scr_pool.as<unsigned char>();
    pool_x = reinterpret_cast<double *>(b + o_px);
    pool_idx = reinterpret_cast<long long *>(b + o_pidx);
    pool_bound = reinterpret_cast<double *>(b + o_pb);
    pool_ver = b + o_pv;
    pool_pm = pm ? reinterpret_cast<double *>(b + o_ppm) : nullptr;
    pool_cm = cm ? b + o_pcm : nullptr;
    CUDA_TRY(cudaMemsetAsync(base, 0, 48, C().stream));
    state = SCREENING;
    return 0;
  }

  // EI at the prior variance, PoF = 1, no guards: the bound pass's parameters, bound[m - out_off]
  static AcqParams bound_params(const AcqParams &ap, double *bound, long long out_off) {
    AcqParams bp = ap;
    bp.sumsq = nullptr;
    bp.has_ymax = 0;
    bp.lb = bp.ub = nullptr;
    bp.cons_mask = nullptr;
    bp.acq = bound;
    bp.out_off = out_off;
    bp.blk_val = nullptr;
    bp.blk_idx = nullptr;
    return bp;
  }

  // The FP32 tier over the chunk of ap: hi and lo of candidate m at [m - out_off], and with cnt the survivors
  // !(hi < thr (1 - 2^-32)) per 128 candidates
  void launch_f32(const ScoreCall &c, const AcqParams &ap, const ChunkIO &io, long long out_off, long long *cnt_out,
                  cudaStream_t st) {
    ScreenF32Params sp{};
    sp.Xs = io.xs;
    sp.m0 = ap.m0;
    sp.M = ap.m0 + ap.chunk;
    sp.in_off = io.off;
    sp.d = c.d;
    sp.nsl = c.nsl;
    for (int q = 0; q < c.nsl; ++q) {
      const boss_gp *h = c.sl[q];
      sp.sl[q] = ScreenSlice{reinterpret_cast<const float4 *>(xt32[q]), reinterpret_cast<const float4 *>(al32[q]),
                             consts + (size_t)SCREEN_NCONST * q, h->invl, h->disc, h->a2, h->n_pad};
    }
    sp.hi = bound_params(ap, bound, out_off);
    sp.lo = sp.hi;
    sp.lo.acq = lo;
    sp.thr = thr * (1.0 - 0x1p-32);
    sp.cnt = cnt_out;
    {
      Timed t(1, st);
      launch_screen_mean_bound(c.sl[0]->kernel_id, c.sl[0]->dp, sp, (ap.chunk + 127) / 128, st);
    }
    ++C().launches;
  }

  // Device-resident FP32 tier: the bounds of every candidate after the first chunk (ap's chunk) on the side stream,
  // at bound[m] and lo[m], beside the first chunk on the library stream.  No threshold exists yet: the counts come
  // after the join (chunk()), with the fused kernel's rule.
  void launch_side(const ScoreCall &c, AcqParams ap, const ChunkIO &io) {
    ap.a2 = a2s;
    ap.any_fail = fail_flag;   // never set (the prior variance a^2 + 1e-18 passes _clip_var), and never read
    launch_f32(c, ap, io, 0, nullptr, C().side);
    cudaEventRecord(C().side_join, C().side);
  }

  // One chunk: the means of every slice (xcov without K*^T), the bounds, the survivors appended to the pool.  The first
  // chunk also sets the threshold from the seed batch and ends screening (the chunk is then scored on the full path
  // from the same staged inputs) when the bound does not separate: T not positive, or more than a quarter of the chunk
  // surviving.  The first chunk takes the FP64 means, so the seed batch, T and that decision are those of the FP64
  // tier; later chunks of the FP32 tier bound EI from mu~ +- E' in one launch of screen_mean_bound_kernel and leave the
  // ambiguous ones to Screen::finish.  With device-resident candidates, the FP32 tier's "chunk" is everything after the
  // first chunk (see score_core), bounded on the side stream while the first chunk runs (launch_side).
  int chunk(const ScoreCall &c, const AcqParams &ap, const ChunkIO &io, int cidx, TopkBufs &tb) {
    const ScoreArgs &a = c.a;
    const long long m0 = ap.m0;
    const int ch = ap.chunk, ncb = (ch + 127) / 128, nb = (ch + 255) / 256;
    const bool t32 = f32 && cidx > 0;
    const AcqParams bp = bound_params(ap, bound, m0);
    const double *bnd = bound, *blo = lo;   // the chunk's bounds, candidate m0 first
    // FP32 tier: hi < thr (1 - 2^-32) drops, lo >= thr (1 + 2^-32) keeps, anything else (NaN too) is ambiguous.  The
    // first chunk (FP64 tier) sets thr in seed().
    if (t32 && side) {   // the side stream's pass (launch_side) has the bounds
      join();
      bnd = bound + m0;
      blo = lo + m0;
    } else if (t32) {
      launch_f32(c, ap, io, m0, cnt, C().stream);
    } else {
      for (int q = 0; q < c.nsl; ++q) {
        const boss_gp *h = c.sl[q];
        const int nks = std::max(1, std::min(h->nblk, (16 * 148 + ncb - 1) / ncb));
        {
          Timed t(1);
          launch_xcov_mean(h->kernel_id, h->dp, xcov_params(h, io.xs, a.M, m0, io.off, c.d, c.CH), dim3(ncb, nks),
                           C().stream);
        }
        reduce_rows_kernel<<<(ncb * 128 + 255) / 256, 256, 0, C().stream>>>(
            C().part_mu.as<double>(), 2 * h->nblk, (size_t)c.CH, C().muv.as<double>() + (size_t)q * c.CH, ncb * 128);
      }
      acq_kernel<<<nb, 256, 0, C().stream>>>(bp);
      C().launches += 2 * c.nsl + 1;
    }
    const size_t c0 = (size_t)(m0 - ap.in_off);   // the chunk's first candidate in the input arrays
    const double *xs_c = ap.Xs + c0 * c.d;
    const double *pm_c = ap.prior_mean ? ap.prior_mean + c0 * a.y_dim : nullptr;
    const unsigned char *cm_c = ap.cons_mask ? ap.cons_mask + c0 : nullptr;
    if (cidx == 0) {
      int rc = seed(c, ch, xs_c, pm_c, cm_c, tb);
      if (rc || !on()) return rc;
    }
    const double thr_drop = t32 ? thr * (1.0 - 0x1p-32) : thr;
    if (!t32 || side) {
      screen_count_kernel<<<ncb, 128, 0, C().stream>>>(bnd, nullptr, ch, thr_drop, cnt);
      ++C().launches;
    }
    screen_scan_kernel<<<1, 1024, 0, C().stream>>>(cnt, ncb, base, cidx & 1);
    CompactParams cpar{bnd, nullptr, ch, thr_drop, t32 ? blo : nullptr, thr * (1.0 + 0x1p-32), cnt, m0, xs_c, pm_c, cm_c,
                       c.d, a.y_dim, pool_x, pool_pm, pool_cm, pool_idx, nullptr, pool_bound, pool_ver};
    screen_compact_kernel<<<ncb, 128, 0, C().stream>>>(cpar);
    C().launches += 2;
    if (cidx == 0) {
      long long surv = 0;
      CUDA_TRY(cudaMemcpyAsync(&surv, base + 1, 8, cudaMemcpyDeviceToHost, C().stream));
      CUDA_TRY(cudaStreamSynchronize(C().stream));
      C().scr_stats[2] = surv;
      n0 = surv;
      if (4 * surv > ch) fall_back();
    }
    return 0;
  }

  // After the last chunk: the ambiguous rows refined in FP64, the threshold re-seeded from the pool's highest bounds,
  // the pool re-compacted; then the pool (survivors in ascending order) through the ordinary path, its first-maximal
  // winner (or its k best) mapped back to the call's indices.
  int finish(const ScoreCall &c, int nchunks, HostStaging &stg) {
    ScoreArgs &a = c.a;
    long long npool = 0;
    CUDA_TRY(cudaMemcpyAsync(&npool, base + (nchunks & 1), 8, cudaMemcpyDeviceToHost, C().stream));
    CUDA_TRY(cudaStreamSynchronize(C().stream));
    int rc = stg.drain_last();
    if (rc) return rc;
    C().scr_stats[0] = 1;
    C().scr_stats[1] = a.M;
    n_amb = 0;
    for (long long r0 = n0; f32 && r0 < npool; r0 += c.CH) {
      rc = refine(c, r0, (int)std::min<long long>(c.CH, npool - r0));
      if (rc) return rc;
    }
    const double *px = pool_x, *ppm = pool_pm;
    const unsigned char *pcm = pool_cm;
    const long long *pidx = pool_idx;
    long long nfin = npool;
    double thr2 = thr;
    const int ns_max = a.topk ? topk_seed_n(a.topk, (int)std::min<long long>(c.CH, a.M)) : SEED_N;
    if (reseed && npool > ns_max) {
      rc = reseed_thr(c, (int)std::min<long long>(npool, c.CH), thr2);
      if (rc) return rc;
    }
    if (n_amb > 0 || thr2 > thr) {   // keep rows with verdict 1 and bound >= thr2 (or NaN), in order
      rc = recompact(c, npool, thr2, nfin);
      if (rc) return rc;
      unsigned char *b = C().scr_pool2.as<unsigned char>();
      px = reinterpret_cast<double *>(b);
      pidx = reinterpret_cast<long long *>(b + p2_off[0]);
      ppm = pool_pm ? reinterpret_cast<double *>(b + p2_off[1]) : nullptr;
      pcm = pool_cm ? b + p2_off[2] : nullptr;
    }
    C().scr_stats[2] = nfin;
    C().scr_amb[0] = n_amb;
    C().scr_amb[1] = npool;
    if (nfin < 1) return fail(BOSS_ERR_STATE, "score: argmax screening kept no candidate");   // the seed's winner always survives
    if (nfin < a.topk) return fail(BOSS_ERR_STATE, "score: top-k screening kept fewer than k candidates");   // the seed's k best survive
    const bool multi_blk = std::all_of(c.sl.begin(), c.sl.begin() + c.nsl, [](const boss_gp *h) { return h->nblk >= 2; });
    if (multi_blk && nfin > SEED_N) {
      rc = var_tier(c, thr2, px, ppm, pcm, pidx, nfin);
      if (rc) return rc;
      if (nfin < std::max<long long>(1, a.topk)) return fail(BOSS_ERR_STATE, "score: the variance tier kept too few candidates");
    }
    SubsetResult r;
    rc = score_subset(c, px, ppm, pcm, nfin, a.top_val, a.top_idx, pidx, false, r);
    if (rc) return rc;
    a.any_fail = r.any_fail;
    if (a.topk) return 0;
    long long idx = -1;
    if (r.best_idx >= 0) {
      CUDA_TRY(cudaMemcpyAsync(&idx, pidx + r.best_idx, 8, cudaMemcpyDeviceToHost, C().stream));
      CUDA_TRY(cudaStreamSynchronize(C().stream));
    }
    if (a.best_val) *a.best_val = r.best_val;
    if (a.best_idx) *a.best_idx = idx;
    return 0;
  }

 private:
  size_t p2_off[3] = {0, 0, 0};   // re-compacted pool: offsets of the indices, prior means, mask entries

  void fall_back() {   // the full path goes on behind the side stream's (wasted) pass
    C().scr_stats[0] = 2;
    state = FELL_BACK;
    join();
  }

  // The seed batch of the first chunk: the exact scores of its highest bounds.  Their best (argmax) or k-th best
  // (top-k) score T is a lower bound of the call's best or k-th best score; bounds below T (1 - 2^-30) cannot reach it.
  int seed(const ScoreCall &c, int ch, const double *xs_c, const double *pm_c, const unsigned char *cm_c, TopkBufs &tb) {
    double Ts;
    int rc = score_seed(c, ch, bound, xs_c, pm_c, cm_c, tb, Ts);
    if (rc) return rc;
    C().scr_stats[1] = ch;
    if (!(Ts >= SCREEN_MIN_T)) {
      fall_back();
      return 0;
    }
    T = Ts;
    thr = T * (1.0 - 0x1p-30);
    return 0;
  }

  // the exact scores of the highest of the n bounds b (candidate i at xs + i d, pm + i y_dim, cm + i): their best
  // (argmax) or k-th best (top-k) score
  int score_seed(const ScoreCall &c, int n, const double *b, const double *xs, const double *pm, const unsigned char *cm,
                 TopkBufs &tb, double &Ts) {
    const ScoreArgs &a = c.a;
    int ns;
    if (a.topk) {   // the S_k highest bounds (NaN bounds last), selected into the top-k buffers
      ns = topk_seed_n(a.topk, n);
      SelectIn in{nullptr, nullptr, 0, b, 0, n, 1};
      int rc = tb.select(in, ns, tb.run_val[0], tb.run_idx[0]);
      if (rc) return rc;
      seed_gather_kernel<<<(ns + 255) / 256, 256, 0, C().stream>>>(tb.run_idx[0], ns, xs, pm, cm, c.d, a.y_dim,
                                                                    seed_x, seed_pm, seed_cm);
    } else {        // the SEED_N highest bounds: bitonic rounds over TOPK_IN-element blocks
      int m = n, par = 0;
      const unsigned long long *kin = nullptr;
      const int *iin = nullptr;
      do {
        const int nbk = (m + TOPK_IN - 1) / TOPK_IN;
        seed_topk_kernel<<<nbk, 1024, 0, C().stream>>>(kin ? nullptr : b, kin, iin, m, tk[par], ti[par]);
        ++C().launches;
        kin = tk[par];
        iin = ti[par];
        par ^= 1;
        m = nbk * SEED_N;
      } while (m > SEED_N);
      ns = std::min(SEED_N, n);
      seed_gather_kernel<<<1, SEED_N, 0, C().stream>>>(iin, ns, xs, pm, cm, c.d, a.y_dim, seed_x, seed_pm, seed_cm);
    }
    ++C().launches;
    std::vector<double> sv((size_t)a.topk);
    std::vector<int64_t> si((size_t)a.topk);
    SubsetResult r;
    int rc = score_subset(c, seed_x, pm ? seed_pm : nullptr, cm ? seed_cm : nullptr, ns, sv.data(), si.data(), nullptr,
                          true, r);
    if (rc) return rc;
    Ts = a.topk ? sv[(size_t)a.topk - 1] : r.best_val;
    return 0;
  }

  // Pool rows [r0, r0 + n) (n <= CH): the ambiguous ones gathered, their FP64 means and bounds (xcov_kernel<.., false>,
  // reduce_rows and the bound of the FP64 tier, so bit for bit the bound that tier computes), today's rule as verdict.
  int refine(const ScoreCall &c, long long r0, int n) {
    const ScoreArgs &a = c.a;
    CUDA_TRY(cudaMemsetAsync(ref_cnt, 0, 4, C().stream));
    screen_amb_gather_kernel<<<(n + 255) / 256, 256, 0, C().stream>>>(
        pool_ver + r0, n, pool_x + (size_t)r0 * c.d, pool_pm ? pool_pm + (size_t)r0 * a.y_dim : nullptr, c.d, a.y_dim,
        (int)r0, ref_x, ref_pm, ref_row, ref_cnt);
    int namb = 0;
    CUDA_TRY(cudaMemcpyAsync(&namb, ref_cnt, 4, cudaMemcpyDeviceToHost, C().stream));
    CUDA_TRY(cudaStreamSynchronize(C().stream));
    C().launches += 1;
    n_amb += namb;
    if (namb == 0) return 0;
    const int ncb = (namb + 127) / 128, nb = (namb + 255) / 256;
    for (int q = 0; q < c.nsl; ++q) {
      const boss_gp *h = c.sl[q];
      const int nks = std::max(1, std::min(h->nblk, (16 * 148 + ncb - 1) / ncb));
      launch_xcov_mean(h->kernel_id, h->dp, xcov_params(h, ref_x, namb, 0, 0, c.d, c.CH), dim3(ncb, nks), C().stream);
      reduce_rows_kernel<<<(ncb * 128 + 255) / 256, 256, 0, C().stream>>>(C().part_mu.as<double>(), 2 * h->nblk, (size_t)c.CH,
                                                                        C().muv.as<double>() + (size_t)q * c.CH, ncb * 128);
    }
    ChunkIO io;
    io.xs = ref_x;
    io.pm = ref_pm;
    AcqParams bp = c.acq_params(0, namb, io);
    bp.M = namb;
    bp.sumsq = nullptr;
    bp.has_ymax = 0;
    bp.lb = bp.ub = nullptr;
    bp.cons_mask = nullptr;
    bp.acq = bound;
    bp.out_off = 0;
    bp.blk_val = nullptr;
    bp.blk_idx = nullptr;
    acq_kernel<<<nb, 256, 0, C().stream>>>(bp);
    screen_amb_scatter_kernel<<<nb, 256, 0, C().stream>>>(bound, ref_row, namb, thr, pool_bound, pool_ver);
    C().launches += 2 * c.nsl + 2;
    return 0;
  }

  // Re-seed (DESIGN.md 2.9): the exact scores of the highest bounds among the first n pool rows still kept.  Any set of
  // real candidates gives a valid threshold; the pool's highest bounds give one close to the call's best score.
  int reseed_thr(const ScoreCall &c, int n, double &thr2) {
    screen_sel_bound_kernel<<<(n + 255) / 256, 256, 0, C().stream>>>(pool_bound, pool_ver, n, bound);
    ++C().launches;
    TopkBufs tb;
    if (c.a.topk) {
      int rc = tb.setup(c.a.topk, c.CH, (int)std::min<long long>(c.CH, c.a.M));
      if (rc) return rc;
    }
    double Ts;
    int rc = score_seed(c, n, bound, pool_x, pool_pm, pool_cm, tb, Ts);
    if (rc) return rc;
    if (Ts > T) thr2 = Ts * (1.0 - 0x1p-30);
    return 0;
  }

  // pool rows with verdict 1 and bound >= thr2 (or NaN), in order, into the second pool buffer; their count -> nfin
  // the second pool buffer for n rows: candidates first, then the offsets in p2_off
  int size_pool2(const ScoreCall &c, long long n) {
    size_t tot = 0;
    const size_t o_x = take(tot, (size_t)n * c.d * 8);
    p2_off[0] = take(tot, (size_t)n * 8);
    p2_off[1] = take(tot, pool_pm ? (size_t)n * c.a.y_dim * 8 : 0);
    p2_off[2] = take(tot, pool_cm ? (size_t)n : 0);
    (void)o_x;
    CUDA_TRY(C().scr_pool2.ensure(tot));
    return 0;
  }

  int recompact(const ScoreCall &c, long long npool, double thr2, long long &nfin) {
    const ScoreArgs &a = c.a;
    int rc = size_pool2(c, npool);
    if (rc) return rc;
    unsigned char *b = C().scr_pool2.as<unsigned char>();
    int par = 0;
    for (long long r0 = 0; r0 < npool; r0 += c.CH, par ^= 1) {
      const int n = (int)std::min<long long>(c.CH, npool - r0), ncb = (n + 127) / 128;
      screen_count_kernel<<<ncb, 128, 0, C().stream>>>(pool_bound + r0, pool_ver + r0, n, thr2, cnt);
      screen_scan_kernel<<<1, 1024, 0, C().stream>>>(cnt, ncb, base + 2, par);
      CompactParams cp{pool_bound + r0, pool_ver + r0, n, thr2, nullptr, 0.0, cnt, 0,
                       pool_x + (size_t)r0 * c.d, pool_pm ? pool_pm + (size_t)r0 * a.y_dim : nullptr,
                       pool_cm ? pool_cm + r0 : nullptr, c.d, a.y_dim,
                       reinterpret_cast<double *>(b), pool_pm ? reinterpret_cast<double *>(b + p2_off[1]) : nullptr,
                       pool_cm ? b + p2_off[2] : nullptr, reinterpret_cast<long long *>(b + p2_off[0]), pool_idx + r0,
                       nullptr, nullptr};
      screen_compact_kernel<<<ncb, 128, 0, C().stream>>>(cp);
      C().launches += 3;
    }
    CUDA_TRY(cudaMemcpyAsync(&nfin, base + 2 + par, 8, cudaMemcpyDeviceToHost, C().stream));
    CUDA_TRY(cudaStreamSynchronize(C().stream));
    return 0;
  }

  // The variance tier (DESIGN.md 2.9): W = L^-1 is lower triangular, so the first row block of V = W K* involves the
  // first 128 training points only, and its column sum of squares S1 is at most the full S.  Per piece of pool rows:
  // K* and the mean partials (xcov_kernel<.., true>), mu reduced as on the exact path, the first row block of V by
  // score_quarter_kernel with nblk = 1 (the same k order and DMMA chain as that block in the full pass; nblk >= 2 in
  // score_slice is its cost model, not a kernel condition), quarter_sumsq_kernel's partials of that block and the
  // fixed-order reduction with the other row blocks' partials taken as +0.  FP addition is monotone and every partial
  // is >= 0, so the computed S1 <= the computed S, and EI at a^2 - S1 with the exact mu, PoF 1 and no guards bounds
  // each row's exact score.  Rows with bound >= thr2 (or NaN) are kept in order, the index map composed; the rows
  // move between the two pool buffers.  A failed variance (a -inf bound) keeps the whole pool, so the exact pass still
  // sees the failure.
  int var_tier(const ScoreCall &c, double thr2, const double *&px, const double *&ppm, const unsigned char *&pcm,
               const long long *&pidx, long long &nfin) {
    const ScoreArgs &a = c.a;
    constexpr int PIECE = 8192;   // rows per pass: V^T scratch of PIECE x n_pad, what the exact pass on PIECE rows takes
    const int piece = std::min(c.CH, PIECE);
    int max_npad = 0;
    for (int q = 0; q < c.nsl; ++q) max_npad = std::max(max_npad, c.sl[q]->n_pad);
    CUDA_TRY(C().vt.ensure((size_t)piece * max_npad * 8));
    const bool to_pool = px != pool_x;   // the rows are in the second buffer: write the first
    if (!to_pool) {
      int rc = size_pool2(c, nfin);
      if (rc) return rc;
    }
    unsigned char *b2 = C().scr_pool2.as<unsigned char>();
    double *ox = to_pool ? pool_x : reinterpret_cast<double *>(b2);
    long long *oidx = to_pool ? pool_idx : reinterpret_cast<long long *>(b2 + p2_off[0]);
    double *opm = !pool_pm ? nullptr : to_pool ? pool_pm : reinterpret_cast<double *>(b2 + p2_off[1]);
    unsigned char *ocm = !pool_cm ? nullptr : to_pool ? pool_cm : b2 + p2_off[2];
    CUDA_TRY(cudaMemsetAsync(fail_flag + 1, 0, 4, C().stream));
    int par = 0;
    for (long long r0 = 0; r0 < nfin; r0 += piece, par ^= 1) {
      const int n = (int)std::min<long long>(piece, nfin - r0), ncb = (n + 127) / 128, ncb32 = (n + NW_NB - 1) / NW_NB;
      const double *xs = px + (size_t)r0 * c.d;
      for (int q = 0; q < c.nsl; ++q) {
        const boss_gp *h = c.sl[q];
        const int nks = std::max(1, std::min(h->nblk, (16 * 148 + ncb - 1) / ncb));
        launch_xcov(h->kernel_id, h->dp, xcov_params(h, xs, n, 0, 0, c.d, c.CH), dim3(ncb, nks), C().stream);
        reduce_rows_kernel<<<(ncb * 128 + 255) / 256, 256, 0, C().stream>>>(C().part_mu.as<double>(), 2 * h->nblk,
                                                                          (size_t)c.CH, C().muv.as<double>() + (size_t)q * c.CH,
                                                                          ncb * 128);
        NarrowParams np{h->W, C().ks.as<double>(), 1, h->ktiles, nullptr, c.CH, C().vt.as<double>()};
        score_quarter_kernel<0, 4, 1><<<dim3(ncb32, 4), NQ_THREADS, NQ_SMEM_BYTES, C().stream>>>(np);
        quarter_sumsq_kernel<<<dim3(ncb32, 1), 256, 0, C().stream>>>(C().vt.as<double>(), h->ktiles,
                                                                    C().part_ss.as<double>(), c.CH);
        reduce_rows2_kernel<<<(ncb * 128 + 255) / 256, 256, 0, C().stream>>>(C().part_ss.as<double>(), 2, (size_t)c.CH,
                                                                           C().sumsq.as<double>() + (size_t)q * c.CH,
                                                                           ncb * 128);
      }
      ChunkIO io;
      io.xs = xs;
      io.pm = ppm ? ppm + (size_t)r0 * a.y_dim : nullptr;
      AcqParams bp = c.acq_params(0, n, io);
      bp.M = n;
      bp.has_ymax = 0;
      bp.lb = bp.ub = nullptr;
      bp.cons_mask = nullptr;
      bp.acq = bound;
      bp.out_off = 0;
      bp.blk_val = nullptr;
      bp.blk_idx = nullptr;
      bp.any_fail = fail_flag + 1;
      acq_kernel<<<(n + 255) / 256, 256, 0, C().stream>>>(bp);
      screen_count_kernel<<<ncb, 128, 0, C().stream>>>(bound, nullptr, n, thr2, cnt);
      screen_scan_kernel<<<1, 1024, 0, C().stream>>>(cnt, ncb, base + 4, par);
      CompactParams cp{bound, nullptr, n, thr2, nullptr, 0.0, cnt, 0, xs, io.pm, pcm ? pcm + r0 : nullptr, c.d, a.y_dim,
                       ox, opm, ocm, oidx, pidx + r0, nullptr, nullptr};
      screen_compact_kernel<<<ncb, 128, 0, C().stream>>>(cp);
      C().launches += 5 * c.nsl + 4;
    }
    long long kept = 0;
    int failed = 0;
    CUDA_TRY(cudaMemcpyAsync(&kept, base + 4 + par, 8, cudaMemcpyDeviceToHost, C().stream));
    CUDA_TRY(cudaMemcpyAsync(&failed, fail_flag + 1, 4, cudaMemcpyDeviceToHost, C().stream));
    CUDA_TRY(cudaStreamSynchronize(C().stream));
    if (failed) return 0;
    C().scr_var[0] = nfin;
    C().scr_var[1] = kept;
    px = ox;
    ppm = opm;
    pcm = ocm;
    pidx = oidx;
    nfin = kept;
    return 0;
  }
};

int score_core(ScoreArgs &a) {
  ScoreCall c(a);
  int rc = c.bind();
  if (rc) return rc;
  a.any_fail = 0;
  if (a.M <= 0) {
    if (a.best_idx) *a.best_idx = -1;
    return 0;
  }
  if (a.dev && !a.internal) {
    rc = wait_for_caller(a.caller_stream);
    if (rc) return rc;
  }
  rc = c.setup();
  if (rc) return rc;
  if (!a.internal) {
    C().scr_stats[0] = C().scr_stats[1] = C().scr_stats[2] = C().scr_amb[0] = C().scr_amb[1] = C().scr_var[0] = C().scr_var[1] = 0;
    for (int64_t &p : C().score_paths) p = 0;
  }
  const int ch0 = (int)std::min<long long>(c.CH, a.M);   // the first chunk
  Screen scr;
  if (Screen::eligible(a, ch0, c.d)) {
    rc = scr.begin(c, ch0);
    if (rc) return rc;
  }
  TopkBufs tb;   // top-k: the running set absorbs every scored chunk
  if (a.topk) {
    rc = tb.setup(a.topk, c.CH, ch0);
    if (rc) return rc;
  }
  HostStaging stg;
  if (!a.dev) {
    rc = stg.plan(a, c.CH, c.d);
    if (rc) return rc;
  }

  timing_begin();
  int cidx = 0;
  for (long long m0 = 0, step = 0; m0 < a.M; m0 += step, ++cidx) {
    // device-resident candidates on the FP32 screening tier: everything after the first chunk in one piece (the
    // screened call's M fits the pool, so an int)
    const int ch = (int)std::min<long long>(scr.on() && scr.f32 && a.dev && cidx > 0 ? a.M : c.CH, a.M - m0);
    step = ch;
    const int slot = cidx & 1;
    ChunkIO io;
    if (a.dev) {
      io = {a.Xs, a.prior_mean, a.prior_mean_grad, a.cons_mask, a.acq, a.mu_out, a.var_out, a.grad, a.status_out, 0,
            a.dmu_out, a.dvar_out};
    } else {
      rc = stg.chunk_inputs(m0, ch, slot, io);
      if (rc) return rc;
    }
    AcqParams ap = c.acq_params(m0, ch, io);
    if (a.topk) {   // the chunk's scores stay on the device, for the running top-k set
      ap.acq = tb.scores;
      ap.out_off = m0;
    }
    if (scr.on()) {
      if (cidx == 0 && scr.side) scr.launch_side(c, c.acq_params(ch, (int)(a.M - ch), io), io);
      rc = scr.chunk(c, ap, io, cidx, tb);
      if (rc) return rc;
    }
    if (!scr.on()) {   // the full path (screening did not take the chunk)
      bool fused = false;
      for (int q = 0; q < c.nsl; ++q) fused = score_slice(c, q, ap, io);
      if (a.pgrad()) {   // the posteriors and their gradients are the output: no acquisition
        PredictGradParams pg{ap, C().dmu.as<double>(), C().dvar.as<double>(), io.pmg, io.mu, io.var, io.dmu, io.dvar, io.st};
        const long long ne = (long long)ch * c.d * c.nsl;
        predict_grad_kernel<<<(unsigned)((ne + 255) / 256), 256, 0, C().stream>>>(pg);
        ++C().launches;
      } else if (!fused) {
        const int nb = (ch + 255) / 256;
        acq_kernel<<<nb, 256, 0, C().stream>>>(ap);
        ++C().launches;
        if (a.want_argmax) {
          argmax_final_kernel<<<1, 256, 0, C().stream>>>(C().blk_val.as<double>(), C().blk_idx.as<long long>(), nb, c.d_best,
                                                         c.d_bidx);
          ++C().launches;
        }
      }
      if (a.topk) {
        rc = tb.absorb(m0, ch);
        if (rc) return rc;
      }
    }
    if (a.grad) {
      AcqGradParams gp2{ap, C().dmu.as<double>(), C().dvar.as<double>(), io.pmg, io.grad};
      if (ap.mix.kind != 0 && ap.has_best)   // Monte-Carlo EI; PoF alone has no Monte-Carlo term
        acq_grad_kernel<true><<<(ch + 127) / 128, 128, 0, C().stream>>>(gp2);
      else
        acq_grad_kernel<false><<<(ch + 127) / 128, 128, 0, C().stream>>>(gp2);
      ++C().launches;
    }
    if (!a.dev) {
      rc = stg.end_chunk(m0, ch, slot);
      if (rc) return rc;
    }
  }
  CUDA_TRY(cudaGetLastError());
  if (scr.on()) return scr.finish(c, cidx, stg);
  if (a.internal && !a.want_argmax && !a.topk && !C().timing) return 0;   // a round of the multi-start driver: it synchronises itself
  // one wait for everything: the (value, index, failure flag) triple -- top-k: the flag behind the k pairs -- is fetched
  // behind the last chunk's outputs, and the last chunk is handed to the caller after the stream has drained
  double res[3] = {0.0, 0.0, 0.0};
  if (a.topk) {
    rc = tb.finish(a.topk_map, a.top_val, a.top_idx);
    if (rc) return rc;
    CUDA_TRY(cudaMemcpyAsync(&res[2], c.d_anyfail, 4, cudaMemcpyDeviceToHost, C().stream));
  } else {
    CUDA_TRY(cudaMemcpyAsync(res, c.d_best, 24, cudaMemcpyDeviceToHost, C().stream));
  }
  CUDA_TRY(cudaStreamSynchronize(C().stream));
  rc = stg.drain_last();
  if (rc) return rc;
  timing_end();
  long long bidx;
  std::memcpy(&bidx, &res[1], 8);
  int af;
  std::memcpy(&af, &res[2], 4);
  a.any_fail = af;
  if (a.want_argmax) {
    if (a.best_val) *a.best_val = res[0];
    if (a.best_idx) *a.best_idx = bidx;
  }
  return 0;
}

// Scoring entry: one device, or -- in multi-device mode, for host arrays and large enough batches -- contiguous
// 128-aligned candidate ranges dealt to the devices (each scores its range against its own replica of the factors;
// a candidate's score does not depend on the batch it arrives in, so the result is bit-identical to the
// single-device call) and the (best value, index) pairs reduced on the host in Julia's argmax order.
int score_dispatch(ScoreArgs &a) {
  const boss_gp *h0 = (a.slices && a.y_dim >= 1 && a.n_samples >= 1) ? a.slices[0] : nullptr;
  const int nsl = a.y_dim * a.n_samples;
  int nd = (g_ndev > 1 && tl_dev < 0 && !a.dev && h0) ? g_ndev : 1;
  if (nd > 1) {
    for (int q = 0; q < nsl && nd > 1; ++q)
      for (int k = 0; k < nd; ++k)
        if (!replica_on(a.slices[q], k)) {
          nd = 1;
          break;
        }
    const long long blocks = (a.M + 127) / 128;
    if (blocks < 2LL * nd) nd = 1;
  }
  if (nd <= 1) {
    Ctx *cx = nullptr;
    if (a.dev || tl_dev >= 0 || !h0)
      cx = ctx_current();
    else
      cx = ctx_of(h0->dev);
    if (!cx) return fail(BOSS_ERR_STATE, h0 && h0->dev < 0 ? "handle is not valid any more (boss_shutdown was called)"
                                                           : "boss_init() has not been called");
    Enter en(cx);
    return score_core(a);
  }
  const long long blocks = (a.M + 127) / 128, per = (blocks + nd - 1) / nd * 128;
  const int d = h0->d;
  std::vector<ScoreArgs> sub(nd, a);
  std::vector<CandGen> gens(nd);
  std::vector<double> bv(nd, 0.0);
  std::vector<int64_t> bi(nd, -1);
  std::vector<long long> first(nd, 0);
  std::vector<std::vector<double>> tv(nd);   // top-k: each device's block top min(k, count), merged below
  std::vector<std::vector<int64_t>> ti(nd);
  int rc = for_each_device(nd, [&](int k, Ctx *) {
    ScoreArgs &s = sub[k];
    const long long off = std::min<long long>(a.M, (long long)k * per), cnt = std::min<long long>(per, a.M - off);
    first[k] = off;
    s.M = cnt;
    if (cnt <= 0) return 0;
    if (a.gen) {
      gens[k] = *a.gen;
      gens[k].first = a.gen->first + off;
      s.gen = &gens[k];
    } else {
      s.Xs = a.Xs + (size_t)off * d;
    }
    if (a.prior_mean) s.prior_mean = a.prior_mean + (size_t)off * a.y_dim;
    if (a.prior_mean_grad) s.prior_mean_grad = a.prior_mean_grad + (size_t)off * d * a.y_dim;
    if (a.cons_mask) s.cons_mask = a.cons_mask + off;
    if (a.acq) s.acq = a.acq + off;
    if (a.grad) s.grad = a.grad + (size_t)off * d;
    if (a.mu_out) s.mu_out = a.mu_out + (size_t)off * nsl;   // predict outputs: nsl per candidate (1 for boss_gp_predict)
    if (a.var_out) s.var_out = a.var_out + (size_t)off * nsl;
    if (a.status_out) s.status_out = a.status_out + (size_t)off * nsl;
    if (a.dmu_out) s.dmu_out = a.dmu_out + (size_t)off * d * nsl;
    if (a.dvar_out) s.dvar_out = a.dvar_out + (size_t)off * d * nsl;
    s.best_val = &bv[k];
    s.best_idx = &bi[k];
    if (a.topk) {
      s.topk = std::min<long long>(a.topk, cnt);
      tv[k].resize((size_t)s.topk);
      ti[k].resize((size_t)s.topk);
      s.top_val = tv[k].data();
      s.top_idx = ti[k].data();
    }
    return score_core(s);
  });
  if (rc) return rc;
  a.any_fail = 0;
  double best_v = 0.0;
  long long best_i = -1;
  for (int k = 0; k < nd; ++k) {
    if (sub[k].M <= 0) continue;
    a.any_fail |= sub[k].any_fail;
    if (a.want_argmax && bi[k] >= 0) {
      const long long gi = first[k] + bi[k];
      if (best_i < 0 || acq_better_host(bv[k], gi, best_v, best_i)) {
        best_v = bv[k];
        best_i = gi;
      }
    }
  }
  if (a.want_argmax) {
    if (a.best_val) *a.best_val = best_v;
    if (a.best_idx) *a.best_idx = best_i;
  }
  if (a.topk) {   // the k best of the devices' lists in the same order: the set the single-device call selects
    std::vector<std::pair<double, long long>> all;
    for (int k = 0; k < nd; ++k)
      for (size_t e = 0; e < tv[k].size(); ++e) all.emplace_back(tv[k][e], first[k] + ti[k][e]);
    std::sort(all.begin(), all.end(), [](const std::pair<double, long long> &x, const std::pair<double, long long> &y) {
      return acq_better_host(x.first, x.second, y.first, y.second);
    });
    for (long long e = 0; e < a.topk; ++e) {
      a.top_val[e] = all[(size_t)e].first;
      a.top_idx[e] = all[(size_t)e].second;
    }
  }
  return 0;
}

}  // namespace

// the fields every scoring entry point sets; the others start out null / false / zero
static ScoreArgs score_args(const boss_gp *const *slices, int y_dim, int n_samples, const double *Xs, int64_t M,
                            const double *prior_mean, const double *coefs, const double *best, const double *y_max,
                            const double *lb, const double *ub, const uint8_t *cons_mask) {
  ScoreArgs a{};
  a.slices = slices;
  a.y_dim = y_dim;
  a.n_samples = n_samples;
  a.Xs = Xs;
  a.M = M;
  a.prior_mean = prior_mean;
  a.coefs = coefs;
  a.best = best;
  a.y_max = y_max;
  a.lb = lb;
  a.ub = ub;
  a.cons_mask = cons_mask;
  return a;
}

// the box bounds of the acquisition come as a pair or not at all
static int check_lb_ub(const char *who, const double *lb, const double *ub) {
  if ((lb == nullptr) != (ub == nullptr)) return fail(BOSS_ERR_ARG, std::string(who) + ": lb and ub must be given together");
  return 0;
}

static int predict_impl(const char *who, const boss_gp *gp, const double *Xs, int64_t M, const double *prior_mean_s,
                        double *mu, double *var, int32_t *status, bool dev, void *stream) {
  if (!gp || (!Xs && M > 0)) return fail(BOSS_ERR_ARG, std::string(who) + ": bad arguments");
  const boss_gp *sl[1] = {gp};
  ScoreArgs a = score_args(sl, 1, 1, Xs, M, prior_mean_s, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr);
  a.mu_out = mu;
  a.var_out = var;
  a.status_out = status;
  a.dev = dev;
  a.caller_stream = stream;
  int rc = score_dispatch(a);
  if (rc) return rc;
  return a.any_fail ? BOSS_NEG_VARIANCE : 0;
}

int boss_gp_predict(const boss_gp *gp, const double *Xs, int64_t M, const double *prior_mean_s, double *mu,
                    double *var, int32_t *status) {
  return predict_impl("boss_gp_predict", gp, Xs, M, prior_mean_s, mu, var, status, false, nullptr);
}

int boss_gp_predict_dev(const boss_gp *gp, const double *Xs_dev, int64_t M, const double *prior_mean_s_dev,
                        double *mu_dev, double *var_dev, int32_t *status_dev, void *stream) {
  return predict_impl("boss_gp_predict_dev", gp, Xs_dev, M, prior_mean_s_dev, mu_dev, var_dev, status_dev, true, stream);
}

static int ei_score_impl(const boss_gp *const *slices, int y_dim, int n_samples, const double *Xs, int64_t M,
                         const double *prior_mean_s, const double *fit_coefs, const double *best,
                         const double *y_max, const double *lb, const double *ub, const uint8_t *cons_mask,
                         double *acq, double *grad, double *best_val, int64_t *best_idx, bool dev,
                         const double *prior_mean_grad = nullptr, void *stream = nullptr, const MixParams *mix = nullptr) {
  if (!slices || y_dim < 1 || n_samples < 1 || (!Xs && M > 0) || (!fit_coefs && !mix))
    return fail(BOSS_ERR_ARG, "boss_ei_score: bad arguments");
  int rc = check_lb_ub("boss_ei_score", lb, ub);
  if (rc) return rc;
  ScoreArgs a = score_args(slices, y_dim, n_samples, Xs, M, prior_mean_s, fit_coefs, best, y_max, lb, ub, cons_mask);
  a.acq = acq;
  a.grad = grad;
  a.prior_mean_grad = prior_mean_grad;
  a.best_val = best_val;
  a.best_idx = best_idx;
  a.dev = dev;
  a.caller_stream = stream;
  a.mix = mix;
  a.want_argmax = (best_val != nullptr) || (best_idx != nullptr);
  return score_dispatch(a);
}

int boss_ei_score(const boss_gp *const *slices, int y_dim, int n_samples, const double *Xs, int64_t M,
                  const double *prior_mean_s, const double *fit_coefs, const double *best, const double *y_max,
                  const double *lb, const double *ub, const uint8_t *cons_mask, double *acq, double *grad,
                  double *best_val, int64_t *best_idx) {
  return ei_score_impl(slices, y_dim, n_samples, Xs, M, prior_mean_s, fit_coefs, best, y_max, lb, ub, cons_mask, acq,
                       grad, best_val, best_idx, false);
}

int boss_ei_score_dev(const boss_gp *const *slices, int y_dim, int n_samples, const double *Xs_dev, int64_t M,
                      const double *prior_mean_s_dev, const double *fit_coefs, const double *best,
                      const double *y_max, const double *lb, const double *ub, const uint8_t *cons_mask_dev,
                      double *acq_dev, double *grad_dev, double *best_val, int64_t *best_idx, void *stream) {
  return ei_score_impl(slices, y_dim, n_samples, Xs_dev, M, prior_mean_s_dev, fit_coefs, best, y_max, lb, ub,
                       cons_mask_dev, acq_dev, grad_dev, best_val, best_idx, true, nullptr, stream);
}

// The k best candidates of boss_ei_score's scores (header: order, limits); screened like the argmax when `best` is set
// (DESIGN.md 2.10), otherwise the full path keeps a running top-k set on the device.
static int ei_score_topk_impl(const boss_gp *const *slices, int y_dim, int n_samples, const double *Xs, int64_t M,
                              const double *prior_mean_s, const double *fit_coefs, const double *best,
                              const double *y_max, const double *lb, const double *ub, const uint8_t *cons_mask,
                              int64_t k, double *top_val, int64_t *top_idx, bool dev, void *stream,
                              const MixParams *mix = nullptr) {
  if (!slices || y_dim < 1 || n_samples < 1 || !Xs || M < 1 || (!fit_coefs && !mix) || !top_val || !top_idx)
    return fail(BOSS_ERR_ARG, "boss_ei_score_topk: bad arguments");
  if (k < 1 || k > M || k > TOPK_MAX) return fail(BOSS_ERR_ARG, "boss_ei_score_topk: k must be in 1..min(M, 8192)");
  int rc = check_lb_ub("boss_ei_score_topk", lb, ub);
  if (rc) return rc;
  ScoreArgs a = score_args(slices, y_dim, n_samples, Xs, M, prior_mean_s, fit_coefs, best, y_max, lb, ub, cons_mask);
  a.dev = dev;
  a.caller_stream = stream;
  a.topk = k;
  a.top_val = top_val;
  a.top_idx = top_idx;
  a.mix = mix;
  return score_dispatch(a);
}

int boss_ei_score_topk(const boss_gp *const *slices, int y_dim, int n_samples, const double *Xs, int64_t M,
                       const double *prior_mean_s, const double *fit_coefs, const double *best, const double *y_max,
                       const double *lb, const double *ub, const uint8_t *cons_mask, int64_t k, double *top_val,
                       int64_t *top_idx) {
  return ei_score_topk_impl(slices, y_dim, n_samples, Xs, M, prior_mean_s, fit_coefs, best, y_max, lb, ub, cons_mask, k,
                            top_val, top_idx, false, nullptr);
}

int boss_ei_score_topk_dev(const boss_gp *const *slices, int y_dim, int n_samples, const double *Xs_dev, int64_t M,
                           const double *prior_mean_s_dev, const double *fit_coefs, const double *best,
                           const double *y_max, const double *lb, const double *ub, const uint8_t *cons_mask_dev,
                           int64_t k, double *top_val, int64_t *top_idx, void *stream) {
  return ei_score_topk_impl(slices, y_dim, n_samples, Xs_dev, M, prior_mean_s_dev, fit_coefs, best, y_max, lb, ub,
                            cons_mask_dev, k, top_val, top_idx, true, stream);
}

// Monte-Carlo EI of a NonlinFitness from the small expression set of MixParams (score.cuh), on the device:
// replaces expected_improvement(::NonlinFitness, ...) (src/acquisitions/expected_improvement.jl:104-111) inside the
// same construct_ei cases (:68-90).  eps is y_dim x n_eps (column-major, the reference's sample_eps matrix, :119);
// with n_samples > 1 posteriors (BI) posterior s gets column s (n_eps must equal n_samples, :87-90).
// The MixParams of one MC-EI call (the validation every boss_mcei_* entry point shares); eps stays a host pointer
static int mix_params(const char *who, int y_dim, int n_samples, int fit_kind, double fit_c0, const double *fit_c,
                      const double *fit_q, const double *fit_t, const double *eps, int n_eps, MixParams &mix) {
  const std::string w(who);
  if (fit_kind < 1 || fit_kind > 4) return fail(BOSS_ERR_ARG, w + ": fit_kind must be 1 (affine), 2 (quadratic), 3 (max) or 4 (min)");
  if (!eps || n_eps < 1 || y_dim < 1 || y_dim > MAX_YDIM) return fail(BOSS_ERR_ARG, w + ": bad eps / y_dim");
  if (n_eps > MIX_MAX_EPS) return fail(BOSS_ERR_ARG, w + ": more than 4096 eps samples");
  if (n_samples > 1 && n_eps != n_samples)
    return fail(BOSS_ERR_ARG, w + ": with BI posteriors eps must hold one column per posterior");
  mix = MixParams{};
  mix.kind = fit_kind;
  mix.n_eps = n_eps;
  mix.c0 = fit_c0;
  for (int i = 0; i < y_dim; ++i) {
    mix.c[i] = fit_c ? fit_c[i] : 0.0;
    mix.q[i] = fit_q ? fit_q[i] : 0.0;
    mix.t[i] = fit_t ? fit_t[i] : 0.0;
  }
  mix.eps_host = eps;
  return 0;
}

int boss_mcei_score(const boss_gp *const *slices, int y_dim, int n_samples, const double *Xs, int64_t M,
                    const double *prior_mean_s, int fit_kind, double fit_c0, const double *fit_c, const double *fit_q,
                    const double *fit_t, const double *eps, int n_eps, const double *best, const double *y_max,
                    const double *lb, const double *ub, const uint8_t *cons_mask, double *acq, double *best_val,
                    int64_t *best_idx) {
  MixParams mix;
  int rc = mix_params("boss_mcei_score", y_dim, n_samples, fit_kind, fit_c0, fit_c, fit_q, fit_t, eps, n_eps, mix);
  if (rc) return rc;
  return ei_score_impl(slices, y_dim, n_samples, Xs, M, prior_mean_s, nullptr, best, y_max, lb, ub, cons_mask, acq, nullptr,
                       best_val, best_idx, false, nullptr, nullptr, &mix);
}

int boss_mcei_value_grad(const boss_gp *const *slices, int y_dim, int n_samples, const double *Xs, int64_t M,
                         const double *prior_mean_s, const double *prior_mean_grad_s, int fit_kind, double fit_c0,
                         const double *fit_c, const double *fit_q, const double *fit_t, const double *eps, int n_eps,
                         const double *best, const double *y_max, const double *lb, const double *ub,
                         const uint8_t *cons_mask, double *acq, double *grad) {
  if (!grad) return fail(BOSS_ERR_ARG, "boss_mcei_value_grad: grad is NULL");
  MixParams mix;
  int rc = mix_params("boss_mcei_value_grad", y_dim, n_samples, fit_kind, fit_c0, fit_c, fit_q, fit_t, eps, n_eps, mix);
  if (rc) return rc;
  return ei_score_impl(slices, y_dim, n_samples, Xs, M, prior_mean_s, nullptr, best, y_max, lb, ub, cons_mask, acq, grad,
                       nullptr, nullptr, false, prior_mean_grad_s, nullptr, &mix);
}

int boss_mcei_score_topk(const boss_gp *const *slices, int y_dim, int n_samples, const double *Xs, int64_t M,
                         const double *prior_mean_s, int fit_kind, double fit_c0, const double *fit_c,
                         const double *fit_q, const double *fit_t, const double *eps, int n_eps, const double *best,
                         const double *y_max, const double *lb, const double *ub, const uint8_t *cons_mask, int64_t k,
                         double *top_val, int64_t *top_idx) {
  MixParams mix;
  int rc = mix_params("boss_mcei_score_topk", y_dim, n_samples, fit_kind, fit_c0, fit_c, fit_q, fit_t, eps, n_eps, mix);
  if (rc) return rc;
  return ei_score_topk_impl(slices, y_dim, n_samples, Xs, M, prior_mean_s, nullptr, best, y_max, lb, ub, cons_mask, k,
                            top_val, top_idx, false, nullptr, &mix);
}

static int ei_score_generated(const CandGen &gen, int64_t M, const boss_gp *const *slices, int y_dim, int n_samples,
                              const double *prior_mean_s, const double *fit_coefs, const double *best, const double *y_max,
                              const double *lb, const double *ub, const uint8_t *cons_mask, double *acq, double *best_val,
                              int64_t *best_idx, double *best_x) {
  if (!slices || y_dim < 1 || n_samples < 1 || !fit_coefs || !slices[0]) return fail(BOSS_ERR_ARG, "boss_ei_score_*: bad arguments");
  int rc = check_lb_ub("boss_ei_score_*", lb, ub);
  if (rc) return rc;
  if (gen.d != slices[0]->d) return fail(BOSS_ERR_ARG, "boss_ei_score_*: x_dim mismatch");
  ScoreArgs a = score_args(slices, y_dim, n_samples, nullptr, M, prior_mean_s, fit_coefs, best, y_max, lb, ub, cons_mask);
  a.acq = acq;
  int64_t bi = -1;
  double bv = 0.0;
  a.best_val = &bv;
  a.best_idx = &bi;
  a.want_argmax = true;
  a.gen = &gen;
  rc = score_dispatch(a);
  if (rc) return rc;
  if (best_val) *best_val = bv;
  if (best_idx) *best_idx = bi < 0 ? bi : gen.first + bi;                  // global index
  if (best_x && bi >= 0)
    for (int j = 0; j < gen.d; ++j) best_x[j] = cand_coord(gen, gen.first + bi, j);   // same arithmetic as the device generator
  return 0;
}

int boss_ei_score_grid(const boss_gp *const *slices, int y_dim, int n_samples, int d, const double *grid_lo,
                       const double *grid_step, const int64_t *grid_count, int64_t first, int64_t M,
                       const double *prior_mean_s, const double *fit_coefs, const double *best, const double *y_max,
                       const double *lb, const double *ub, const uint8_t *cons_mask, double *acq, double *best_val,
                       int64_t *best_idx, double *best_x) {
  if (d < 1 || d > 32 || !grid_lo || !grid_step || !grid_count || first < 0)
    return fail(BOSS_ERR_ARG, "boss_ei_score_grid: bad grid");
  CandGen gen{};
  gen.mode = 1;
  gen.d = d;
  gen.first = first;
  int64_t total = 1;
  for (int j = 0; j < d; ++j) {
    if (grid_count[j] < 1) return fail(BOSS_ERR_ARG, "boss_ei_score_grid: grid_count must be >= 1");
    gen.lo[j] = grid_lo[j];
    gen.step[j] = grid_step[j];
    gen.count[j] = grid_count[j];
    if (total > ((int64_t)1 << 40)) return fail(BOSS_ERR_ARG, "boss_ei_score_grid: grid too large");
    total *= grid_count[j];
  }
  if (M < 0) M = total - first;
  if (first + M > total) return fail(BOSS_ERR_ARG, "boss_ei_score_grid: shard exceeds the grid");
  return ei_score_generated(gen, M, slices, y_dim, n_samples, prior_mean_s, fit_coefs, best, y_max, lb, ub, cons_mask, acq,
                            best_val, best_idx, best_x);
}

int boss_ei_score_uniform(const boss_gp *const *slices, int y_dim, int n_samples, int d, uint64_t seed, int64_t first,
                          int64_t M, const double *box_lb, const double *box_ub, const double *prior_mean_s,
                          const double *fit_coefs, const double *best, const double *y_max, const uint8_t *cons_mask,
                          double *acq, double *best_val, int64_t *best_idx, double *best_x) {
  if (d < 1 || d > 32 || !box_lb || !box_ub || M < 0 || first < 0)
    return fail(BOSS_ERR_ARG, "boss_ei_score_uniform: bad arguments");
  CandGen gen{};
  gen.mode = 2;
  gen.d = d;
  gen.seed = seed;
  gen.first = first;
  for (int j = 0; j < d; ++j) {
    gen.lo[j] = box_lb[j];
    gen.step[j] = box_ub[j] - box_lb[j];
  }
  return ei_score_generated(gen, M, slices, y_dim, n_samples, prior_mean_s, fit_coefs, best, y_max, box_lb, box_ub,
                            cons_mask, acq, best_val, best_idx, best_x);
}

// Device-resident lock-step multi-start maximisation of the acquisition (multistart.cuh).
// the whole multi-start solve inside the current context (all starts on this device)
static int multistart_single(const boss_gp *const *slices, int y_dim, int n_samples, const double *starts, int64_t M,
                             int iters, int history, const double *prior_mean_affine, const double *fit_coefs,
                             const double *best, const double *y_max, const double *lb, const double *ub,
                             const uint8_t *discrete_mask, double *x_out, double *f_out, double *best_x,
                             double *best_val, int64_t *best_idx, int *evals_out, const MixParams *mix) {
  const int d = slices[0]->d;
  if (d > MS_MAXD) return fail(BOSS_ERR_ARG, "boss_ei_maximize_multistart: x_dim > 32");
  const int H = std::max(1, std::min(history, MS_MAXH - 1));
  const int RC = H + 1;   // ring capacity: H live pairs + one free slot for the pair being formed
  if (iters < 0) iters = 0;
  const size_t Md = (size_t)M * d;
  // the compact batch of a round holds `fan` trial points per unfinished start: up to MS_FAN_BATCH points once the
  // step-size fan is on (few starts left), never more than M points before that
  const size_t cap = (size_t)std::max<long long>(M, MS_FAN_BATCH), capd = cap * d;
  // carve one workspace: X g dirn | Sh Yh | f t | [affine mean scratch] | Xc gc fc | [MC-EI eps] | counters, per-start ints
  const size_t n_aff = prior_mean_affine ? (size_t)y_dim * (d + 1) + cap * y_dim + capd * y_dim : 0;
  const size_t n_eps = mix ? (size_t)y_dim * mix->n_eps : 0;
  const size_t n_dbl = 3 * Md + 2 * (size_t)RC * Md + 2 * (size_t)M + n_aff + 2 * capd + cap + n_eps;
  CUDA_TRY(C().ms_buf.ensure(n_dbl * 8 + (size_t)M * 24 + cap * 4 + 64));
  double *base = C().ms_buf.as<double>();
  MsState st{};
  st.d = d;
  st.H = RC;
  st.iters = iters;
  st.M = M;
  st.X = base;
  st.g = st.X + Md;
  st.dirn = st.g + Md;
  st.Sh = st.dirn + Md;
  st.Yh = st.Sh + (size_t)RC * Md;
  st.f = st.Yh + (size_t)RC * Md;
  st.t = st.f + M;
  double *aff = st.t + M, *pm = aff + (size_t)y_dim * (d + 1), *pmg = pm + cap * y_dim;
  if (prior_mean_affine)
    CUDA_TRY(cudaMemcpyAsync(aff, prior_mean_affine, (size_t)y_dim * (d + 1) * 8, cudaMemcpyHostToDevice, C().stream));
  st.Xc = st.t + M + n_aff;
  st.gc = st.Xc + capd;
  st.fc = st.gc + capd;
  // MC-EI: eps goes to the device once per solve; every round's scoring call then skips its own upload and wait
  MixParams mixd{};
  if (mix) {
    mixd = *mix;
    mixd.eps = st.fc + cap;
    mixd.eps_host = nullptr;
    CUDA_TRY(cudaMemcpyAsync(const_cast<double *>(mixd.eps), mix->eps_host, n_eps * 8, cudaMemcpyHostToDevice, C().stream));
  }
  st.counters = reinterpret_cast<int *>(st.fc + cap + n_eps);
  st.hist_len = st.counters + 4;
  st.hist_start = st.hist_len + M;
  st.trials = st.hist_start + M;
  st.steps = st.trials + M;
  st.state = st.steps + M;
  st.nev = st.state + M;
  st.idx = st.nev + M;      // [cap]
  st.fan = 1;
  double span = 0.0;
  for (int j = 0; j < d; ++j) {
    st.lb[j] = lb[j];
    st.ub[j] = ub[j];
    span = std::max(span, ub[j] - lb[j]);
  }
  st.step0 = 0.1 * span;
  const unsigned nbm = (unsigned)((M + 127) / 128);

  long long evaluated = 0;
  auto eval = [&](const double *Xp, long long Mp, double *fp, double *gp, bool want_best, double *bv, int64_t *bi) -> int {
    ScoreArgs a = score_args(slices, y_dim, n_samples, Xp, Mp, nullptr, fit_coefs, best, y_max, lb, ub, nullptr);
    evaluated += Mp;
    if (prior_mean_affine) {
      ms_affine_mean_kernel<<<(unsigned)((Mp + 127) / 128), 128, 0, C().stream>>>(Xp, Mp, d, y_dim, aff, pm, pmg);
      ++C().launches;
      a.prior_mean = pm;
      a.prior_mean_grad = gp ? pmg : nullptr;
    }
    a.acq = fp;
    a.grad = gp;
    a.best_val = bv;
    a.best_idx = bi;
    a.dev = true;
    a.internal = true;
    a.want_argmax = want_best;
    a.mix = mix ? &mixd : nullptr;
    return score_core(a);
  };

  // the pageable `starts` go through the synchronous copy path: the workspace is free (stream idle) at this point
  CUDA_TRY(cudaMemcpyAsync(st.Xc, starts, Md * 8, cudaMemcpyHostToDevice, C().stream));
  CUDA_TRY(cudaStreamSynchronize(C().stream));
  ms_init_kernel<<<nbm, 128, 0, C().stream>>>(st, st.Xc);
  ++C().launches;
  int rc = eval(st.X, M, st.f, st.g, false, nullptr, nullptr);
  if (rc) return rc;
  ms_sanitize_kernel<<<nbm, 128, 0, C().stream>>>(st.f, M);
  ++C().launches;
  // rounds: every unfinished start advances by one function evaluation.  A start needs `iters` accepted steps plus its
  // rejected trials; the budget below lets a start reject every other trial on average before it is cut off.
  const int max_rounds = iters > 0 ? 2 * iters + MS_MAX_TRIALS : 0;
  st.budget = max_rounds;   // enforced per start (ms_advance_kernel); the round loop below then ends by itself
  int active = iters > 0 ? (int)M : 0;
  const bool trace = getenv("BOSS_MS_TRACE") != nullptr;   // one line per round on stderr: round, batch size
  const bool use_fan = getenv("BOSS_MS_NO_FAN") == nullptr;
  CUDA_TRY(cudaMemsetAsync(st.counters, 0, 16, C().stream));
  int hc[3] = {0, 0, 0};
  for (int round = 0; round < max_rounds && active > 0; ++round) {
    // Step-size fan: below ~64 points a pass over W costs the same whatever the batch holds (the DMMA accumulation
    // chain of the last row block bounds it), so the next few backtracking trials are evaluated speculatively.
    int fan = 1;
    if (use_fan) fan = active <= 10 ? 6 : active <= 21 ? 3 : active <= 128 ? 2 : 1;
    fan = (int)std::max<size_t>(1, std::min<size_t>(fan, cap / (size_t)active));
    st.fan = fan;
    if (trace) {
      static thread_local double t_prev = 0.0;
      timespec ts;
      clock_gettime(CLOCK_MONOTONIC, &ts);
      const double t_now = ts.tv_sec * 1e6 + ts.tv_nsec * 1e-3;
      fprintf(stderr, "boss multistart: round %d active %d fan %d prev_round_us %.0f\n", round, active, fan,
              round ? t_now - t_prev : 0.0);
      t_prev = t_now;
    }
    CUDA_TRY(cudaMemsetAsync(st.counters, 0, 8, C().stream));
    ms_propose_kernel<<<nbm, 128, 0, C().stream>>>(st);
    rc = eval(st.Xc, (long long)active * fan, st.fc, st.gc, false, nullptr, nullptr);   // the compact list's length
    if (rc) return rc;
    ms_advance_kernel<<<(active + 127) / 128, 128, 0, C().stream>>>(st, active);
    C().launches += 2;
    CUDA_TRY(cudaMemcpyAsync(hc, st.counters, 12, cudaMemcpyDeviceToHost, C().stream));
    CUDA_TRY(cudaStreamSynchronize(C().stream));
    if (hc[0] != active * fan) return fail(BOSS_ERR_STATE, "boss_ei_maximize_multistart: internal batch-length mismatch");
    active = hc[1];
  }
  // what one-trial-per-round backtracking evaluates (same trajectory): first + trial + final evaluations
  const long long sequential_evals = 2 * M + hc[2];
  // final rounding of discrete dimensions and re-evaluation (optimization.jl:116-117), argmax over the starts
  const unsigned long long disc = mask_bits(discrete_mask, d);
  if (disc) ms_round_kernel<<<(unsigned)((Md + 255) / 256), 256, 0, C().stream>>>(st.X, M, d, disc);
  double bv = 0.0;
  int64_t bi = -1;
  rc = eval(st.X, M, st.f, nullptr, true, &bv, &bi);
  if (rc) return rc;
  if (x_out) CUDA_TRY(cudaMemcpyAsync(x_out, st.X, Md * 8, cudaMemcpyDeviceToHost, C().stream));
  if (f_out) CUDA_TRY(cudaMemcpyAsync(f_out, st.f, (size_t)M * 8, cudaMemcpyDeviceToHost, C().stream));
  if (best_x && bi >= 0) CUDA_TRY(cudaMemcpyAsync(best_x, st.X + (size_t)bi * d, (size_t)d * 8, cudaMemcpyDeviceToHost, C().stream));
  CUDA_TRY(cudaStreamSynchronize(C().stream));
  if (best_val) *best_val = bv;
  if (best_idx) *best_idx = bi;
  // work in units of full-batch evaluations: the evaluations of the sequential search; the speculative extra trials
  // of the fan (evaluated - sequential_evals of them) are reported through BOSS_MS_TRACE only
  if (trace)
    fprintf(stderr, "boss multistart: evaluated %lld points, %lld of them needed by the sequential search\n", evaluated,
            sequential_evals);
  if (evals_out) *evals_out = (int)((sequential_evals + M - 1) / M);
  return 0;
}

// one device, or contiguous ranges of starts dealt to the devices; mix == null: LinFitness (fit_coefs)
static int maximize_multistart_impl(const boss_gp *const *slices, int y_dim, int n_samples, const double *starts,
                                    int64_t M, int iters, int history, const double *prior_mean_affine,
                                    const double *fit_coefs, const double *best, const double *y_max, const double *lb,
                                    const double *ub, const uint8_t *discrete_mask, double *x_out, double *f_out,
                                    double *best_x, double *best_val, int64_t *best_idx, int *evals_out,
                                    const MixParams *mix) {
  if (!slices || !slices[0] || y_dim < 1 || n_samples < 1 || !starts || M < 1 || (!fit_coefs && !mix) || !lb || !ub)
    return fail(BOSS_ERR_ARG, "boss_ei_maximize_multistart: bad arguments (the box lb/ub is required)");
  const int nsl = y_dim * n_samples;
  for (int q = 0; q < nsl; ++q)
    if (!slices[q]) return fail(BOSS_ERR_ARG, "boss_ei_maximize_multistart: NULL slice handle");
  const int d = slices[0]->d;
  int nd = (g_ndev > 1 && tl_dev < 0) ? g_ndev : 1;
  for (int q = 0; q < nsl && nd > 1; ++q)
    for (int k = 0; k < nd; ++k)
      if (!replica_on(slices[q], k)) {
        nd = 1;
        break;
      }
  if (M < 256LL * nd) nd = 1;
  if (nd <= 1) {
    Ctx *cx = tl_dev >= 0 ? ctx_current() : ctx_of(slices[0]->dev);
    if (!cx) return fail(BOSS_ERR_STATE, "boss_ei_maximize_multistart: no usable device context for the handle");
    Enter en(cx);
    return multistart_single(slices, y_dim, n_samples, starts, M, iters, history, prior_mean_affine, fit_coefs, best, y_max,
                             lb, ub, discrete_mask, x_out, f_out, best_x, best_val, best_idx, evals_out, mix);
  }
  // multi-device: the starts are independent local solves (optimize_multistart, src/utils/optim_multistart.jl:10-90):
  // contiguous ranges of starts per device, the winners compared on the host in Julia's argmax order
  const int64_t per = ((M + nd - 1) / nd + 127) / 128 * 128;
  std::vector<double> bv(nd, 0.0), bx((size_t)nd * d, 0.0);
  std::vector<int64_t> bi(nd, -1), first(nd, 0), cnt(nd, 0);
  std::vector<int> ev(nd, 0);
  int rc = for_each_device(nd, [&](int k, Ctx *) {
    first[k] = std::min<int64_t>(M, (int64_t)k * per);
    cnt[k] = std::min<int64_t>(per, M - first[k]);
    if (cnt[k] <= 0) return 0;
    return multistart_single(slices, y_dim, n_samples, starts + (size_t)first[k] * d, cnt[k], iters, history,
                             prior_mean_affine, fit_coefs, best, y_max, lb, ub, discrete_mask,
                             x_out ? x_out + (size_t)first[k] * d : nullptr, f_out ? f_out + first[k] : nullptr,
                             bx.data() + (size_t)k * d, &bv[k], &bi[k], &ev[k], mix);
  });
  if (rc) return rc;
  double v = -std::numeric_limits<double>::infinity();
  int64_t ix = -1;
  int kbest = -1;
  for (int k = 0; k < nd; ++k) {
    if (cnt[k] <= 0 || bi[k] < 0) continue;
    const int64_t gi = first[k] + bi[k];
    if (ix < 0 || acq_better_host(bv[k], gi, v, ix)) {
      v = bv[k];
      ix = gi;
      kbest = k;
    }
  }
  if (best_val) *best_val = v;
  if (best_idx) *best_idx = ix;
  if (best_x && kbest >= 0)
    for (int j = 0; j < d; ++j) best_x[j] = bx[(size_t)kbest * d + j];
  if (evals_out) {
    *evals_out = 0;
    for (int k = 0; k < nd; ++k) *evals_out = std::max(*evals_out, ev[k]);
  }
  return 0;
}

int boss_ei_maximize_multistart(const boss_gp *const *slices, int y_dim, int n_samples, const double *starts, int64_t M,
                                int iters, int history, const double *prior_mean_affine, const double *fit_coefs,
                                const double *best, const double *y_max, const double *lb, const double *ub,
                                const uint8_t *discrete_mask, double *x_out, double *f_out, double *best_x,
                                double *best_val, int64_t *best_idx, int *evals_out) {
  if (!fit_coefs) return fail(BOSS_ERR_ARG, "boss_ei_maximize_multistart: bad arguments (the box lb/ub is required)");
  return maximize_multistart_impl(slices, y_dim, n_samples, starts, M, iters, history, prior_mean_affine, fit_coefs, best,
                                  y_max, lb, ub, discrete_mask, x_out, f_out, best_x, best_val, best_idx, evals_out,
                                  nullptr);
}

int boss_mcei_maximize_multistart(const boss_gp *const *slices, int y_dim, int n_samples, const double *starts,
                                  int64_t M, int iters, int history, const double *prior_mean_affine, int fit_kind,
                                  double fit_c0, const double *fit_c, const double *fit_q, const double *fit_t,
                                  const double *eps, int n_eps, const double *best, const double *y_max,
                                  const double *lb, const double *ub, const uint8_t *discrete_mask, double *x_out,
                                  double *f_out, double *best_x, double *best_val, int64_t *best_idx, int *evals_out) {
  MixParams mix;
  int rc = mix_params("boss_mcei_maximize_multistart", y_dim, n_samples, fit_kind, fit_c0, fit_c, fit_q, fit_t, eps, n_eps,
                      mix);
  if (rc) return rc;
  return maximize_multistart_impl(slices, y_dim, n_samples, starts, M, iters, history, prior_mean_affine, nullptr, best,
                                  y_max, lb, ub, discrete_mask, x_out, f_out, best_x, best_val, best_idx, evals_out, &mix);
}

int boss_ei_value_grad(const boss_gp *const *slices, int y_dim, int n_samples, const double *Xs, int64_t M,
                       const double *prior_mean_s, const double *prior_mean_grad_s, const double *fit_coefs,
                       const double *best, const double *y_max, const double *lb, const double *ub,
                       const uint8_t *cons_mask, double *acq, double *grad) {
  if (!grad) return fail(BOSS_ERR_ARG, "boss_ei_value_grad: grad is NULL");
  return ei_score_impl(slices, y_dim, n_samples, Xs, M, prior_mean_s, fit_coefs, best, y_max, lb, ub, cons_mask, acq,
                       grad, nullptr, nullptr, false, prior_mean_grad_s);
}

int boss_ei_value_grad_dev(const boss_gp *const *slices, int y_dim, int n_samples, const double *Xs_dev, int64_t M,
                           const double *prior_mean_s_dev, const double *prior_mean_grad_s_dev,
                           const double *fit_coefs, const double *best, const double *y_max, const double *lb,
                           const double *ub, const uint8_t *cons_mask_dev, double *acq_dev, double *grad_dev,
                           void *stream) {
  if (!grad_dev) return fail(BOSS_ERR_ARG, "boss_ei_value_grad_dev: grad is NULL");
  return ei_score_impl(slices, y_dim, n_samples, Xs_dev, M, prior_mean_s_dev, fit_coefs, best, y_max, lb, ub,
                       cons_mask_dev, acq_dev, grad_dev, nullptr, nullptr, true, prior_mean_grad_s_dev, stream);
}

int boss_gp_predict_grad(const boss_gp *const *slices, int y_dim, int n_samples, const double *Xs, int64_t M,
                         const double *prior_mean_s, const double *prior_mean_grad_s, double *mu, double *var,
                         double *dmu, double *dvar, int32_t *status) {
  if (!slices || y_dim < 1 || n_samples < 1 || (!Xs && M > 0))
    return fail(BOSS_ERR_ARG, "boss_gp_predict_grad: bad arguments");
  if (!dmu && !dvar)
    return fail(BOSS_ERR_ARG, "boss_gp_predict_grad: dmu and dvar are both NULL (boss_gp_predict gives mu and var alone)");
  ScoreArgs a = score_args(slices, y_dim, n_samples, Xs, M, prior_mean_s, nullptr, nullptr, nullptr, nullptr, nullptr,
                           nullptr);
  a.prior_mean_grad = prior_mean_grad_s;
  a.mu_out = mu;
  a.var_out = var;
  a.status_out = status;
  a.dmu_out = dmu;
  a.dvar_out = dvar;
  int rc = score_dispatch(a);
  if (rc) return rc;
  return a.any_fail ? BOSS_NEG_VARIANCE : 0;
}

int boss_gp_cov(const boss_gp *gp, const double *Xs, int64_t M, const double *prior_mean_s, double *mu, double *cov) {
  if (!gp || !Xs || !cov || M < 1) return fail(BOSS_ERR_ARG, "boss_gp_cov: bad arguments");
  REQUIRE_HANDLE_CTX(gp);
  if (M > 8192) return fail(BOSS_ERR_ARG, "boss_gp_cov: M > 8192 (the full covariance is meant for small batches)");
  const boss_gp *h = gp;
  const int d = h->d, ncb = (int)((M + 127) / 128), Mp = ncb * 128, cnt = Mp;
  const size_t blk_elems = (size_t)Mp * h->n_pad;
  CUDA_TRY(C().ks.ensure(blk_elems * 8));
  CUDA_TRY(C().vt.ensure(blk_elems * 8));
  CUDA_TRY(C().part_mu.ensure((size_t)2 * h->nblk * Mp * 8));
  CUDA_TRY(C().part_ss.ensure((size_t)2 * h->nblk * Mp * 8));
  CUDA_TRY(C().muv.ensure((size_t)Mp * 8));
  CUDA_TRY(C().cov_p.ensure((size_t)Mp * Mp * 8));
  CUDA_TRY(C().cov_stage.ensure((size_t)M * M * 8));
  CUDA_TRY(C().xs_stage.ensure((size_t)Mp * d * 8));
  CUDA_TRY(C().mu_stage.ensure((size_t)Mp * 8));
  CUDA_TRY(C().small.ensure(64));
  if (prior_mean_s) CUDA_TRY(C().pm_stage.ensure((size_t)M * 8));
  int *d_fail = C().small.as<int>();
  CUDA_TRY(cudaMemsetAsync(d_fail, 0, 4, C().stream));
  CUDA_TRY(cudaMemcpyAsync(C().xs_stage.p, Xs, (size_t)M * d * 8, cudaMemcpyHostToDevice, C().stream));
  if (prior_mean_s) CUDA_TRY(cudaMemcpyAsync(C().pm_stage.p, prior_mean_s, (size_t)M * 8, cudaMemcpyHostToDevice, C().stream));
  const int want = (2 * 148 + ncb - 1) / ncb;
  const int nks = std::max(1, std::min(h->nblk, want));
  const int nsp = pick_row_splits(ncb, h->nblk);
  launch_xcov(h->kernel_id, h->dp, xcov_params(h, C().xs_stage.as<double>(), M, 0, 0, d, Mp), dim3(ncb, nks), C().stream);
  reduce_rows_kernel<<<(cnt + 255) / 256, 256, 0, C().stream>>>(C().part_mu.as<double>(), 2 * h->nblk, (size_t)Mp,
                                                             C().muv.as<double>(), cnt);
  ScoreParams sp{};
  sp.W = h->W;
  sp.Ks = C().ks.as<double>();
  sp.nblk = h->nblk;
  sp.ktiles = h->ktiles;
  sp.ss_part = C().part_ss.as<double>();
  sp.ld = Mp;
  sp.VT = C().vt.as<double>();
  score_trmm_kernel<<<dim3(ncb, nsp), GEMM_THREADS, GEMM_SMEM_BYTES, C().stream>>>(sp);
  GemmNtParams gm{C().vt.as<double>(), C().vt.as<double>(), C().cov_p.as<double>(), h->ktiles, Mp / TK, 1};
  gemm_nt_kernel<<<dim3(ncb, ncb), GEMM_THREADS, GEMM_SMEM_BYTES, C().stream>>>(gm);
  CovFinishParams cf{};
  cf.Xs = C().xs_stage.as<double>();
  cf.M = (int)M;
  cf.d = d;
  cf.ktilesC = Mp / TK;
  cf.invl = h->invl;
  cf.disc_bits = h->disc;
  cf.a2 = h->a2;
  cf.C = C().cov_p.as<double>();
  cf.mu = C().muv.as<double>();
  cf.prior_mean = prior_mean_s ? C().pm_stage.as<double>() : nullptr;
  cf.mu_out = mu ? C().mu_stage.as<double>() : nullptr;
  cf.cov = C().cov_stage.as<double>();
  cf.any_fail = d_fail;
  cf.rq_a = h->rq_a;
  launch_cov_finish(h->kernel_id, h->dp, cf, dim3((unsigned)((M + 15) / 16), (unsigned)((M + 15) / 16)), C().stream);
  C().launches += 5;
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaMemcpyAsync(cov, C().cov_stage.p, (size_t)M * M * 8, cudaMemcpyDeviceToHost, C().stream));
  if (mu) CUDA_TRY(cudaMemcpyAsync(mu, C().mu_stage.p, (size_t)M * 8, cudaMemcpyDeviceToHost, C().stream));
  int hfail = 0;
  CUDA_TRY(cudaMemcpyAsync(&hfail, d_fail, 4, cudaMemcpyDeviceToHost, C().stream));
  CUDA_TRY(cudaStreamSynchronize(C().stream));
  return hfail ? BOSS_NEG_VARIANCE : 0;
}

// ---------------------------------------------------------------------------------------------
// batched log marginal likelihood
// ---------------------------------------------------------------------------------------------
// restores the context's main stream when a log-likelihood window leaves early (its groups run on their own streams)
struct StreamGuard {
  cudaStream_t keep;
  StreamGuard() : keep(C().stream) {}
  ~StreamGuard() { C().stream = keep; }
};

// Prior-mean Jacobian of boss_gp_loglik_grad_batch_mean: J (sample s at J + s*ldj, ldj == 0 shared, n x k column-major
// inside a sample) in, alpha^T J (S x k) out.  Only the gradient mode takes one.
struct MeanJac {
  const double *J;
  int k;
  int64_t ldj;
  double *grad_mean;
};

// one batch inside the current context
// internal: a call from inside another entry point on device inputs already ordered on the library stream (the
// hyper-parameter driver, boss_gp_map_multistart): no caller-stream wait, and the call returns without synchronising
static int loglik_core(const double *X, int d, int n, const double *Ymm, int64_t ldy, const double *ls,
                       const double *amp, const double *noise, KernelSpec ks, const uint8_t *discrete_mask, int64_t S,
                       double *loglik, bool dev, double *grad, boss_gp **fit_out, void *caller_stream,
                       const MeanJac *mj = nullptr, bool internal = false) {
  const int dp = pick_dp(d), kernel_id = ks.kid;
  if (S == 0) return 0;
  if (dev && !internal) {
    int rc = wait_for_caller(caller_stream);
    if (rc) return rc;
  }
  StreamGuard stream_guard;
  const int n_pad = round_up(n, TM), nblk = n_pad / TM, ktiles = n_pad / TK;
  const size_t mat = (size_t)n_pad * n_pad;
  const unsigned long long disc = mask_bits(discrete_mask, d);

  const bool need_w = grad || fit_out;        // gradient and batched-fit modes also form W = L^-1, W^T and alpha
  const bool small = n <= SMALL_N && !need_w; // warp-register path (small.cuh): no workspace at all
  // sub-batch so that L + Winv (+ W, W^T and the trtri scratch) stay within a 32 GiB workspace
  const size_t per = (need_w ? 3 : 1) * mat * 8 + (size_t)(need_w ? 2 * nblk : nblk) * TM * TM * 8;
  long long Sb = std::max<long long>(1, std::min<long long>(S, (32ll << 30) / (long long)per));
  Sb = std::min<long long>(Sb, 32768);
  if (small) Sb = 1;
  if (!small) {
    CUDA_TRY(C().chol_L.ensure((size_t)Sb * mat * 8));
    CUDA_TRY(C().chol_Winv.ensure((size_t)Sb * nblk * TM * TM * 8));
  }
  const int ntiles = nblk * (nblk + 1) / 2;
  const size_t tt_stride = (size_t)std::max(1, nblk - 1) * TM * TM;
  if (need_w) {
    CUDA_TRY(C().chol_W.ensure((size_t)Sb * mat * 8));
    CUDA_TRY(C().chol_WT.ensure((size_t)Sb * mat * 8));
    CUDA_TRY(C().ll_vec.ensure((size_t)Sb * n_pad * 3 * 8));                 // delta_pad | w | alpha
    if (grad) CUDA_TRY(C().ll_part.ensure((size_t)Sb * ntiles * (dp + 2) * 8));
  }

  // device copies of the inputs when called with host pointers
  const double *dX = X, *dY = Ymm, *dls = ls, *damp = amp, *dnoise = noise, *dJ = mj ? mj->J : nullptr;
  double *dll = loglik;
  const size_t ycount = ldy ? (size_t)S * ldy : (size_t)n;
  // the last sample's Jacobian ends at k*n: a caller stride ldj > k*n need not be padded after it
  const size_t jcount = !mj ? 0 : (size_t)mj->k * n + (mj->ldj ? (size_t)(S - 1) * mj->ldj : 0);
  // misc: [X | Y | J | ls | amp | noise | ll] (host variant) then grad | grad_mean (host variant, gradient mode) then
  // logdet_blk[Sb*nblk] | ssq_blk[Sb*nblk] | r, w [Sb*n_pad] | status[Sb]
  size_t off = 0, oX = 0, oY = 0, oJ = 0, ols = 0, oamp = 0, onoise = 0, oll = 0;
  if (!dev) {
    oX = off; off += (size_t)n * d;
    oY = off; off += ycount;
    oJ = off; off += jcount;
    ols = off; off += (size_t)S * d;
    oamp = off; off += S;
    onoise = off; off += S;
    oll = off; off += S;
  }
  size_t ogr = 0, ogm = 0;
  if (!dev && grad) {
    ogr = off; off += (size_t)S * (d + 2);
  }
  if (!dev && mj) {
    ogm = off; off += (size_t)S * mj->k;
  }
  const size_t old_ = off;
  off += (size_t)Sb * nblk;
  const size_t ossq = off;                      // |w_j|^2 per block, then r and w of the in-line forward substitution
  off += (size_t)Sb * nblk;
  const size_t orv = off;
  off += small ? 0 : (size_t)Sb * n_pad;
  const size_t owv = off;
  off += small ? 0 : (size_t)Sb * n_pad;
  const size_t ost = off;
  off += (size_t)(Sb + 1) / 2 + 1;
  CUDA_TRY(C().chol_misc.ensure(off * 8));
  double *misc = C().chol_misc.as<double>();
  if (!dev) {
    CUDA_TRY(cudaMemcpyAsync(misc + oX, X, (size_t)n * d * 8, cudaMemcpyHostToDevice, C().stream));
    CUDA_TRY(cudaMemcpyAsync(misc + oY, Ymm, ycount * 8, cudaMemcpyHostToDevice, C().stream));
    if (mj) {
      CUDA_TRY(cudaMemcpyAsync(misc + oJ, mj->J, jcount * 8, cudaMemcpyHostToDevice, C().stream));
      dJ = misc + oJ;
    }
    CUDA_TRY(cudaMemcpyAsync(misc + ols, ls, (size_t)S * d * 8, cudaMemcpyHostToDevice, C().stream));
    CUDA_TRY(cudaMemcpyAsync(misc + oamp, amp, (size_t)S * 8, cudaMemcpyHostToDevice, C().stream));
    CUDA_TRY(cudaMemcpyAsync(misc + onoise, noise, (size_t)S * 8, cudaMemcpyHostToDevice, C().stream));
    dX = misc + oX; dY = misc + oY; dls = misc + ols; damp = misc + oamp; dnoise = misc + onoise; dll = misc + oll;
  }
  double *dgrad = (grad && !dev) ? misc + ogr : grad;
  double *dgm = !mj ? nullptr : dev ? mj->grad_mean : misc + ogm;
  double *logdet_blk = misc + old_;
  int *status = reinterpret_cast<int *>(misc + ost);

  if (!internal) timing_begin();
  if (small) {
    SmallLoglikParams sp{};
    sp.X = dX;
    sp.d = d;
    sp.n = n;
    sp.ymm = dY;
    sp.ldy = ldy;
    sp.ls = dls;
    sp.amp = damp;
    sp.noise = dnoise;
    sp.disc_bits = disc;
    sp.S = S;
    sp.loglik = dll;
    sp.rq_a = ks.rq_a;
    Timed t(2);
    launch_loglik_small(kernel_id, dp, sp, (int)((S + SMALL_WARPS - 1) / SMALL_WARPS), C().stream);
    ++C().launches;
  }
  // A window of up to Sb matrices is live at a time.  Inside a window the matrices are processed as up to
  // LL_GROUPS independent groups on separate streams: one group's latency-bound steps (diagonal-block
  // factorisation, forward solve) and partially filled last waves overlap with another group's GEMM launches.
  cudaStream_t main_stream = C().stream;
  const size_t winv_stride = (size_t)nblk * TM * TM;
  for (long long s0 = 0; s0 < S && !small; s0 += Sb) {
    const int sb = (int)std::min<long long>(Sb, S - s0);
    // 4 concurrent groups for long factorisations; 2 for small matrices, whose diagonal-block launches (one CTA per
    // matrix, two to an SM) then come closer to filling the GPU (C3, 512 matrices of n = 512: 1.57 vs 1.61 ms)
    int want_groups = nblk <= 6 ? 2 : 4;
    if (const char *e = getenv("BOSS_LL_GROUPS")) want_groups = std::max(1, std::min(LL_GROUPS, atoi(e)));
    const int ngroups = (C().timing || sb < 2 * want_groups) ? 1 : want_groups;   // per-kernel-class timing needs one stream
    const int gsz = (sb + ngroups - 1) / ngroups;
    if (ngroups > 1) CUDA_TRY(cudaEventRecord(C().ll_fork, main_stream));
    int rc_all = 0;
    for (int gi = 0; gi < ngroups; ++gi) {
      const int wo = gi * gsz;                           // offset of the group inside the window
      const int gs = std::min(gsz, sb - wo);
      if (gs <= 0) break;
      const long long so = s0 + wo;                      // offset of the group inside the batch
      if (ngroups > 1) {
        C().stream = C().ll_stream[gi];
        CUDA_TRY(cudaStreamWaitEvent(C().stream, C().ll_fork, 0));
      }
      double *Lg = C().chol_L.as<double>() + (size_t)wo * mat;
      double *Wig = C().chol_Winv.as<double>() + (size_t)wo * winv_stride;
      double *ldg = logdet_blk + (size_t)wo * nblk;
      int *stg = status + wo;
      double *Wg = need_w ? C().chol_W.as<double>() + (size_t)wo * mat : nullptr;
      double *WTg = need_w ? C().chol_WT.as<double>() + (size_t)wo * mat : nullptr;
      double *TTg = nullptr;   // the fused triangular-inverse step keeps T on chip
      CUDA_TRY(cudaMemsetAsync(stg, 0, (size_t)gs * 4, C().stream));
      BuildKParams bk{};
      bk.X = dX;
      bk.d = d;
      bk.n = n;
      bk.nblk = nblk;
      bk.ktiles = ktiles;
      bk.ls = dls + (size_t)so * d;
      bk.amp = damp + so;
      bk.noise = dnoise + so;
      bk.disc_bits = disc;
      bk.K = Lg;
      bk.K_stride = mat;
      bk.status = stg;
      bk.rq_a = ks.rq_a;
      // Fused diagonal step (K_jj generated on chip + SYRK + potrf in one 2-CTA/SM kernel) for small matrices, where the
      // three short launches and the tile's HBM trip dominate (C3, n = 512: 1.61 -> 1.55 ms); for long k-ranges the
      // dedicated SYRK kernel (5-stage ring, 218 registers) runs its DMMAs at 75 % of the SM's rate against 51 % for the
      // 128-register fused one (11.8 vs 17.5 us per 128-block of k at n = 2048), so larger matrices keep the separate steps.
      const bool fuse_diag = nblk <= 6;
      bk.skip_diag = fuse_diag ? 1 : 0;     // the diagonal tiles are generated inside potrf_fused_kernel
      if (!(fuse_diag && nblk == 1)) {
        Timed t(1);
        launch_build_k(kernel_id, dp, bk, dim3(nblk * (nblk + 1) / 2, gs), C().stream);
        ++C().launches;
      }
      if (need_w) {   // zero initial state of W and W^T (strictly-upper resp. strictly-lower blocks are never written)
        CUDA_TRY(cudaMemsetAsync(Wg, 0, (size_t)gs * mat * 8, C().stream));
        CUDA_TRY(cudaMemsetAsync(WTg, 0, (size_t)gs * mat * 8, C().stream));
      }
      FwdInline fw{dY + (ldy ? (size_t)so * ldy : 0), ldy, n, n_pad, misc + orv + (size_t)wo * n_pad,
                   misc + owv + (size_t)wo * n_pad, misc + ossq + (size_t)wo * nblk};
      int rc = run_cholesky(Lg, mat, Wig, winv_stride, nblk, ktiles, gs, ldg, stg, Wg, WTg, TTg, mat, tt_stride, false, &fw,
                            fuse_diag ? &bk : nullptr, kernel_id, dp, fit_out != nullptr);
      if (rc) rc_all = rc;
      loglik_finish_kernel<<<(gs + 127) / 128, 128, 0, C().stream>>>(ldg, fw.ssq, stg, nblk, n, gs, dll + so);
      ++C().launches;
      double *vec = C().ll_vec.as<double>();
      double *dpad = vec + (size_t)wo * n_pad, *wv = vec + ((size_t)Sb + wo) * n_pad, *al = vec + ((size_t)2 * Sb + wo) * n_pad;
      if (need_w) {   // alpha = W^T (W delta)
        pad_delta_kernel<<<dim3((n_pad + 255) / 256, gs), 256, 0, C().stream>>>(dY + (ldy ? (size_t)so * ldy : 0), ldy, n, n_pad, dpad);
        matvec_p_kernel<<<dim3(n_pad / 64, gs), 256, 0, C().stream>>>(Wg, dpad, wv, ktiles, mat, n_pad, n_pad);
        matvec_p_kernel<<<dim3(n_pad / 64, gs), 256, 0, C().stream>>>(WTg, wv, al, ktiles, mat, n_pad, n_pad);
        C().launches += 3;
      }
      if (mj) {   // prior-mean gradient alpha^T J: reads alpha only, so the hyper-parameter gradient below is unchanged
        loglik_mean_grad_kernel<<<dim3(mj->k, gs), 128, 0, C().stream>>>(al, n_pad, dJ + (size_t)so * mj->ldj, mj->ldj, n,
                                                                        mj->k, stg, dgm + (size_t)so * mj->k);
        ++C().launches;
      }
      if (grad) {
        // K^-1 = W^T W over the factor's storage;  tile partial sums;  final scaling
        double *partg = C().ll_part.as<double>() + (size_t)wo * ntiles * (dp + 2);
        KinvParams kp{WTg, mat, Lg, mat, nblk, ktiles};
        {
          Timed t(2);
          kinv_wtw_kernel<<<dim3(ntiles, gs), GEMM_THREADS, GEMM_SMEM_BYTES, C().stream>>>(kp);
        }
        LlGradParams lg{};
        lg.X = dX;
        lg.d = d;
        lg.n = n;
        lg.nblk = nblk;
        lg.ktiles = ktiles;
        lg.ls = dls + (size_t)so * d;
        lg.amp = damp + so;
        lg.noise = dnoise + so;
        lg.disc_bits = disc;
        lg.Kinv = Lg;
        lg.K_stride = mat;
        lg.alpha = al;
        lg.part = partg;
        lg.rq_a = ks.rq_a;
        {
          Timed t(1);
          launch_loglik_grad_tile(kernel_id, dp, lg, dim3(ntiles, gs), C().stream);
        }
        loglik_grad_final_kernel<<<(gs + 127) / 128, 128, 0, C().stream>>>(partg, ntiles, dp, d, lg.ls, lg.amp, lg.noise, stg,
                                                                        dgrad + (size_t)so * (d + 2), gs);
        C().launches += 3;
      }
      if (ngroups > 1) {
        CUDA_TRY(cudaEventRecord(C().ll_join[gi], C().stream));
        C().stream = main_stream;
        CUDA_TRY(cudaStreamWaitEvent(main_stream, C().ll_join[gi], 0));
      }
    }
    C().stream = main_stream;
    if (rc_all) return rc_all;
    if (fit_out) {
      // batched posterior fit: detach every factorisation of the window into its own handle
      std::vector<int> hst(sb);
      std::vector<double> hll(sb);
      CUDA_TRY(cudaMemcpyAsync(hst.data(), status, (size_t)sb * 4, cudaMemcpyDeviceToHost, C().stream));
      CUDA_TRY(cudaMemcpyAsync(hll.data(), dll + s0, (size_t)sb * 8, cudaMemcpyDeviceToHost, C().stream));
      CUDA_TRY(cudaStreamSynchronize(C().stream));
      double *vec = C().ll_vec.as<double>();
      for (int q = 0; q < sb; ++q) {
        const long long sidx = s0 + q;
        fit_out[sidx] = nullptr;
        if (hst[q] != 0) continue;
        boss_gp *h = new boss_gp();
        h->n = n; h->d = d; h->n_pad = n_pad; h->nblk = nblk; h->ktiles = ktiles; h->kernel_id = kernel_id; h->dp = dp;
        h->rq_a = ks.rq_a;
        h->disc = disc;
        h->amp = amp[sidx] + MIN_PARAM_VALUE;
        h->noise = noise[sidx] + MIN_PARAM_VALUE;
        h->a2 = h->amp * h->amp;
        h->loglik = hll[q];
        cudaError_t e = cudaSuccess;
        for (auto pr : {std::make_pair(&h->L, mat * 8), std::make_pair(&h->W, mat * 8), std::make_pair(&h->WT, mat * 8),
                        std::make_pair(&h->alpha, (size_t)n_pad * 8), std::make_pair(&h->Xt, (size_t)n_pad * dp * 8),
                        std::make_pair(&h->invl, (size_t)dp * 8), std::make_pair(&h->wvec, (size_t)n_pad * 8),
                        std::make_pair(&h->ymm, (size_t)n_pad * 8)})
          if (e == cudaSuccess) e = pool_alloc(pr.first, pr.second);
        if (e != cudaSuccess) {
          h->free_dev();
          delete h;
          return fail(BOSS_ERR_CUDA, std::string("boss_gp_fit_batch: ") + cudaGetErrorString(e));
        }
        std::vector<double> invl(dp, 0.0);
        for (int i = 0; i < d; ++i) invl[i] = 1.0 / (ls[(size_t)sidx * d + i] + MIN_PARAM_VALUE);
        cudaMemcpyAsync(h->invl, invl.data(), (size_t)dp * 8, cudaMemcpyHostToDevice, C().stream);
        cudaStreamSynchronize(C().stream);   // invl is a stack temporary
        cudaMemcpyAsync(h->L, C().chol_L.as<double>() + (size_t)q * mat, mat * 8, cudaMemcpyDeviceToDevice, C().stream);
        cudaMemcpyAsync(h->W, C().chol_W.as<double>() + (size_t)q * mat, mat * 8, cudaMemcpyDeviceToDevice, C().stream);
        cudaMemcpyAsync(h->WT, C().chol_WT.as<double>() + (size_t)q * mat, mat * 8, cudaMemcpyDeviceToDevice, C().stream);
        cudaMemcpyAsync(h->ymm, vec + (size_t)q * n_pad, (size_t)n_pad * 8, cudaMemcpyDeviceToDevice, C().stream);
        cudaMemcpyAsync(h->wvec, vec + ((size_t)Sb + q) * n_pad, (size_t)n_pad * 8, cudaMemcpyDeviceToDevice, C().stream);
        cudaMemcpyAsync(h->alpha, vec + ((size_t)2 * Sb + q) * n_pad, (size_t)n_pad * 8, cudaMemcpyDeviceToDevice, C().stream);
        scale_train_kernel<<<(n_pad * dp + 255) / 256, 256, 0, C().stream>>>(dX, d, n, n_pad, dp, h->invl, disc, h->Xt);
        ++C().launches;
        h->dev = C().device;
        h->rep[h->dev] = h;
        C().live.insert(h);
        fit_out[sidx] = h;
      }
      CUDA_TRY(cudaGetLastError());
      CUDA_TRY(cudaStreamSynchronize(C().stream));
    }
  }
  CUDA_TRY(cudaGetLastError());
  if (!dev) CUDA_TRY(cudaMemcpyAsync(loglik, dll, (size_t)S * 8, cudaMemcpyDeviceToHost, C().stream));
  if (!dev && grad) CUDA_TRY(cudaMemcpyAsync(grad, dgrad, (size_t)S * (d + 2) * 8, cudaMemcpyDeviceToHost, C().stream));
  if (!dev && mj)
    CUDA_TRY(cudaMemcpyAsync(mj->grad_mean, dgm, (size_t)S * mj->k * 8, cudaMemcpyDeviceToHost, C().stream));
  if (internal) return 0;
  CUDA_TRY(cudaStreamSynchronize(C().stream));
  timing_end();
  if (!dev) {
    int any = 0;
    for (int64_t s = 0; s < S; ++s)
      if (std::isinf(loglik[s]) && loglik[s] < 0) any = 1;
    return any ? BOSS_NOT_POSDEF : 0;
  }
  return 0;
}

// Argument checks (the reference's asserts, src/models/gaussian_process.jl:227-229, are made on the host where the
// hyper-parameters are host arrays), then one device or -- multi-device mode, host arrays -- contiguous sample ranges
// dealt to the devices.  A sample's value does not depend on the batch it is evaluated in (left-looking
// factorisation, fixed-order sums), so the sharded result is bit-identical to the single-device one.
static int loglik_impl(const double *X, int d, int n, const double *Ymm, int64_t ldy, const double *ls,
                       const double *amp, const double *noise, int kernel_id, const uint8_t *discrete_mask, int64_t S,
                       double *loglik, bool dev, double *grad = nullptr, boss_gp **fit_out = nullptr,
                       void *caller_stream = nullptr, const MeanJac *mj = nullptr) {
  if (!X || !Ymm || !ls || !amp || !noise || !loglik || d < 1 || n < 1 || S < 0)
    return fail(BOSS_ERR_ARG, "boss_gp_loglik_batch: bad arguments");
  KernelSpec ks;
  if (!decode_kernel(kernel_id, &ks)) return fail(BOSS_ERR_ARG, "boss_gp_loglik_batch: unknown kernel_id");
  if (pick_dp(d) < 0) return fail(BOSS_ERR_ARG, "boss_gp_loglik_batch: x_dim > 32 is not supported");
  if (!dev) {
    for (int64_t s = 0; s < S; ++s) {
      for (int i = 0; i < d; ++i)
        if (!(ls[(size_t)s * d + i] >= 0)) return fail(BOSS_ERR_ARG, "boss_gp_loglik_batch: negative (or NaN) lengthscale");
      if (!(amp[s] >= 0) || !(noise[s] >= 0))
        return fail(BOSS_ERR_ARG, "boss_gp_loglik_batch: negative (or NaN) amplitude / noise_std");
    }
  }
  const int nd = (g_ndev > 1 && tl_dev < 0 && !dev && !fit_out && S >= 2LL * g_ndev) ? g_ndev : 1;
  if (nd <= 1) {
    REQUIRE_INIT();
    return loglik_core(X, d, n, Ymm, ldy, ls, amp, noise, ks, discrete_mask, S, loglik, dev, grad, fit_out, caller_stream,
                       mj);
  }
  const int64_t per = (S + nd - 1) / nd;
  int rc = for_each_device(nd, [&](int k, Ctx *) {
    const int64_t s0 = std::min<int64_t>(S, (int64_t)k * per), cnt = std::min<int64_t>(per, S - s0);
    if (cnt <= 0) return 0;
    MeanJac mjk{};
    if (mj) mjk = MeanJac{mj->J + (size_t)s0 * mj->ldj, mj->k, mj->ldj, mj->grad_mean + (size_t)s0 * mj->k};
    return loglik_core(X, d, n, ldy ? Ymm + (size_t)s0 * ldy : Ymm, ldy, ls + (size_t)s0 * d, amp + s0, noise + s0, ks,
                       discrete_mask, cnt, loglik + s0, false, grad ? grad + (size_t)s0 * (d + 2) : nullptr,
                       fit_out ? fit_out + s0 : nullptr, nullptr, mj ? &mjk : nullptr);
  });
  return rc;
}

int boss_gp_loglik_batch(const double *X, int d, int n, const double *Y_minus_mean, int64_t ldy,
                         const double *lengthscales, const double *amplitude, const double *noise_std, int kernel_id,
                         const uint8_t *discrete_mask, int64_t S, double *loglik) {
  return loglik_impl(X, d, n, Y_minus_mean, ldy, lengthscales, amplitude, noise_std, kernel_id, discrete_mask, S,
                     loglik, false);
}
int boss_gp_loglik_batch_dev(const double *X_dev, int d, int n, const double *Y_minus_mean_dev, int64_t ldy,
                             const double *lengthscales_dev, const double *amplitude_dev, const double *noise_std_dev,
                             int kernel_id, const uint8_t *discrete_mask, int64_t S, double *loglik_dev, void *stream) {
  return loglik_impl(X_dev, d, n, Y_minus_mean_dev, ldy, lengthscales_dev, amplitude_dev, noise_std_dev, kernel_id,
                     discrete_mask, S, loglik_dev, true, nullptr, nullptr, stream);
}

int boss_gp_fit_batch(const double *X, int d, int n, const double *Y_minus_mean, int64_t ldy, const double *lengthscales,
                      const double *amplitude, const double *noise_std, int kernel_id, const uint8_t *discrete_mask,
                      int64_t S, boss_gp **out, double *loglik_out) {
  if (!out) return fail(BOSS_ERR_ARG, "boss_gp_fit_batch: out is NULL");
  for (int64_t s = 0; s < S; ++s) out[s] = nullptr;
  std::vector<double> ll((size_t)std::max<int64_t>(S, 1));
  int rc;
  if (g_ndev > 1 && tl_dev < 0 && S > 0) {
    // multi-device mode: every device fits all S posteriors (replicas), exactly like boss_gp_fit
    const int nd = g_ndev;
    std::vector<std::vector<boss_gp *>> reps(nd, std::vector<boss_gp *>((size_t)S, nullptr));
    std::vector<std::vector<double>> lls(nd, std::vector<double>((size_t)S, 0.0));
    KernelSpec ks;
    if (!X || !Y_minus_mean || !lengthscales || !amplitude || !noise_std || d < 1 || n < 1 ||
        !decode_kernel(kernel_id, &ks) || pick_dp(d) < 0)
      return fail(BOSS_ERR_ARG, "boss_gp_fit_batch: bad arguments");
    rc = for_each_device(nd, [&](int k, Ctx *) {
      return loglik_core(X, d, n, Y_minus_mean, ldy, lengthscales, amplitude, noise_std, ks, discrete_mask, S,
                         lls[k].data(), false, nullptr, reps[k].data(), nullptr);
    });
    ll = lls[0];
    if (rc >= 0) {
      for (int64_t s = 0; s < S; ++s) {
        bool all = true;
        for (int k = 0; k < nd; ++k) all = all && reps[k][s];
        if (!all) {   // not positive definite (on every device alike)
          for (int k = 0; k < nd; ++k) free_replica(reps[k][s]);
          continue;
        }
        std::vector<boss_gp *> r(nd);
        for (int k = 0; k < nd; ++k) r[k] = reps[k][s];
        out[s] = link_replicas(r);
      }
    } else {
      const std::string keep = tl_err;
      for (int k = 0; k < nd; ++k)
        for (boss_gp *r : reps[k]) free_replica(r);
      tl_err = keep;
    }
  } else {
    rc = loglik_impl(X, d, n, Y_minus_mean, ldy, lengthscales, amplitude, noise_std, kernel_id, discrete_mask, S, ll.data(),
                     false, nullptr, out);
    if (rc < 0)
      for (int64_t s = 0; s < S; ++s)
        if (out[s]) {
          boss_gp_free(out[s]);
          out[s] = nullptr;
        }
  }
  if (loglik_out)
    for (int64_t s = 0; s < S; ++s) loglik_out[s] = ll[s];
  return rc;
}

int boss_gp_loglik_grad_batch(const double *X, int d, int n, const double *Y_minus_mean, int64_t ldy,
                              const double *lengthscales, const double *amplitude, const double *noise_std, int kernel_id,
                              const uint8_t *discrete_mask, int64_t S, double *loglik, double *grad) {
  if (!grad) return fail(BOSS_ERR_ARG, "boss_gp_loglik_grad_batch: grad is NULL");
  return loglik_impl(X, d, n, Y_minus_mean, ldy, lengthscales, amplitude, noise_std, kernel_id, discrete_mask, S, loglik,
                     false, grad);
}
int boss_gp_loglik_grad_batch_dev(const double *X_dev, int d, int n, const double *Y_minus_mean_dev, int64_t ldy,
                                  const double *lengthscales_dev, const double *amplitude_dev, const double *noise_std_dev,
                                  int kernel_id, const uint8_t *discrete_mask, int64_t S, double *loglik_dev,
                                  double *grad_dev, void *stream) {
  if (!grad_dev) return fail(BOSS_ERR_ARG, "boss_gp_loglik_grad_batch_dev: grad is NULL");
  return loglik_impl(X_dev, d, n, Y_minus_mean_dev, ldy, lengthscales_dev, amplitude_dev, noise_std_dev, kernel_id,
                     discrete_mask, S, loglik_dev, true, grad_dev, nullptr, stream);
}

// ---------------------------------------------------------------------------------------------
// device-resident MAP fit of the hyper-parameters (OptimizationMAP, DESIGN.md 2.15)
// ---------------------------------------------------------------------------------------------
// The (slice, start) pairs [pair0, pair0 + Mloc) inside the current context: the acquisition driver's projected L-BFGS
// state machine (multistart.cuh) at capacity MS_MAP_MAXD, every round's trial points evaluated by one internal
// loglik_core call between map_prep_kernel and map_prior_kernel.  Returns each pair's final value and raw parameters
// (raw_out [Mloc][P], as evaluated on the device) and the number of evaluations made.
static int map_multistart_single(const double *X, int d, int n, int y_dim, const double *Y, KernelSpec ks,
                                 const uint8_t *discrete_mask, const int32_t *kind, const double *par,
                                 const double *starts_z, int64_t pair0, int64_t Mslice, int64_t Mloc, int iters,
                                 int history, double *raw_out, double *f_out, long long *evals) {
  const int P = d + 2;
  const int H = std::max(1, std::min(history, MS_MAXH - 1));
  const int RC = H + 1;
  if (iters < 0) iters = 0;
  const long long M = Mloc;
  const size_t MP = (size_t)M * P, cap = (size_t)M;   // step-size fan 1: a round's batch holds at most M points
  // one workspace: X g dirn | Sh Yh | f t | Xc gc fc | ls amp noise ybuf ll graw | X Y par | counters, per-start ints,
  // idx, kinds
  const size_t n_dbl = 3 * MP + 2 * (size_t)RC * MP + 2 * (size_t)M + 2 * cap * P + cap +
                       cap * d + 2 * cap + cap * n + cap + cap * P + (size_t)n * d + (size_t)y_dim * n +
                       (size_t)y_dim * P * 2;
  CUDA_TRY(C().ms_buf.ensure(n_dbl * 8 + (size_t)M * 24 + cap * 4 + (size_t)y_dim * P * 4 + 64));
  double *base = C().ms_buf.as<double>();
  MsStateT<MS_MAP_MAXD> st{};
  st.d = P;
  st.H = RC;
  st.iters = iters;
  st.M = M;
  st.X = base;
  st.g = st.X + MP;
  st.dirn = st.g + MP;
  st.Sh = st.dirn + MP;
  st.Yh = st.Sh + (size_t)RC * MP;
  st.f = st.Yh + (size_t)RC * MP;
  st.t = st.f + M;
  st.Xc = st.t + M;
  st.gc = st.Xc + cap * P;
  st.fc = st.gc + cap * P;
  double *ls = st.fc + cap, *amp = ls + cap * d, *noise = amp + cap, *ybuf = noise + cap, *ll = ybuf + cap * n,
         *graw = ll + cap, *dX = graw + cap * P, *dY = dX + (size_t)n * d, *dpar = dY + (size_t)y_dim * n;
  st.counters = reinterpret_cast<int *>(dpar + (size_t)y_dim * P * 2);
  st.hist_len = st.counters + 4;
  st.hist_start = st.hist_len + M;
  st.trials = st.hist_start + M;
  st.steps = st.trials + M;
  st.state = st.steps + M;
  st.nev = st.state + M;
  st.idx = st.nev + M;      // [cap]
  int *dkind = st.idx + cap;
  st.fan = 1;
  for (int j = 0; j < P; ++j) {
    st.lb[j] = -30.0;
    st.ub[j] = 30.0;
  }
  st.step0 = 0.1 * 60.0;
  const unsigned nbm = (unsigned)((M + 127) / 128);

  // X, the Y rows, the prior tables and the starts go to the device once per solve (pageable sources: synchronous
  // staging, the workspace is idle here)
  CUDA_TRY(cudaMemcpyAsync(dX, X, (size_t)n * d * 8, cudaMemcpyHostToDevice, C().stream));
  CUDA_TRY(cudaMemcpyAsync(dY, Y, (size_t)y_dim * n * 8, cudaMemcpyHostToDevice, C().stream));
  CUDA_TRY(cudaMemcpyAsync(dpar, par, (size_t)y_dim * P * 2 * 8, cudaMemcpyHostToDevice, C().stream));
  CUDA_TRY(cudaMemcpyAsync(dkind, kind, (size_t)y_dim * P * 4, cudaMemcpyHostToDevice, C().stream));
  CUDA_TRY(cudaMemcpyAsync(st.Xc, starts_z, MP * 8, cudaMemcpyHostToDevice, C().stream));
  CUDA_TRY(cudaStreamSynchronize(C().stream));

  long long evaluated = 0;
  auto eval = [&](const double *Zp, const int *idxp, long long cnt, double *fp, double *gp) -> int {
    MapEvalParams ep{};
    ep.Z = Zp;
    ep.idx = idxp;
    ep.count = cnt;
    ep.pair0 = pair0;
    ep.M = Mslice;
    ep.d = d;
    ep.n = n;
    ep.kind = dkind;
    ep.par = dpar;
    ep.Y = dY;
    ep.ls = ls;
    ep.amp = amp;
    ep.noise = noise;
    ep.ybuf = ybuf;
    ep.ll = ll;
    ep.graw = graw;
    ep.f = fp;
    ep.g = gp;
    evaluated += cnt;
    map_prep_kernel<<<(unsigned)cnt, 128, 0, C().stream>>>(ep);
    ++C().launches;
    int rc = loglik_core(dX, d, n, ybuf, n, ls, amp, noise, ks, discrete_mask, cnt, ll, true, graw, nullptr, nullptr,
                         nullptr, true);
    if (rc) return rc;
    map_prior_kernel<<<(unsigned)((cnt + 127) / 128), 128, 0, C().stream>>>(ep);
    ++C().launches;
    return 0;
  };

  ms_init_kernel<<<nbm, 128, 0, C().stream>>>(st, st.Xc);
  ++C().launches;
  int rc = eval(st.X, nullptr, M, st.f, st.g);
  if (rc) return rc;
  const int max_rounds = iters > 0 ? 2 * iters + MS_MAX_TRIALS : 0;
  st.budget = max_rounds;
  int active = iters > 0 ? (int)M : 0;
  const bool trace = getenv("BOSS_MS_TRACE") != nullptr;   // one line per round on stderr: round, batch size
  CUDA_TRY(cudaMemsetAsync(st.counters, 0, 16, C().stream));
  int hc[3] = {0, 0, 0};
  int rounds = 0;
  double t_prev = 0.0;
  for (int round = 0; round < max_rounds && active > 0; ++round, ++rounds) {
    if (trace) {
      timespec ts;
      clock_gettime(CLOCK_MONOTONIC, &ts);
      const double t_now = ts.tv_sec * 1e6 + ts.tv_nsec * 1e-3;
      fprintf(stderr, "boss map multistart: round %d active %d prev_round_us %.0f\n", round, active,
              round ? t_now - t_prev : 0.0);
      t_prev = t_now;
    }
    CUDA_TRY(cudaMemsetAsync(st.counters, 0, 8, C().stream));
    ms_propose_kernel<<<nbm, 128, 0, C().stream>>>(st);
    ++C().launches;
    rc = eval(st.Xc, st.idx, active, st.fc, st.gc);
    if (rc) return rc;
    ms_advance_kernel<<<(active + 127) / 128, 128, 0, C().stream>>>(st, active);
    ++C().launches;
    CUDA_TRY(cudaMemcpyAsync(hc, st.counters, 12, cudaMemcpyDeviceToHost, C().stream));
    CUDA_TRY(cudaStreamSynchronize(C().stream));
    if (hc[0] != active) return fail(BOSS_ERR_STATE, "boss_gp_map_multistart: internal batch-length mismatch");
    active = hc[1];
  }
  // raw values of the final points, exactly as the evaluations saw them
  MapEvalParams ep{};
  ep.Z = st.X;
  ep.count = M;
  ep.pair0 = pair0;
  ep.M = Mslice;
  ep.d = d;
  ep.n = n;
  ep.kind = dkind;
  ep.par = dpar;
  ep.ls = ls;
  ep.amp = amp;
  ep.noise = noise;
  map_prep_kernel<<<(unsigned)M, 128, 0, C().stream>>>(ep);
  ++C().launches;
  CUDA_TRY(cudaGetLastError());
  std::vector<double> hls((size_t)M * d), hamp(M), hnoise(M);
  CUDA_TRY(cudaMemcpyAsync(hls.data(), ls, (size_t)M * d * 8, cudaMemcpyDeviceToHost, C().stream));
  CUDA_TRY(cudaMemcpyAsync(hamp.data(), amp, (size_t)M * 8, cudaMemcpyDeviceToHost, C().stream));
  CUDA_TRY(cudaMemcpyAsync(hnoise.data(), noise, (size_t)M * 8, cudaMemcpyDeviceToHost, C().stream));
  CUDA_TRY(cudaMemcpyAsync(f_out, st.f, (size_t)M * 8, cudaMemcpyDeviceToHost, C().stream));
  CUDA_TRY(cudaStreamSynchronize(C().stream));
  for (long long m = 0; m < M; ++m) {
    for (int j = 0; j < d; ++j) raw_out[m * P + j] = hls[m * d + j];
    raw_out[m * P + d] = hamp[m];
    raw_out[m * P + d + 1] = hnoise[m];
  }
  if (trace)
    fprintf(stderr, "boss map multistart: rounds %d evaluations %lld (pairs %lld)\n", rounds, evaluated, M);
  *evals = evaluated;
  return 0;
}

int boss_gp_map_multistart(const double *X, int d, int n, int y_dim, const double *Y_minus_mean, int kernel_id,
                           const uint8_t *discrete_mask, const int32_t *prior_kind, const double *prior_par,
                           const double *starts, int64_t M, int iters, int history, double *params_out, double *f_out,
                           double *best_params, double *best_val, int64_t *best_idx, int *evals_out) {
  if (!X || !Y_minus_mean || !prior_kind || !prior_par || !starts || d < 1 || n < 1 || M < 1 || y_dim < 1 ||
      y_dim > 16)
    return fail(BOSS_ERR_ARG, "boss_gp_map_multistart: bad arguments");
  if (d > 32) return fail(BOSS_ERR_ARG, "boss_gp_map_multistart: x_dim > 32 is not supported");
  KernelSpec ks;
  if (!decode_kernel(kernel_id, &ks)) return fail(BOSS_ERR_ARG, "boss_gp_map_multistart: unknown kernel_id");
  const int P = d + 2;
  const int64_t total = (int64_t)y_dim * M;
  for (int e = 0; e < y_dim * P; ++e)
    if (prior_kind[e] < 0 || prior_kind[e] > 3)
      return fail(BOSS_ERR_ARG, "boss_gp_map_multistart: unknown prior kind");
  // the search runs in z = log(raw) for the free entries; a pinned (Dirac) entry stays at z = 0
  std::vector<double> z((size_t)total * P);
  for (int64_t q = 0; q < total; ++q) {
    const int sl = (int)(q / M);
    for (int j = 0; j < P; ++j) {
      const double v = starts[(size_t)q * P + j];
      if (prior_kind[sl * P + j] == 0) {
        z[(size_t)q * P + j] = 0.0;
        continue;
      }
      if (!(std::isfinite(v) && v > 0.0))
        return fail(BOSS_ERR_ARG, "boss_gp_map_multistart: a free start entry is not finite and > 0");
      z[(size_t)q * P + j] = std::log(v);
    }
  }
  std::vector<double> raw((size_t)total * P), f((size_t)total);
  // multi-device: contiguous ranges of (slice, start) pairs; a pair's trajectory does not depend on the others
  const int nd = (g_ndev > 1 && tl_dev < 0 && total >= 2LL * g_ndev) ? g_ndev : 1;
  std::vector<long long> ev(nd, 0);
  int rc;
  if (nd <= 1) {
    REQUIRE_INIT();
    rc = map_multistart_single(X, d, n, y_dim, Y_minus_mean, ks, discrete_mask, prior_kind, prior_par, z.data(), 0, M,
                               total, iters, history, raw.data(), f.data(), &ev[0]);
  } else {
    const int64_t per = (total + nd - 1) / nd;
    rc = for_each_device(nd, [&](int k, Ctx *) {
      const int64_t first = std::min<int64_t>(total, (int64_t)k * per), cnt = std::min<int64_t>(per, total - first);
      if (cnt <= 0) return 0;
      return map_multistart_single(X, d, n, y_dim, Y_minus_mean, ks, discrete_mask, prior_kind, prior_par,
                                   z.data() + (size_t)first * P, first, M, cnt, iters, history,
                                   raw.data() + (size_t)first * P, f.data() + first, &ev[k]);
    });
  }
  if (rc) return rc;
  // per slice: Julia's first maximal index over the starts; -1 / -Inf when every start failed
  for (int i = 0; i < y_dim; ++i) {
    double bv = -std::numeric_limits<double>::infinity();
    int64_t bi = -1;
    for (int64_t s = 0; s < M; ++s) {
      const double v = f[(size_t)i * M + s];
      if (v > bv) {
        bv = v;
        bi = s;
      }
    }
    if (best_val) best_val[i] = bv;
    if (best_idx) best_idx[i] = bi;
    if (best_params)
      for (int j = 0; j < P; ++j)
        best_params[(size_t)i * P + j] = bi >= 0 ? raw[((size_t)i * M + bi) * P + j] : std::nan("");
  }
  if (params_out) std::memcpy(params_out, raw.data(), raw.size() * 8);
  if (f_out) std::memcpy(f_out, f.data(), f.size() * 8);
  if (evals_out) {
    long long tot = 0;
    for (long long e : ev) tot += e;
    *evals_out = (int)((tot + total - 1) / total);
  }
  return 0;
}

static int check_mean_jac(const char *who, int n, const double *grad, const double *mean_jac, int k, int64_t ldj,
                          const double *grad_mean) {
  if (!grad) return fail(BOSS_ERR_ARG, std::string(who) + ": grad is NULL");
  if (!mean_jac || !grad_mean) return fail(BOSS_ERR_ARG, std::string(who) + ": mean_jac or grad_mean is NULL");
  if (k < 1) return fail(BOSS_ERR_ARG, std::string(who) + ": k < 1");
  if (ldj != 0 && ldj < (int64_t)k * n) return fail(BOSS_ERR_ARG, std::string(who) + ": ldj is neither 0 nor >= k*n");
  return 0;
}

int boss_gp_loglik_grad_batch_mean(const double *X, int d, int n, const double *Y_minus_mean, int64_t ldy,
                                   const double *mean_jac, int k, int64_t ldj, const double *lengthscales,
                                   const double *amplitude, const double *noise_std, int kernel_id,
                                   const uint8_t *discrete_mask, int64_t S, double *loglik, double *grad,
                                   double *grad_mean) {
  if (int rc = check_mean_jac("boss_gp_loglik_grad_batch_mean", n, grad, mean_jac, k, ldj, grad_mean)) return rc;
  const MeanJac mj{mean_jac, k, ldj, grad_mean};
  return loglik_impl(X, d, n, Y_minus_mean, ldy, lengthscales, amplitude, noise_std, kernel_id, discrete_mask, S, loglik,
                     false, grad, nullptr, nullptr, &mj);
}
int boss_gp_loglik_grad_batch_mean_dev(const double *X_dev, int d, int n, const double *Y_minus_mean_dev, int64_t ldy,
                                       const double *mean_jac_dev, int k, int64_t ldj, const double *lengthscales_dev,
                                       const double *amplitude_dev, const double *noise_std_dev, int kernel_id,
                                       const uint8_t *discrete_mask, int64_t S, double *loglik_dev, double *grad_dev,
                                       double *grad_mean_dev, void *stream) {
  if (int rc = check_mean_jac("boss_gp_loglik_grad_batch_mean_dev", n, grad_dev, mean_jac_dev, k, ldj, grad_mean_dev))
    return rc;
  const MeanJac mj{mean_jac_dev, k, ldj, grad_mean_dev};
  return loglik_impl(X_dev, d, n, Y_minus_mean_dev, ldy, lengthscales_dev, amplitude_dev, noise_std_dev, kernel_id,
                     discrete_mask, S, loglik_dev, true, grad_dev, nullptr, stream, &mj);
}

// ---------------------------------------------------------------------------------------------
// debug hooks
// ---------------------------------------------------------------------------------------------
static void pack_host(const double *dense, int R, int C, int Rp, int Cp, std::vector<double> &out) {
  out.assign((size_t)Rp * Cp, 0.0);
  const int kt = Cp / TK;
  for (int r = 0; r < R; ++r)
    for (int c = 0; c < C; ++c) out[p_index(r, c, kt)] = dense[(size_t)r * C + c];
}

int boss_dbg_gemm_nt(const double *A, const double *B, int M, int N, int K, double *Cout) {
  REQUIRE_INIT();
  const int Mp = round_up(M, TM), Np = round_up(N, TM), Kp = round_up(K, TK);
  std::vector<double> pa, pb;
  pack_host(A, M, K, Mp, Kp, pa);
  pack_host(B, N, K, Np, Kp, pb);
  double *dA, *dB, *dC;
  CUDA_TRY(cudaMalloc(&dA, pa.size() * 8));
  CUDA_TRY(cudaMalloc(&dB, pb.size() * 8));
  CUDA_TRY(cudaMalloc(&dC, (size_t)Mp * Np * 8));
  // copies on the context's stream: it does not synchronise with the legacy default stream, so a plain cudaMemcpy
  // from pageable memory could still be in flight when the kernel reads its destination
  CUDA_TRY(cudaMemcpyAsync(dA, pa.data(), pa.size() * 8, cudaMemcpyHostToDevice, C().stream));
  CUDA_TRY(cudaMemcpyAsync(dB, pb.data(), pb.size() * 8, cudaMemcpyHostToDevice, C().stream));
  GemmNtParams p{dA, dB, dC, Kp / TK, Np / TK, 0};
  gemm_nt_kernel<<<dim3(Np / TM, Mp / TM), GEMM_THREADS, GEMM_SMEM_BYTES, C().stream>>>(p);
  ++C().launches;
  CUDA_TRY(cudaGetLastError());
  std::vector<double> pc((size_t)Mp * Np);
  CUDA_TRY(cudaMemcpyAsync(pc.data(), dC, pc.size() * 8, cudaMemcpyDeviceToHost, C().stream));
  CUDA_TRY(cudaStreamSynchronize(C().stream));
  for (int r = 0; r < M; ++r)
    for (int c = 0; c < N; ++c) Cout[(size_t)r * N + c] = pc[p_index(r, c, Np / TK)];
  cudaFree(dA);
  cudaFree(dB);
  cudaFree(dC);
  return 0;
}

__global__ void dbg_kernel_fn_kernel(int which, const double *t, double *out, int n) {
  __shared__ double tab[EXPTAB_N];
  exptab_init(tab);
  __syncthreads();
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const double x = t[i];
    double v;
    switch (which) {
      case 0: v = fast_exp_neg(x, tab); break;
      case 1: v = fast_sqrt(x); break;
      case 2: v = kappa_fast<0>(x, tab, 0.0); break;
      case 3: v = kappa_fast<1>(x, tab, 0.0); break;
      case 4: v = kappa_fast<2>(x, tab, 0.0); break;
      case 5: v = kappa_dr_over_r_fast<0>(x, tab, 0.0); break;
      case 6: v = kappa_dr_over_r_fast<1>(x, tab, 0.0); break;
      default: v = kappa_dr_over_r_fast<2>(x, tab, 0.0); break;
    }
    out[i] = v;
  }
}
int boss_dbg_kernel_fn(int which, const double *t, int n, double *out) {
  REQUIRE_INIT();
  if (which < 0 || which > 7 || n < 0) return fail(BOSS_ERR_ARG, "boss_dbg_kernel_fn: bad argument");
  double *dt, *dout;
  CUDA_TRY(cudaMalloc(&dt, (size_t)n * 8 + 8));
  CUDA_TRY(cudaMalloc(&dout, (size_t)n * 8 + 8));
  CUDA_TRY(cudaMemcpyAsync(dt, t, (size_t)n * 8, cudaMemcpyHostToDevice, C().stream));   // stream-ordered, as above
  dbg_kernel_fn_kernel<<<148, 256, 0, C().stream>>>(which, dt, dout, n);
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaMemcpyAsync(out, dout, (size_t)n * 8, cudaMemcpyDeviceToHost, C().stream));
  CUDA_TRY(cudaStreamSynchronize(C().stream));
  cudaFree(dt);
  cudaFree(dout);
  return 0;
}

int boss_dbg_kernel_fn_id(int kernel_id, int which, const double *d2, int n, double *out) {
  REQUIRE_INIT();
  KernelSpec ks;
  if (!decode_kernel(kernel_id, &ks)) return fail(BOSS_ERR_ARG, "boss_dbg_kernel_fn_id: unknown kernel_id");
  if (which < 0 || which > 3 || n < 0 || (n > 0 && (!d2 || !out)))
    return fail(BOSS_ERR_ARG, "boss_dbg_kernel_fn_id: bad argument");
  if (n == 0) return 0;
  double *dt, *dout;
  CUDA_TRY(cudaMalloc(&dt, (size_t)n * 8));
  CUDA_TRY(cudaMalloc(&dout, (size_t)n * 8));
  CUDA_TRY(cudaMemcpyAsync(dt, d2, (size_t)n * 8, cudaMemcpyHostToDevice, C().stream));
  switch (ks.kid) {
    case 0: dbg_kernel_fn_id_kernel<0><<<148, 256, 0, C().stream>>>(which, ks.rq_a, dt, dout, n); break;
    case 1: dbg_kernel_fn_id_kernel<1><<<148, 256, 0, C().stream>>>(which, ks.rq_a, dt, dout, n); break;
    case 2: dbg_kernel_fn_id_kernel<2><<<148, 256, 0, C().stream>>>(which, ks.rq_a, dt, dout, n); break;
    case 3: dbg_kernel_fn_id_kernel<3><<<148, 256, 0, C().stream>>>(which, ks.rq_a, dt, dout, n); break;
    default: dbg_kernel_fn_id_kernel<4><<<148, 256, 0, C().stream>>>(which, ks.rq_a, dt, dout, n); break;
  }
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaMemcpyAsync(out, dout, (size_t)n * 8, cudaMemcpyDeviceToHost, C().stream));
  CUDA_TRY(cudaStreamSynchronize(C().stream));
  cudaFree(dt);
  cudaFree(dout);
  return 0;
}

__global__ void rz_scan_kernel(const unsigned char *p, size_t nbytes, unsigned long long *bad) {
  unsigned long long c = 0;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < nbytes; i += (size_t)gridDim.x * blockDim.x)
    c += p[i] != 0xA5;
  if (c) atomicAdd(bad, c);
}
// Scans the guard bands of every live device allocation of the calling thread's device (BOSS_DEBUG_REDZONE=1).
// Returns the number of overwritten guard bytes (0 = clean), -1 when red zones are off; *n_allocs = allocations scanned.
int64_t boss_dbg_check_redzones(int64_t *n_allocs) {
  if (n_allocs) *n_allocs = 0;
  if (!redzones_on()) return -1;
  REQUIRE_INIT();
  CUDA_TRY(cudaDeviceSynchronize());
  unsigned long long *bad = nullptr;
  CUDA_TRY(cudaMalloc(&bad, 8));
  CUDA_TRY(cudaMemset(bad, 0, 8));
  int64_t cnt = 0;
  {
    std::lock_guard<std::mutex> lk(g_rz_mu);
    for (auto &kv : g_rz) {
      const RzEntry &e = kv.second;
      if (e.device != C().device) continue;
      const size_t user = (e.bytes + 255) & ~(size_t)255;
      rz_scan_kernel<<<64, 256>>>(reinterpret_cast<const unsigned char *>(e.base), RZ_BYTES, bad);
      rz_scan_kernel<<<64, 256>>>(reinterpret_cast<const unsigned char *>(e.base) + RZ_BYTES + e.bytes, user - e.bytes + RZ_BYTES, bad);
      ++cnt;
    }
  }
  unsigned long long h = 0;
  CUDA_TRY(cudaMemcpy(&h, bad, 8, cudaMemcpyDeviceToHost));
  cudaFree(bad);
  if (n_allocs) *n_allocs = cnt;
  return (int64_t)h;
}

// Negative control of the red-zone check: one byte written just past a fresh 1000-byte allocation and one just before
// it must be reported (returns the number of guard bytes found overwritten: 2), and nothing after the buffer is freed.
int64_t boss_dbg_redzone_selftest(void) {
  if (!redzones_on()) return -1;
  void *p = nullptr;
  if (dev_malloc(&p, 1000) != cudaSuccess) return -2;
  const int64_t before = boss_dbg_check_redzones(nullptr);
  cudaMemset(static_cast<char *>(p) + 1000, 0, 1);
  cudaMemset(static_cast<char *>(p) - 1, 0, 1);
  const int64_t after = boss_dbg_check_redzones(nullptr);
  dev_free(p);
  return after - before;
}

int boss_dbg_factors(const boss_gp *gp, double *L, double *W, double *alpha) {
  if (!gp) return fail(BOSS_ERR_ARG, "boss_dbg_factors: NULL handle");
  if (tl_dev >= 0 && replica_on(gp, tl_dev)) gp = replica_on(gp, tl_dev);   // inspect a specific replica
  REQUIRE_HANDLE_CTX(gp);
  const size_t mat = (size_t)gp->n_pad * gp->n_pad;
  std::vector<double> buf(mat);
  const int n = gp->n;
  if (L) {
    CUDA_TRY(cudaMemcpy(buf.data(), gp->L, mat * 8, cudaMemcpyDeviceToHost));
    for (int r = 0; r < n; ++r)
      for (int c = 0; c < n; ++c) L[(size_t)r * n + c] = (c <= r) ? buf[p_index(r, c, gp->ktiles)] : 0.0;
  }
  if (W) {
    CUDA_TRY(cudaMemcpy(buf.data(), gp->W, mat * 8, cudaMemcpyDeviceToHost));
    for (int r = 0; r < n; ++r)
      for (int c = 0; c < n; ++c) W[(size_t)r * n + c] = buf[p_index(r, c, gp->ktiles)];
  }
  if (alpha) CUDA_TRY(cudaMemcpy(alpha, gp->alpha, (size_t)n * 8, cudaMemcpyDeviceToHost));
  return 0;
}

// Argmax screening of the last scoring call on the current device (DESIGN.md 2.9): out[0] = 0 not screened, 1 screened,
// 2 fell back to the full path after the first chunk; out[1] = candidates bounded; out[2] = candidates that survived.
int boss_dbg_screen_stats(int64_t *out) {
  REQUIRE_INIT();
  for (int i = 0; i < 3; ++i) out[i] = C().scr_stats[i];
  return 0;
}

// The paths score_slice took in the last scoring call on the current device, counted per (chunk, slice) pass: out[0] wide
// with the fused epilogue, out[1] wide without it (row splits, a slice other than the last, or BOSS_UNFUSED_SCORE),
// out[2] narrow, out[3] quarter; out[4] the passes that ran the x-gradient pipeline.  Nested calls of a screened or
// multi-start call add to their caller's counts.  The counts are reset once the call has bound its slices and set up its
// workspaces: a call that fails before that, or has M <= 0, leaves the previous call's counts (as scr_stats does).
int boss_dbg_score_paths(int64_t *out) {
  REQUIRE_INIT();
  for (int i = 0; i < 5; ++i) out[i] = C().score_paths[i];
  return 0;
}

// The FP32 mean tier of the last screened call (DESIGN.md 2.9): out[0] = candidates in the ambiguous band (refined in
// FP64), out[1] = the pool as the chunks left it (definite keeps and ambiguous candidates), before refinement and re-seed.
int boss_dbg_screen_ambiguous(int64_t *out) {
  REQUIRE_INIT();
  out[0] = C().scr_amb[0];
  out[1] = C().scr_amb[1];
  return 0;
}
int boss_dbg_screen_var(int64_t *out) {
  REQUIRE_INIT();
  out[0] = C().scr_var[0];
  out[1] = C().scr_var[1];
  return 0;
}

// For M candidates (column-major d x M host array): the FP32 tier's mean mu~ and bound E, and the FP64 tier's mean
// (K*^T alpha, without a prior mean), computed by the kernels the screen runs.
int boss_dbg_screen_mean(const boss_gp *gp, const double *Xs, int64_t M, double *mu32, double *E, double *mu64) {
  if (!gp || M < 1 || M > (1 << 22) || !Xs) return fail(BOSS_ERR_ARG, "boss_dbg_screen_mean: bad argument");
  if (!kid_has_f32_tier(gp->kernel_id))
    return fail(BOSS_ERR_ARG, "boss_dbg_screen_mean: the FP32 mean tier does not exist for this kernel");
  REQUIRE_HANDLE_CTX(gp);
  const int d = gp->d, ld = (int)((M + 127) / 128 * 128), ncb = ld / 128;
  const int nks = std::max(1, std::min(gp->nblk, (16 * 148 + ncb - 1) / ncb));
  double *dx = nullptr, *dpart = nullptr, *dout = nullptr, *dA = nullptr;
  float *dxt = nullptr, *dal = nullptr;
  CUDA_TRY(cudaMalloc(&dx, (size_t)M * d * 8));
  CUDA_TRY(cudaMalloc(&dpart, (size_t)2 * gp->nblk * ld * 8));
  CUDA_TRY(cudaMalloc(&dout, (size_t)3 * ld * 8));
  CUDA_TRY(cudaMalloc(&dA, SCREEN_NCONST * 8));
  CUDA_TRY(cudaMalloc(&dxt, (size_t)gp->n_pad * ((gp->dp + 7) / 8 * 8) * 8));
  CUDA_TRY(cudaMalloc(&dal, (size_t)gp->n_pad * 8));
  CUDA_TRY(cudaMemcpyAsync(dx, Xs, (size_t)M * d * 8, cudaMemcpyHostToDevice, C().stream));
  screen_consts_kernel<<<1, 1024, 0, C().stream>>>(gp->Xt, gp->alpha, gp->n, gp->n_pad, gp->dp, dxt, dal, dA);
  ScreenF32Params sp{};
  sp.Xs = dx;
  sp.M = M;
  sp.d = d;
  sp.nsl = 1;
  sp.sl[0] = ScreenSlice{reinterpret_cast<const float4 *>(dxt), reinterpret_cast<const float4 *>(dal), dA, gp->invl,
                         gp->disc, gp->a2, gp->n_pad};
  sp.mu_out = dout;
  sp.e_out = dout + ld;
  sp.ld = ld;
  launch_screen_mean_bound(gp->kernel_id, gp->dp, sp, ncb, C().stream);
  XcovParams xp = xcov_params(gp, dx, M, 0, 0, d, ld);
  xp.mu_part = dpart;
  launch_xcov_mean(gp->kernel_id, gp->dp, xp, dim3(ncb, nks), C().stream);
  reduce_rows_kernel<<<(ld + 255) / 256, 256, 0, C().stream>>>(dpart, 2 * gp->nblk, (size_t)ld, dout + 2 * ld, ld);
  CUDA_TRY(cudaGetLastError());
  std::vector<double> h((size_t)3 * ld);
  CUDA_TRY(cudaMemcpyAsync(h.data(), dout, h.size() * 8, cudaMemcpyDeviceToHost, C().stream));
  CUDA_TRY(cudaStreamSynchronize(C().stream));
  for (int64_t i = 0; i < M; ++i) {
    if (mu32) mu32[i] = h[i];
    if (E) E[i] = h[ld + i];
    if (mu64) mu64[i] = h[2 * (size_t)ld + i];
  }
  cudaFree(dx);
  cudaFree(dpart);
  cudaFree(dout);
  cudaFree(dA);
  cudaFree(dxt);
  cudaFree(dal);
  return 0;
}

// kappa_f32<kid>((float)(r^2)) of the FP32 mean tier for n distances r (kid 0 SE, 1 Matern32, 2 Matern52)
int boss_dbg_kappa_f32(int kid, const double *r, int n, double *out) {
  REQUIRE_INIT();
  if (kid < 0 || kid > 2 || n < 0) return fail(BOSS_ERR_ARG, "boss_dbg_kappa_f32: bad argument");
  double *dr, *dout;
  CUDA_TRY(cudaMalloc(&dr, (size_t)n * 8 + 8));
  CUDA_TRY(cudaMalloc(&dout, (size_t)n * 8 + 8));
  // on the library stream: a pageable cudaMemcpy may return before its DMA lands, and that stream does not wait for it
  CUDA_TRY(cudaMemcpyAsync(dr, r, (size_t)n * 8, cudaMemcpyHostToDevice, C().stream));
  launch_kappa_f32_sweep(kid, dr, n, dout, C().stream);
  CUDA_TRY(cudaMemcpyAsync(out, dout, (size_t)n * 8, cudaMemcpyDeviceToHost, C().stream));
  CUDA_TRY(cudaStreamSynchronize(C().stream));
  cudaFree(dr);
  cudaFree(dout);
  return 0;
}

int boss_dbg_mma_d2(int dp, const float *u, const float *t, const float *nu, const float *nt, int mt, int nt_tiles,
                    float *d2) {
  REQUIRE_INIT();
  if (dp < 1 || dp > 32 || mt < 1 || nt_tiles < 1 || mt > 4096 || nt_tiles > 4096 || !u || !t || !nu || !nt || !d2)
    return fail(BOSS_ERR_ARG, "boss_dbg_mma_d2: bad argument");
  const int dpp = dp <= 8 ? 8 : dp <= 16 ? 16 : 32;   // the kernels' k-steps: padded dimensions 2-8, 12-16, 32
  const size_t m = (size_t)16 * mt, n = (size_t)8 * nt_tiles;
  float *du, *dt, *dnu, *dnt, *dd;
  CUDA_TRY(cudaMalloc(&du, m * dpp * 4));
  CUDA_TRY(cudaMalloc(&dt, n * dpp * 4));
  CUDA_TRY(cudaMalloc(&dnu, m * 4));
  CUDA_TRY(cudaMalloc(&dnt, n * 4));
  CUDA_TRY(cudaMalloc(&dd, m * n * 4));
  CUDA_TRY(cudaMemcpyAsync(du, u, m * dpp * 4, cudaMemcpyHostToDevice, C().stream));
  CUDA_TRY(cudaMemcpyAsync(dt, t, n * dpp * 4, cudaMemcpyHostToDevice, C().stream));
  CUDA_TRY(cudaMemcpyAsync(dnu, nu, m * 4, cudaMemcpyHostToDevice, C().stream));
  CUDA_TRY(cudaMemcpyAsync(dnt, nt, n * 4, cudaMemcpyHostToDevice, C().stream));
  launch_mma_d2(dpp, du, dt, dnu, dnt, mt, nt_tiles, dd, C().stream);
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaMemcpyAsync(d2, dd, m * n * 4, cudaMemcpyDeviceToHost, C().stream));
  CUDA_TRY(cudaStreamSynchronize(C().stream));
  cudaFree(du);
  cudaFree(dt);
  cudaFree(dnu);
  cudaFree(dnt);
  cudaFree(dd);
  return 0;
}

}  // extern "C"

"""ctypes binding of libboss_b200.so (include/boss_b200.h).  No CPU fallback: importing this module
without the built CUDA library raises, and every call raises BossError on a CUDA / argument error."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libboss_b200.so")

if not os.path.exists(LIB_PATH):
    raise ImportError(
        f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
        "(nvcc -gencode arch=compute_100a,code=sm_100a).  boss_b200 has no CPU fallback.")

lib = C.CDLL(LIB_PATH)

BOSS_OK, BOSS_NOT_POSDEF, BOSS_NEG_VARIANCE = 0, 1, 2
KERNEL_SE, KERNEL_MATERN32, KERNEL_MATERN52, KERNEL_MATERN12 = 0, 1, 2, 3
RQ_SLOTS = 512   # BOSS_RQ_SLOTS: distinct RationalQuadratic shape parameters a process can register

_dp = C.POINTER(C.c_double)
_u8p = C.POINTER(C.c_uint8)
_i32p = C.POINTER(C.c_int32)
_i64p = C.POINTER(C.c_int64)
_vp = C.c_void_p

EXPORTS = {
    "boss_init": (C.c_int, [C.c_int]),
    "boss_init_multi": (C.c_int, [C.c_int]),
    "boss_set_device": (C.c_int, [C.c_int]),
    "boss_n_devices": (C.c_int, []),
    "boss_shutdown": (None, []),
    "boss_last_error": (C.c_char_p, []),
    "boss_version": (C.c_int, []),
    "boss_device": (C.c_int, []),
    "boss_stream": (_vp, []),
    "boss_gp_fit": (C.c_int, [_vp, C.c_int, C.c_int, _vp, _vp, C.c_double, C.c_double, C.c_int, _vp,
                              C.POINTER(_vp), _dp]),
    "boss_gp_fit_batch": (C.c_int, [_vp, C.c_int, C.c_int, _vp, C.c_int64, _vp, _vp, _vp, C.c_int, _vp, C.c_int64,
                                    C.POINTER(_vp), _vp]),
    "boss_gp_append": (C.c_int, [_vp, _vp, C.c_double, _dp]),
    "boss_gp_free": (None, [_vp]),
    "boss_gp_n": (C.c_int, [_vp]),
    "boss_gp_d": (C.c_int, [_vp]),
    "boss_gp_predict": (C.c_int, [_vp, _vp, C.c_int64, _vp, _vp, _vp, _vp]),
    "boss_gp_predict_dev": (C.c_int, [_vp, _vp, C.c_int64, _vp, _vp, _vp, _vp, _vp]),
    "boss_gp_predict_grad": (C.c_int, [_vp, C.c_int, C.c_int, _vp, C.c_int64, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "boss_gp_cov": (C.c_int, [_vp, _vp, C.c_int64, _vp, _vp, _vp]),
    "boss_ei_score": (C.c_int, [_vp, C.c_int, C.c_int, _vp, C.c_int64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                _dp, _i64p]),
    "boss_ei_score_dev": (C.c_int, [_vp, C.c_int, C.c_int, _vp, C.c_int64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                    _vp, _dp, _i64p, _vp]),
    "boss_ei_score_topk": (C.c_int, [_vp, C.c_int, C.c_int, _vp, C.c_int64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, C.c_int64,
                                     _vp, _vp]),
    "boss_ei_score_topk_dev": (C.c_int, [_vp, C.c_int, C.c_int, _vp, C.c_int64, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                         C.c_int64, _vp, _vp, _vp]),
    "boss_ei_score_grid": (C.c_int, [_vp, C.c_int, C.c_int, C.c_int, _vp, _vp, _vp, C.c_int64, C.c_int64, _vp, _vp, _vp, _vp,
                                     _vp, _vp, _vp, _vp, _dp, _i64p, _vp]),
    "boss_ei_score_uniform": (C.c_int, [_vp, C.c_int, C.c_int, C.c_int, C.c_uint64, C.c_int64, C.c_int64, _vp, _vp, _vp,
                                        _vp, _vp, _vp, _vp, _vp, _dp, _i64p, _vp]),
    "boss_ei_maximize_multistart": (C.c_int, [_vp, C.c_int, C.c_int, _vp, C.c_int64, C.c_int, C.c_int, _vp, _vp, _vp, _vp, _vp,
                                              _vp, _vp, _vp, _vp, _vp, _dp, _i64p, C.POINTER(C.c_int)]),
    "boss_ei_value_grad": (C.c_int, [_vp, C.c_int, C.c_int, _vp, C.c_int64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                     _vp]),
    "boss_ei_value_grad_dev": (C.c_int, [_vp, C.c_int, C.c_int, _vp, C.c_int64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                         _vp, _vp, _vp]),
    "boss_mcei_score": (C.c_int, [_vp, C.c_int, C.c_int, _vp, C.c_int64, _vp, C.c_int, C.c_double, _vp, _vp, _vp, _vp,
                                  C.c_int, _vp, _vp, _vp, _vp, _vp, _vp, _dp, _i64p]),
    "boss_mcei_value_grad": (C.c_int, [_vp, C.c_int, C.c_int, _vp, C.c_int64, _vp, _vp, C.c_int, C.c_double, _vp, _vp,
                                       _vp, _vp, C.c_int, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "boss_mcei_maximize_multistart": (C.c_int, [_vp, C.c_int, C.c_int, _vp, C.c_int64, C.c_int, C.c_int, _vp, C.c_int,
                                                C.c_double, _vp, _vp, _vp, _vp, C.c_int, _vp, _vp, _vp, _vp, _vp, _vp,
                                                _vp, _vp, _dp, _i64p, C.POINTER(C.c_int)]),
    "boss_mcei_score_topk": (C.c_int, [_vp, C.c_int, C.c_int, _vp, C.c_int64, _vp, C.c_int, C.c_double, _vp, _vp, _vp,
                                       _vp, C.c_int, _vp, _vp, _vp, _vp, _vp, C.c_int64, _vp, _vp]),
    "boss_gp_loglik_batch": (C.c_int, [_vp, C.c_int, C.c_int, _vp, C.c_int64, _vp, _vp, _vp, C.c_int, _vp, C.c_int64,
                                       _vp]),
    "boss_gp_loglik_batch_dev": (C.c_int, [_vp, C.c_int, C.c_int, _vp, C.c_int64, _vp, _vp, _vp, C.c_int, _vp,
                                           C.c_int64, _vp, _vp]),
    "boss_gp_loglik_grad_batch": (C.c_int, [_vp, C.c_int, C.c_int, _vp, C.c_int64, _vp, _vp, _vp, C.c_int, _vp, C.c_int64,
                                            _vp, _vp]),
    "boss_gp_loglik_grad_batch_dev": (C.c_int, [_vp, C.c_int, C.c_int, _vp, C.c_int64, _vp, _vp, _vp, C.c_int, _vp,
                                                C.c_int64, _vp, _vp, _vp]),
    "boss_gp_loglik_grad_batch_mean": (C.c_int, [_vp, C.c_int, C.c_int, _vp, C.c_int64, _vp, C.c_int, C.c_int64, _vp, _vp,
                                                 _vp, C.c_int, _vp, C.c_int64, _vp, _vp, _vp]),
    "boss_gp_loglik_grad_batch_mean_dev": (C.c_int, [_vp, C.c_int, C.c_int, _vp, C.c_int64, _vp, C.c_int, C.c_int64, _vp,
                                                     _vp, _vp, C.c_int, _vp, C.c_int64, _vp, _vp, _vp, _vp]),
    "boss_gp_map_multistart": (C.c_int, [_vp, C.c_int, C.c_int, C.c_int, _vp, C.c_int, _vp, _vp, _vp, _vp, C.c_int64,
                                         C.c_int, C.c_int, _vp, _vp, _vp, _vp, _vp, C.POINTER(C.c_int)]),
    "boss_set_timing": (None, [C.c_int]),
    "boss_last_kernel_ms": (C.c_double, [C.c_int]),
    "boss_last_kernel_count": (C.c_int, [C.c_int]),
    "boss_launch_count": (C.c_int64, []),
    "boss_dbg_gemm_nt": (C.c_int, [_vp, _vp, C.c_int, C.c_int, C.c_int, _vp]),
    "boss_dbg_factors": (C.c_int, [_vp, _vp, _vp, _vp]),
    "boss_dbg_kernel_fn": (C.c_int, [C.c_int, _vp, C.c_int, _vp]),
    "boss_kernel_rational_quadratic": (C.c_int, [C.c_double, C.POINTER(C.c_int)]),
    "boss_dbg_kernel_fn_id": (C.c_int, [C.c_int, C.c_int, _vp, C.c_int, _vp]),
    "boss_dbg_check_redzones": (C.c_int64, [_i64p]),
    "boss_dbg_redzone_selftest": (C.c_int64, []),
    "boss_dbg_screen_stats": (C.c_int, [_i64p]),
    "boss_dbg_score_paths": (C.c_int, [_i64p]),
    "boss_dbg_screen_ambiguous": (C.c_int, [_i64p]),
    "boss_dbg_screen_var": (C.c_int, [_i64p]),
    "boss_dbg_screen_mean": (C.c_int, [_vp, _vp, C.c_int64, _vp, _vp, _vp]),
    "boss_dbg_kappa_f32": (C.c_int, [C.c_int, _vp, C.c_int, _vp]),
    "boss_dbg_mma_d2": (C.c_int, [C.c_int, _vp, _vp, _vp, _vp, C.c_int, C.c_int, _vp]),
}
for _name, (_res, _args) in EXPORTS.items():
    _f = getattr(lib, _name)          # AttributeError here = header and library disagree
    _f.restype = _res
    _f.argtypes = _args


class BossError(RuntimeError):
    pass


def last_error() -> str:
    return lib.boss_last_error().decode()


def _check(rc: int, what: str) -> int:
    if rc < 0:
        raise BossError(f"{what} failed ({rc}): {last_error()}")
    return rc


_rq_ids: dict[float, int] = {}


def kernel_rational_quadratic(rq_a: float) -> int:
    """The kernel_id of RationalQuadraticKernel(alpha = rq_a): (1 + r^2 / (2 rq_a))^-rq_a.  Ids come from a
    process-lifetime table in the library (no device needed) and are cached here per value."""
    a = float(rq_a)
    kid = _rq_ids.get(a)
    if kid is None:
        out = C.c_int(-1)
        _check(lib.boss_kernel_rational_quadratic(a, C.byref(out)), "boss_kernel_rational_quadratic")
        kid = _rq_ids[a] = int(out.value)
    return kid


def init(device: int = 0) -> None:
    _check(lib.boss_init(int(device)), "boss_init")


def init_multi(n_gpus: int) -> None:
    """One process drives GPUs 0..n_gpus-1: fits are replicated, host-pointer scoring / log-likelihood / multi-start
    calls are sharded inside the library (include/boss_b200.h, Devices)."""
    _check(lib.boss_init_multi(int(n_gpus)), "boss_init_multi")


def set_device(device: int) -> None:
    """Pin the calling thread to one initialised device (-1 = unpin)."""
    _check(lib.boss_set_device(int(device)), "boss_set_device")


def n_devices() -> int:
    return int(lib.boss_n_devices())


def stream_ptr() -> int:
    return int(lib.boss_stream() or 0)


def shutdown() -> None:
    lib.boss_shutdown()


def _f64(a, shape=None):
    a = np.ascontiguousarray(a, dtype=np.float64)
    if shape is not None:
        assert a.shape == shape, (a.shape, shape)
    return a


def _ptr(a):
    return None if a is None else a.ctypes.data_as(_vp)


def _cols(X):
    """d x M matrix (BOSS.jl orientation) -> M x d C-contiguous = column-major d x M in memory."""
    X = np.asarray(X, dtype=np.float64)
    if X.ndim == 1:
        X = X[:, None]
    return np.ascontiguousarray(X.T)


class GP:
    """Owner of one `boss_gp*` (one output slice, one hyper-parameter vector)."""

    def __init__(self, handle, n, d, loglik):
        self._h = handle
        self.n, self.d, self.loglik = n, d, loglik

    @property
    def handle(self):
        if not self._h:
            raise BossError("GP handle already freed")
        return self._h

    def free(self):
        if self._h:
            lib.boss_gp_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def gp_fit(X, y_minus_mean, lengthscales, amplitude, noise_std, kernel_id=KERNEL_MATERN52, discrete_mask=None):
    """-> GP, or None when K is not positive definite (BOSS_NOT_POSDEF)."""
    Xc = _cols(X)
    n, d = Xc.shape
    y = _f64(y_minus_mean, (n,))
    ls = _f64(lengthscales, (d,))
    dm = None if discrete_mask is None else np.ascontiguousarray(discrete_mask, dtype=np.uint8)
    out = _vp()
    ll = C.c_double()
    rc = _check(lib.boss_gp_fit(_ptr(Xc), d, n, _ptr(y), _ptr(ls), float(amplitude), float(noise_std), int(kernel_id),
                                _ptr(dm), C.byref(out), C.byref(ll)), "boss_gp_fit")
    if rc == BOSS_NOT_POSDEF:
        return None
    return GP(out, n, d, ll.value)


def gp_fit_batch(X, Y_minus_mean, lengthscales, amplitude, noise_std, kernel_id=KERNEL_MATERN52, discrete_mask=None):
    """S fits in one call.  lengthscales (S, d), amplitude (S,), noise_std (S,), Y_minus_mean (n,) or (S, n).
    -> list of GP (None where not positive definite)."""
    Xc = _cols(X)
    n, d = Xc.shape
    ls = _f64(lengthscales)
    S = ls.shape[0]
    assert ls.shape == (S, d)
    amp = _f64(amplitude, (S,))
    ns = _f64(noise_std, (S,))
    Y = _f64(Y_minus_mean)
    ldy = 0 if Y.ndim == 1 else n
    assert Y.shape == ((n,) if ldy == 0 else (S, n))
    dm = None if discrete_mask is None else np.ascontiguousarray(discrete_mask, dtype=np.uint8)
    out = (_vp * S)()
    ll = np.empty(S)
    _check(lib.boss_gp_fit_batch(_ptr(Xc), d, n, _ptr(Y), ldy, _ptr(ls), _ptr(amp), _ptr(ns), int(kernel_id), _ptr(dm), S,
                                 out, _ptr(ll)), "boss_gp_fit_batch")
    return [GP(_vp(out[s]), n, d, float(ll[s])) if out[s] else None for s in range(S)]


def gp_append(gp: GP, x_new, y_minus_mean_new) -> bool:
    """Rank-1 extension of the factor cache by one data point (same hyper-parameters).  False = not PD (unchanged)."""
    x = _f64(np.asarray(x_new, dtype=np.float64).reshape(-1), (gp.d,))
    ll = C.c_double()
    rc = _check(lib.boss_gp_append(gp.handle, _ptr(x), float(y_minus_mean_new), C.byref(ll)), "boss_gp_append")
    if rc == BOSS_NOT_POSDEF:
        return False
    gp.n += 1
    gp.loglik = ll.value
    return True


def gp_predict(gp: GP, Xs, prior_mean_s=None):
    """-> mu (M,), var (M,), status (M,) int32."""
    Xc = _cols(Xs)
    M = Xc.shape[0]
    pm = None if prior_mean_s is None else _f64(prior_mean_s, (M,))
    mu = np.empty(M)
    var = np.empty(M)
    st = np.empty(M, dtype=np.int32)
    _check(lib.boss_gp_predict(gp.handle, _ptr(Xc), M, _ptr(pm), _ptr(mu), _ptr(var), _ptr(st)), "boss_gp_predict")
    return mu, var, st


def gp_predict_grad(slices, y_dim, n_samples, Xs, prior_mean_s=None, prior_mean_grad_s=None):
    """Posterior means, variances and their x-gradients of all P = n_samples * y_dim posteriors in one call
    (include/boss_b200.h, boss_gp_predict_grad).  slices: flat list, sample-major (slices[s*y_dim+i]);
    prior_mean_s (y_dim, M) and prior_mean_grad_s (y_dim, d, M) are shared by the samples.
    -> mu (P, M), var (P, M), dmu (P, d, M), dvar (P, d, M), status (P, M) int32; mu, var and status equal
    gp_predict's per slice bit for bit."""
    Xc = _cols(Xs)
    M, d = Xc.shape
    assert len(slices) == y_dim * n_samples
    P = y_dim * n_samples
    arr = _slice_array(slices)
    pm = None if prior_mean_s is None else np.ascontiguousarray(np.asarray(prior_mean_s, dtype=np.float64).T)
    pmg = None if prior_mean_grad_s is None else np.ascontiguousarray(
        np.transpose(np.asarray(prior_mean_grad_s, dtype=np.float64), (2, 1, 0)))   # (M, d, y_dim)
    mu = np.empty((M, P)); var = np.empty((M, P))
    dmu = np.empty((M, d, P)); dvar = np.empty((M, d, P))
    st = np.empty((M, P), dtype=np.int32)
    _check(lib.boss_gp_predict_grad(arr, y_dim, n_samples, _ptr(Xc), M, _ptr(pm), _ptr(pmg), _ptr(mu), _ptr(var),
                                    _ptr(dmu), _ptr(dvar), _ptr(st)), "boss_gp_predict_grad")
    return mu.T, var.T, np.transpose(dmu, (2, 1, 0)), np.transpose(dvar, (2, 1, 0)), st.T


def gp_cov(gp: GP, Xs, prior_mean_s=None):
    """mean_and_cov(::GaussianProcessPosterior, X): -> mu (M,), cov (M, M) with the diagonal clipped, rc."""
    Xc = _cols(Xs)
    M = Xc.shape[0]
    pm = None if prior_mean_s is None else _f64(prior_mean_s, (M,))
    mu = np.empty(M)
    cov = np.empty((M, M))
    rc = _check(lib.boss_gp_cov(gp.handle, _ptr(Xc), M, _ptr(pm), _ptr(mu), _ptr(cov)), "boss_gp_cov")
    return mu, cov, rc


def _slice_array(slices):
    flat = [g.handle for g in slices]
    arr = (_vp * len(flat))(*flat)
    return arr


def ei_score(slices, y_dim, n_samples, Xs, coefs, best, y_max, lb=None, ub=None, cons_mask=None, prior_mean_s=None,
             want_acq=True):
    """slices: flat list, sample-major (slices[s*y_dim+i]).  -> acq (M,) or None, best_val, best_idx."""
    Xc = _cols(Xs)
    M, d = Xc.shape
    assert len(slices) == y_dim * n_samples
    arr = _slice_array(slices)
    co = _f64(coefs, (y_dim,))
    b = None if best is None else np.array([best], dtype=np.float64)
    ym = None if y_max is None else _f64(y_max, (y_dim,))
    lbv = None if lb is None else _f64(lb, (d,))
    ubv = None if ub is None else _f64(ub, (d,))
    cm = None if cons_mask is None else np.ascontiguousarray(cons_mask, dtype=np.uint8)
    pm = None if prior_mean_s is None else np.ascontiguousarray(np.asarray(prior_mean_s, dtype=np.float64).T)
    acq = np.empty(M) if want_acq else None
    bv = C.c_double()
    bi = C.c_int64()
    _check(lib.boss_ei_score(arr, y_dim, n_samples, _ptr(Xc), M, _ptr(pm), _ptr(co), _ptr(b), _ptr(ym), _ptr(lbv),
                             _ptr(ubv), _ptr(cm), _ptr(acq), None, C.byref(bv), C.byref(bi)), "boss_ei_score")
    return acq, bv.value, bi.value


def ei_score_topk(slices, y_dim, n_samples, Xs, coefs, best, y_max, k, lb=None, ub=None, cons_mask=None,
                  prior_mean_s=None):
    """The k best candidates of ei_score's scores, selected on the device (include/boss_b200.h, boss_ei_score_topk).
    -> top_val (k,), top_idx (k,) int64: descending under Julia's isless (NaN first), ties to the lower index."""
    Xc = _cols(Xs)
    M, d = Xc.shape
    assert len(slices) == y_dim * n_samples
    arr = _slice_array(slices)
    co = _f64(coefs, (y_dim,))
    b = None if best is None else np.array([best], dtype=np.float64)
    ym = None if y_max is None else _f64(y_max, (y_dim,))
    lbv = None if lb is None else _f64(lb, (d,))
    ubv = None if ub is None else _f64(ub, (d,))
    cm = None if cons_mask is None else np.ascontiguousarray(cons_mask, dtype=np.uint8)
    pm = None if prior_mean_s is None else np.ascontiguousarray(np.asarray(prior_mean_s, dtype=np.float64).T)
    k = int(k)
    tv = np.empty(max(k, 0))
    ti = np.empty(max(k, 0), dtype=np.int64)
    _check(lib.boss_ei_score_topk(arr, y_dim, n_samples, _ptr(Xc), M, _ptr(pm), _ptr(co), _ptr(b), _ptr(ym), _ptr(lbv),
                                  _ptr(ubv), _ptr(cm), k, _ptr(tv), _ptr(ti)), "boss_ei_score_topk")
    return tv, ti


def ei_score_topk_dev(slices, y_dim, n_samples, Xs_ptr, M, coefs, best, y_max, k, lb=None, ub=None, prior_mean_ptr=None,
                      cons_mask_ptr=None, stream=None):
    """Device-pointer variant of ei_score_topk (arguments as ei_score_dev).  -> top_val (k,), top_idx (k,) on the host."""
    arr = _slice_array(slices)
    co = _f64(coefs, (y_dim,))
    b = None if best is None else np.array([best], dtype=np.float64)
    ym = None if y_max is None else _f64(y_max, (y_dim,))
    lbv = None if lb is None else _f64(lb)
    ubv = None if ub is None else _f64(ub)
    k = int(k)
    tv = np.empty(max(k, 0))
    ti = np.empty(max(k, 0), dtype=np.int64)
    _check(lib.boss_ei_score_topk_dev(arr, y_dim, n_samples, _vp(Xs_ptr), int(M),
                                      _vp(prior_mean_ptr) if prior_mean_ptr else None, _ptr(co), _ptr(b), _ptr(ym),
                                      _ptr(lbv), _ptr(ubv), _vp(cons_mask_ptr) if cons_mask_ptr else None, k, _ptr(tv),
                                      _ptr(ti), _vp(stream) if stream else None), "boss_ei_score_topk_dev")
    return tv, ti


FIT_AFFINE, FIT_QUADRATIC, FIT_MAX, FIT_MIN = 1, 2, 3, 4


def mcei_score(slices, y_dim, n_samples, Xs, fit_kind, eps, best, y_max, c0=0.0, c=None, q=None, t=None, lb=None, ub=None,
               cons_mask=None, prior_mean_s=None, want_acq=True):
    """Monte-Carlo EI of a NonlinFitness expression (include/boss_b200.h, boss_mcei_score) on the device.
    eps: (y_dim, K).  -> acq (M,) or None, best_val, best_idx."""
    Xc = _cols(Xs)
    M, d = Xc.shape
    arr = _slice_array(slices)
    ep = np.ascontiguousarray(np.asarray(eps, dtype=np.float64).reshape(y_dim, -1).T)    # (K, y_dim) = column-major y_dim x K
    K = ep.shape[0]
    cv, qv, tv = _opt(c), _opt(q), _opt(t)
    b = None if best is None else np.array([best], dtype=np.float64)
    ym = None if y_max is None else _f64(y_max, (y_dim,))
    lbv = None if lb is None else _f64(lb, (d,))
    ubv = None if ub is None else _f64(ub, (d,))
    cm = None if cons_mask is None else np.ascontiguousarray(cons_mask, dtype=np.uint8)
    pm = None if prior_mean_s is None else np.ascontiguousarray(np.asarray(prior_mean_s, dtype=np.float64).T)
    acq = np.empty(M) if want_acq else None
    bv = C.c_double()
    bi = C.c_int64()
    _check(lib.boss_mcei_score(arr, y_dim, n_samples, _ptr(Xc), M, _ptr(pm), int(fit_kind), float(c0), _ptr(cv), _ptr(qv),
                               _ptr(tv), _ptr(ep), K, _ptr(b), _ptr(ym), _ptr(lbv), _ptr(ubv), _ptr(cm), _ptr(acq),
                               C.byref(bv), C.byref(bi)), "boss_mcei_score")
    return acq, bv.value, bi.value


def _eps_cols(eps, y_dim):
    """eps (y_dim, K) -> (K, y_dim) C-contiguous = column-major y_dim x K, and K."""
    ep = np.ascontiguousarray(np.asarray(eps, dtype=np.float64).reshape(y_dim, -1).T)
    return ep, ep.shape[0]


def mcei_value_grad(slices, y_dim, n_samples, Xs, fit_kind, eps, best, y_max, c0=0.0, c=None, q=None, t=None, lb=None,
                    ub=None, cons_mask=None, prior_mean_s=None, prior_mean_grad_s=None):
    """Value and x-gradient of mcei_score's Monte-Carlo EI (include/boss_b200.h, boss_mcei_value_grad).
    -> acq (M,), grad (d, M).  prior_mean_grad_s: (y_dim, d, M)."""
    Xc = _cols(Xs)
    M, d = Xc.shape
    arr = _slice_array(slices)
    ep, K = _eps_cols(eps, y_dim)
    cv, qv, tv = _opt(c), _opt(q), _opt(t)
    b = None if best is None else np.array([best], dtype=np.float64)
    ym = None if y_max is None else _f64(y_max, (y_dim,))
    lbv = None if lb is None else _f64(lb, (d,))
    ubv = None if ub is None else _f64(ub, (d,))
    cm = None if cons_mask is None else np.ascontiguousarray(cons_mask, dtype=np.uint8)
    pm = None if prior_mean_s is None else np.ascontiguousarray(np.asarray(prior_mean_s, dtype=np.float64).T)
    pmg = None if prior_mean_grad_s is None else np.ascontiguousarray(
        np.transpose(np.asarray(prior_mean_grad_s, dtype=np.float64), (2, 1, 0)))   # (M, d, y_dim)
    acq = np.empty(M)
    grad = np.empty((M, d))
    _check(lib.boss_mcei_value_grad(arr, y_dim, n_samples, _ptr(Xc), M, _ptr(pm), _ptr(pmg), int(fit_kind), float(c0),
                                    _ptr(cv), _ptr(qv), _ptr(tv), _ptr(ep), K, _ptr(b), _ptr(ym), _ptr(lbv), _ptr(ubv),
                                    _ptr(cm), _ptr(acq), _ptr(grad)), "boss_mcei_value_grad")
    return acq, grad.T


def mcei_maximize_multistart(slices, y_dim, n_samples, starts, fit_kind, eps, best, y_max, lb, ub, c0=0.0, c=None,
                             q=None, t=None, iters=60, history=8, discrete_mask=None, prior_mean_affine=None):
    """ei_maximize_multistart on mcei_score's Monte-Carlo EI (boss_mcei_maximize_multistart).
    -> X (d, M), f (M,), best_x (d,), best_val, best_idx, evals."""
    Xc = _cols(starts)
    M, d = Xc.shape
    arr = _slice_array(slices)
    ep, K = _eps_cols(eps, y_dim)
    cv, qv, tv = _opt(c), _opt(q), _opt(t)
    b = None if best is None else np.array([best], dtype=np.float64)
    ym = _opt(y_max)
    lbv, ubv = _f64(lb, (d,)), _f64(ub, (d,))
    dm = _opt(discrete_mask, np.uint8)
    xo = np.empty((M, d)); fo = np.empty(M); bx = np.empty(d)
    bv, bi, ev = C.c_double(), C.c_int64(), C.c_int()
    aff = None if prior_mean_affine is None else _f64(prior_mean_affine, (y_dim, d + 1))
    _check(lib.boss_mcei_maximize_multistart(arr, y_dim, n_samples, _ptr(Xc), M, int(iters), int(history), _ptr(aff),
                                             int(fit_kind), float(c0), _ptr(cv), _ptr(qv), _ptr(tv), _ptr(ep), K, _ptr(b),
                                             _ptr(ym), _ptr(lbv), _ptr(ubv), _ptr(dm), _ptr(xo), _ptr(fo), _ptr(bx),
                                             C.byref(bv), C.byref(bi), C.byref(ev)), "boss_mcei_maximize_multistart")
    return xo.T, fo, bx, bv.value, bi.value, ev.value


def mcei_score_topk(slices, y_dim, n_samples, Xs, fit_kind, eps, best, y_max, k, c0=0.0, c=None, q=None, t=None, lb=None,
                    ub=None, cons_mask=None, prior_mean_s=None):
    """The k best candidates of mcei_score's scores, selected on the device (boss_mcei_score_topk; order as
    ei_score_topk).  -> top_val (k,), top_idx (k,) int64."""
    Xc = _cols(Xs)
    M, d = Xc.shape
    arr = _slice_array(slices)
    ep, K = _eps_cols(eps, y_dim)
    cv, qv, tv_ = _opt(c), _opt(q), _opt(t)
    b = None if best is None else np.array([best], dtype=np.float64)
    ym = None if y_max is None else _f64(y_max, (y_dim,))
    lbv = None if lb is None else _f64(lb, (d,))
    ubv = None if ub is None else _f64(ub, (d,))
    cm = None if cons_mask is None else np.ascontiguousarray(cons_mask, dtype=np.uint8)
    pm = None if prior_mean_s is None else np.ascontiguousarray(np.asarray(prior_mean_s, dtype=np.float64).T)
    k = int(k)
    top_v = np.empty(max(k, 0))
    top_i = np.empty(max(k, 0), dtype=np.int64)
    _check(lib.boss_mcei_score_topk(arr, y_dim, n_samples, _ptr(Xc), M, _ptr(pm), int(fit_kind), float(c0), _ptr(cv),
                                    _ptr(qv), _ptr(tv_), _ptr(ep), K, _ptr(b), _ptr(ym), _ptr(lbv), _ptr(ubv), _ptr(cm), k,
                                    _ptr(top_v), _ptr(top_i)), "boss_mcei_score_topk")
    return top_v, top_i


def _opt(a, dtype=np.float64):
    return None if a is None else np.ascontiguousarray(a, dtype=dtype)


def ei_score_grid(slices, y_dim, n_samples, grid_lo, grid_step, grid_count, coefs, best, y_max, lb=None, ub=None,
                  first=0, M=-1, cons_mask=None, prior_mean_s=None, want_acq=False):
    """Grid candidates generated on the device.  -> acq (or None), best_val, best_idx (global), best_x (d,)."""
    lo, st = _f64(grid_lo), _f64(grid_step)
    d = lo.shape[0]
    cnt = np.ascontiguousarray(grid_count, dtype=np.int64)
    total = int(np.prod(cnt))
    m = total - first if M < 0 else M
    arr = _slice_array(slices)
    co = _f64(coefs, (y_dim,))
    b = None if best is None else np.array([best], dtype=np.float64)
    ym, lbv, ubv = _opt(y_max), _opt(lb), _opt(ub)
    cm = _opt(cons_mask, np.uint8)
    pm = None if prior_mean_s is None else np.ascontiguousarray(np.asarray(prior_mean_s, dtype=np.float64).T)
    acq = np.empty(m) if want_acq else None
    bv, bi, bx = C.c_double(), C.c_int64(), np.empty(d)
    _check(lib.boss_ei_score_grid(arr, y_dim, n_samples, d, _ptr(lo), _ptr(st), _ptr(cnt), int(first), int(M), _ptr(pm),
                                  _ptr(co), _ptr(b), _ptr(ym), _ptr(lbv), _ptr(ubv), _ptr(cm), _ptr(acq), C.byref(bv),
                                  C.byref(bi), _ptr(bx)), "boss_ei_score_grid")
    return acq, bv.value, bi.value, bx


def ei_score_uniform(slices, y_dim, n_samples, seed, M, box_lb, box_ub, coefs, best, y_max, first=0, cons_mask=None,
                     prior_mean_s=None, want_acq=False):
    """Uniform-box candidates generated on the device (stateless counter hash).  -> acq, best_val, best_idx, best_x."""
    lbv, ubv = _f64(box_lb), _f64(box_ub)
    d = lbv.shape[0]
    arr = _slice_array(slices)
    co = _f64(coefs, (y_dim,))
    b = None if best is None else np.array([best], dtype=np.float64)
    ym = _opt(y_max)
    cm = _opt(cons_mask, np.uint8)
    pm = None if prior_mean_s is None else np.ascontiguousarray(np.asarray(prior_mean_s, dtype=np.float64).T)
    acq = np.empty(M) if want_acq else None
    bv, bi, bx = C.c_double(), C.c_int64(), np.empty(d)
    _check(lib.boss_ei_score_uniform(arr, y_dim, n_samples, d, int(seed), int(first), int(M), _ptr(lbv), _ptr(ubv),
                                     _ptr(pm), _ptr(co), _ptr(b), _ptr(ym), _ptr(cm), _ptr(acq), C.byref(bv), C.byref(bi),
                                     _ptr(bx)), "boss_ei_score_uniform")
    return acq, bv.value, bi.value, bx


def ei_maximize_multistart(slices, y_dim, n_samples, starts, coefs, best, y_max, lb, ub, iters=60, history=8,
                           discrete_mask=None, prior_mean_affine=None):
    """Device-resident lock-step multi-start L-BFGS.  -> X (d, M), f (M,), best_x (d,), best_val, best_idx, evals."""
    Xc = _cols(starts)
    M, d = Xc.shape
    arr = _slice_array(slices)
    co = _f64(coefs, (y_dim,))
    b = None if best is None else np.array([best], dtype=np.float64)
    ym = _opt(y_max)
    lbv, ubv = _f64(lb, (d,)), _f64(ub, (d,))
    dm = _opt(discrete_mask, np.uint8)
    xo = np.empty((M, d)); fo = np.empty(M); bx = np.empty(d)
    bv, bi, ev = C.c_double(), C.c_int64(), C.c_int()
    aff = None if prior_mean_affine is None else _f64(prior_mean_affine, (y_dim, d + 1))
    _check(lib.boss_ei_maximize_multistart(arr, y_dim, n_samples, _ptr(Xc), M, int(iters), int(history), _ptr(aff),
                                           _ptr(co), _ptr(b),
                                           _ptr(ym), _ptr(lbv), _ptr(ubv), _ptr(dm), _ptr(xo), _ptr(fo), _ptr(bx),
                                           C.byref(bv), C.byref(bi), C.byref(ev)), "boss_ei_maximize_multistart")
    return xo.T, fo, bx, bv.value, bi.value, ev.value


def uniform_candidates(seed, first, M, box_lb, box_ub):
    """Host reproduction of the device generator (tests, and callers that want the coordinates of an index)."""
    lbv, ubv = _f64(box_lb), _f64(box_ub)
    d = lbv.shape[0]
    ctr = (np.arange(first, first + M, dtype=np.uint64)[:, None] * np.uint64(d) + np.arange(d, dtype=np.uint64)[None, :])
    with np.errstate(over="ignore"):
        z = np.uint64(seed) + (ctr + np.uint64(1)) * np.uint64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        z = z ^ (z >> np.uint64(31))
    u = (z >> np.uint64(11)).astype(np.float64) * (1.0 / 9007199254740992.0)
    return (lbv[None, :] + u * (ubv - lbv)[None, :]).T          # d x M  (lb + u*w is one rounding apart from fma at most)


def ei_value_grad(slices, y_dim, n_samples, Xs, coefs, best, y_max, lb=None, ub=None, cons_mask=None,
                  prior_mean_s=None, prior_mean_grad_s=None):
    """-> acq (M,), grad (d, M).  prior_mean_grad_s: (y_dim, d, M)."""
    Xc = _cols(Xs)
    M, d = Xc.shape
    arr = _slice_array(slices)
    co = _f64(coefs, (y_dim,))
    b = None if best is None else np.array([best], dtype=np.float64)
    ym = None if y_max is None else _f64(y_max, (y_dim,))
    lbv = None if lb is None else _f64(lb, (d,))
    ubv = None if ub is None else _f64(ub, (d,))
    cm = None if cons_mask is None else np.ascontiguousarray(cons_mask, dtype=np.uint8)
    pm = None if prior_mean_s is None else np.ascontiguousarray(np.asarray(prior_mean_s, dtype=np.float64).T)
    pmg = None if prior_mean_grad_s is None else np.ascontiguousarray(
        np.transpose(np.asarray(prior_mean_grad_s, dtype=np.float64), (2, 1, 0)))   # (M, d, y_dim)
    acq = np.empty(M)
    grad = np.empty((M, d))
    _check(lib.boss_ei_value_grad(arr, y_dim, n_samples, _ptr(Xc), M, _ptr(pm), _ptr(pmg), _ptr(co), _ptr(b), _ptr(ym),
                                  _ptr(lbv), _ptr(ubv), _ptr(cm), _ptr(acq), _ptr(grad)), "boss_ei_value_grad")
    return acq, grad.T


def ei_value_grad_dev(slices, y_dim, n_samples, Xs_ptr, M, coefs, best, y_max, acq_ptr, grad_ptr, lb=None, ub=None,
                      prior_mean_ptr=None, prior_mean_grad_ptr=None, stream=None):
    """`stream`: raw cudaStream_t the device arrays were produced on (None = legacy default stream)."""
    arr = _slice_array(slices)
    co = _f64(coefs, (y_dim,))
    b = None if best is None else np.array([best], dtype=np.float64)
    ym = None if y_max is None else _f64(y_max, (y_dim,))
    lbv = None if lb is None else _f64(lb)
    ubv = None if ub is None else _f64(ub)
    _check(lib.boss_ei_value_grad_dev(arr, y_dim, n_samples, _vp(Xs_ptr), int(M),
                                      _vp(prior_mean_ptr) if prior_mean_ptr else None,
                                      _vp(prior_mean_grad_ptr) if prior_mean_grad_ptr else None, _ptr(co), _ptr(b),
                                      _ptr(ym), _ptr(lbv), _ptr(ubv), None, _vp(acq_ptr) if acq_ptr else None,
                                      _vp(grad_ptr), _vp(stream) if stream else None), "boss_ei_value_grad_dev")


def ei_score_dev(slices, y_dim, n_samples, Xs_ptr, M, coefs, best, y_max, lb=None, ub=None, acq_ptr=None,
                 prior_mean_ptr=None, cons_mask_ptr=None, stream=None):
    """Device-pointer variant: Xs_ptr etc. are raw CUDA addresses (e.g. torch.Tensor.data_ptr()); `stream` is the raw
    cudaStream_t they were produced on (None = legacy default stream, torch's default)."""
    arr = _slice_array(slices)
    co = _f64(coefs, (y_dim,))
    b = None if best is None else np.array([best], dtype=np.float64)
    ym = None if y_max is None else _f64(y_max, (y_dim,))
    lbv = None if lb is None else _f64(lb)
    ubv = None if ub is None else _f64(ub)
    bv = C.c_double()
    bi = C.c_int64()
    _check(lib.boss_ei_score_dev(arr, y_dim, n_samples, _vp(Xs_ptr), int(M), _vp(prior_mean_ptr) if prior_mean_ptr else None,
                                 _ptr(co), _ptr(b), _ptr(ym), _ptr(lbv), _ptr(ubv),
                                 _vp(cons_mask_ptr) if cons_mask_ptr else None, _vp(acq_ptr) if acq_ptr else None, None,
                                 C.byref(bv), C.byref(bi), _vp(stream) if stream else None), "boss_ei_score_dev")
    return bv.value, bi.value


def loglik_batch(X, Y_minus_mean, lengthscales, amplitude, noise_std, kernel_id=KERNEL_MATERN52, discrete_mask=None):
    """lengthscales (S, d), amplitude (S,), noise_std (S,), Y_minus_mean (n,) shared or (S, n) -> (S,)"""
    Xc = _cols(X)
    n, d = Xc.shape
    ls = _f64(lengthscales)
    S = ls.shape[0]
    assert ls.shape == (S, d)
    amp = _f64(amplitude, (S,))
    ns = _f64(noise_std, (S,))
    Y = _f64(Y_minus_mean)
    ldy = 0 if Y.ndim == 1 else n
    assert Y.shape == ((n,) if ldy == 0 else (S, n))
    dm = None if discrete_mask is None else np.ascontiguousarray(discrete_mask, dtype=np.uint8)
    out = np.empty(S)
    _check(lib.boss_gp_loglik_batch(_ptr(Xc), d, n, _ptr(Y), ldy, _ptr(ls), _ptr(amp), _ptr(ns), int(kernel_id),
                                    _ptr(dm), S, _ptr(out)), "boss_gp_loglik_batch")
    return out


def loglik_grad_batch(X, Y_minus_mean, lengthscales, amplitude, noise_std, kernel_id=KERNEL_MATERN52, discrete_mask=None):
    """-> loglik (S,), grad (S, d + 2) ordered [d lengthscales, amplitude, noise_std]."""
    Xc = _cols(X)
    n, d = Xc.shape
    ls = _f64(lengthscales)
    S = ls.shape[0]
    assert ls.shape == (S, d)
    amp = _f64(amplitude, (S,))
    ns = _f64(noise_std, (S,))
    Y = _f64(Y_minus_mean)
    ldy = 0 if Y.ndim == 1 else n
    dm = None if discrete_mask is None else np.ascontiguousarray(discrete_mask, dtype=np.uint8)
    out = np.empty(S)
    grad = np.empty((S, d + 2))
    _check(lib.boss_gp_loglik_grad_batch(_ptr(Xc), d, n, _ptr(Y), ldy, _ptr(ls), _ptr(amp), _ptr(ns), int(kernel_id),
                                         _ptr(dm), S, _ptr(out), _ptr(grad)), "boss_gp_loglik_grad_batch")
    return out, grad


def loglik_grad_batch_dev(X_ptr, d, n, Y_ptr, ldy, ls_ptr, amp_ptr, noise_ptr, kernel_id, S, out_ptr, grad_ptr,
                          stream=None):
    _check(lib.boss_gp_loglik_grad_batch_dev(_vp(X_ptr), d, n, _vp(Y_ptr), ldy, _vp(ls_ptr), _vp(amp_ptr), _vp(noise_ptr),
                                             int(kernel_id), None, int(S), _vp(out_ptr), _vp(grad_ptr),
                                             _vp(stream) if stream else None),
           "boss_gp_loglik_grad_batch_dev")


def loglik_grad_batch_mean(X, Y_minus_mean, J, lengthscales, amplitude, noise_std, kernel_id=KERNEL_MATERN52,
                           discrete_mask=None):
    """loglik_grad_batch plus the gradient w.r.t. the parameters theta of the prior mean, alpha^T J per sample.
    J = dm(X; theta)/dtheta at the training inputs: (k, n) shared by all samples or (S, k, n) per sample (row c of a
    sample is column c of ForwardDiff.jacobian's n x k matrix).  -> loglik (S,), grad (S, d + 2), grad_mean (S, k)."""
    Xc = _cols(X)
    n, d = Xc.shape
    ls = _f64(lengthscales)
    S = ls.shape[0]
    assert ls.shape == (S, d)
    amp = _f64(amplitude, (S,))
    ns = _f64(noise_std, (S,))
    Y = _f64(Y_minus_mean)
    ldy = 0 if Y.ndim == 1 else n
    Jc = _f64(J)
    assert Jc.ndim in (2, 3) and Jc.shape[-1] == n and (Jc.ndim == 2 or Jc.shape[0] == S)
    k = Jc.shape[-2]
    ldj = 0 if Jc.ndim == 2 else k * n
    dm = None if discrete_mask is None else np.ascontiguousarray(discrete_mask, dtype=np.uint8)
    out = np.empty(S)
    grad = np.empty((S, d + 2))
    gm = np.empty((S, k))
    _check(lib.boss_gp_loglik_grad_batch_mean(_ptr(Xc), d, n, _ptr(Y), ldy, _ptr(Jc), k, ldj, _ptr(ls), _ptr(amp), _ptr(ns),
                                              int(kernel_id), _ptr(dm), S, _ptr(out), _ptr(grad), _ptr(gm)),
           "boss_gp_loglik_grad_batch_mean")
    return out, grad, gm


def loglik_grad_batch_mean_dev(X_ptr, d, n, Y_ptr, ldy, J_ptr, k, ldj, ls_ptr, amp_ptr, noise_ptr, kernel_id, S, out_ptr,
                               grad_ptr, grad_mean_ptr, discrete_mask=None, stream=None):
    dm = None if discrete_mask is None else np.ascontiguousarray(discrete_mask, dtype=np.uint8)
    _check(lib.boss_gp_loglik_grad_batch_mean_dev(_vp(X_ptr), d, n, _vp(Y_ptr), ldy, _vp(J_ptr), int(k), int(ldj),
                                                  _vp(ls_ptr), _vp(amp_ptr), _vp(noise_ptr), int(kernel_id), _ptr(dm),
                                                  int(S), _vp(out_ptr), _vp(grad_ptr), _vp(grad_mean_ptr),
                                                  _vp(stream) if stream else None),
           "boss_gp_loglik_grad_batch_mean_dev")


def loglik_batch_dev(X_ptr, d, n, Y_ptr, ldy, ls_ptr, amp_ptr, noise_ptr, kernel_id, S, out_ptr, discrete_mask=None,
                     stream=None):
    dm = None if discrete_mask is None else np.ascontiguousarray(discrete_mask, dtype=np.uint8)
    _check(lib.boss_gp_loglik_batch_dev(_vp(X_ptr), d, n, _vp(Y_ptr), ldy, _vp(ls_ptr), _vp(amp_ptr), _vp(noise_ptr),
                                        int(kernel_id), _ptr(dm), int(S), _vp(out_ptr), _vp(stream) if stream else None),
           "boss_gp_loglik_batch_dev")


def gp_map_multistart(X, Y_minus_mean, prior_kind, prior_par, starts, kernel_id=KERNEL_MATERN52, discrete_mask=None,
                      iters=40, history=8):
    """Device-resident MAP fit of the hyper-parameters (boss_gp_map_multistart): every output slice on its own, all
    (slice, start) pairs in lock-step.  X (d, n); Y_minus_mean (y_dim, n); prior_kind (y_dim, P) int, prior_par
    (y_dim, P, 2) with P = d + 2 entries [lambda_1..lambda_d, alpha, sigma]; starts (y_dim, M, P) raw values.
    -> params (y_dim, M, P), f (y_dim, M), best_params (y_dim, P), best_val (y_dim,), best_idx (y_dim,), evals."""
    Xc = _cols(X)
    n, d = Xc.shape
    P = d + 2
    Y = _f64(np.atleast_2d(Y_minus_mean))
    y_dim = Y.shape[0]
    assert Y.shape == (y_dim, n)
    kind = np.ascontiguousarray(prior_kind, dtype=np.int32)
    assert kind.shape == (y_dim, P), kind.shape
    par = _f64(prior_par, (y_dim, P, 2))
    st = _f64(starts)
    assert st.ndim == 3 and st.shape[0] == y_dim and st.shape[2] == P, st.shape
    M = st.shape[1]
    dm = _opt(discrete_mask, np.uint8)
    po = np.empty((y_dim, M, P)); fo = np.empty((y_dim, M)); bp = np.empty((y_dim, P))
    bv = np.empty(y_dim); bi = np.empty(y_dim, dtype=np.int64)
    ev = C.c_int()
    _check(lib.boss_gp_map_multistart(_ptr(Xc), d, n, y_dim, _ptr(Y), int(kernel_id), _ptr(dm), _ptr(kind), _ptr(par),
                                      _ptr(st), M, int(iters), int(history), _ptr(po), _ptr(fo), _ptr(bp), _ptr(bv),
                                      _ptr(bi), C.byref(ev)), "boss_gp_map_multistart")
    return po, fo, bp, bv, bi, ev.value


def set_timing(on: bool):
    lib.boss_set_timing(1 if on else 0)


def last_kernel_ms(which: int):
    return lib.boss_last_kernel_ms(which), lib.boss_last_kernel_count(which)


def launch_count() -> int:
    return lib.boss_launch_count()


def dbg_gemm_nt(A, B):
    A = _f64(A)
    B = _f64(B)
    M, K = A.shape
    N = B.shape[0]
    Cm = np.empty((M, N))
    _check(lib.boss_dbg_gemm_nt(_ptr(A), _ptr(B), M, N, K, _ptr(Cm)), "boss_dbg_gemm_nt")
    return Cm


def dbg_kernel_fn(which, t):
    t = _f64(t)
    out = np.empty_like(t)
    _check(lib.boss_dbg_kernel_fn(int(which), _ptr(t), t.size, _ptr(out)), "boss_dbg_kernel_fn")
    return out


def dbg_kernel_fn_id(kernel_id, which, d2):
    """The covariance function of kernel_id at squared distances d2: which = 0 kappa_fast, 1 kappa'(r)/r fast,
    2 kappa (libm), 3 kappa'(r)/r (libm)."""
    d2 = _f64(d2)
    out = np.empty_like(d2)
    _check(lib.boss_dbg_kernel_fn_id(int(kernel_id), int(which), _ptr(d2), d2.size, _ptr(out)), "boss_dbg_kernel_fn_id")
    return out


def dbg_factors(gp: GP):
    n = gp.n
    L = np.empty((n, n))
    W = np.empty((n, n))
    al = np.empty(n)
    _check(lib.boss_dbg_factors(gp.handle, _ptr(L), _ptr(W), _ptr(al)), "boss_dbg_factors")
    return L, W, al


def dbg_check_redzones():
    """(overwritten guard bytes, allocations scanned); (-1, 0) unless the process runs with BOSS_DEBUG_REDZONE=1."""
    n = C.c_int64(0)
    bad = lib.boss_dbg_check_redzones(C.byref(n))
    return int(bad), int(n.value)


def dbg_screen_stats():
    """Argmax / top-k screening of the last scoring call on the current device: (state, candidates bounded, survivors);
    state 0 = not screened, 1 = screened, 2 = fell back to the full path after the first chunk."""
    out = (C.c_int64 * 3)()
    _check(lib.boss_dbg_screen_stats(out), "boss_dbg_screen_stats")
    return int(out[0]), int(out[1]), int(out[2])


def dbg_score_paths():
    """The paths of the last scoring call on the current device, counted per (chunk, slice) pass: dict with keys
    wide_fused, wide_split (wide without the fused epilogue), narrow, quarter, xgrad."""
    out = (C.c_int64 * 5)()
    _check(lib.boss_dbg_score_paths(out), "boss_dbg_score_paths")
    return dict(zip(("wide_fused", "wide_split", "narrow", "quarter", "xgrad"), (int(v) for v in out)))


def dbg_screen_ambiguous():
    """The FP32 mean tier of the last screened call: (candidates in the ambiguous band, pool as the chunks left it --
    definite keeps plus ambiguous candidates -- before the FP64 refinement and the re-seed)."""
    out = (C.c_int64 * 2)()
    _check(lib.boss_dbg_screen_ambiguous(out), "boss_dbg_screen_ambiguous")
    return int(out[0]), int(out[1])


def dbg_screen_var():
    """The variance tier of the last screened call (W's first row block, DESIGN.md 2.9): (pool rows it bounded, rows it
    kept for the exact pass); (0, 0) when it did not run."""
    out = (C.c_int64 * 2)()
    _check(lib.boss_dbg_screen_var(out), "boss_dbg_screen_var")
    return int(out[0]), int(out[1])


def dbg_screen_mean(gp: GP, Xs):
    """(mu~, E, mu64) of the candidates Xs (d x M) under gp: the FP32 tier's mean and error bound, and the FP64 mean
    (K*^T alpha, no prior mean)."""
    Xc = _cols(Xs)
    M = Xc.shape[0]
    mu32, E, mu64 = np.empty(M), np.empty(M), np.empty(M)
    _check(lib.boss_dbg_screen_mean(gp.handle, _ptr(Xc), M, _ptr(mu32), _ptr(E), _ptr(mu64)), "boss_dbg_screen_mean")
    return mu32, E, mu64


def dbg_kappa_f32(kid, r):
    """The FP32 tier's kappa at d2 = float32(r^2) (kid 0 SE, 1 Matern32, 2 Matern52)."""
    r = _f64(r)
    out = np.empty_like(r)
    _check(lib.boss_dbg_kappa_f32(int(kid), _ptr(r), r.size, _ptr(out)), "boss_dbg_kappa_f32")
    return out


def dbg_mma_d2(dp, u, t, nu, nt):
    """The FP32 tier's tensor-core d2 = nu + nt - 2 u.t (before the clamp at 0) for FP32 points u (m x kp, m a
    multiple of 16) and t (n x kp, n a multiple of 8), kp = dp rounded up to the kernels' 8, 16 or 32."""
    u, t = np.ascontiguousarray(u, np.float32), np.ascontiguousarray(t, np.float32)
    nu, nt = np.ascontiguousarray(nu, np.float32), np.ascontiguousarray(nt, np.float32)
    m, n = u.shape[0], t.shape[0]
    out = np.empty((m, n), np.float32)
    _check(lib.boss_dbg_mma_d2(int(dp), u.ctypes.data, t.ctypes.data, nu.ctypes.data, nt.ctypes.data, m // 16, n // 8,
                               out.ctypes.data), "boss_dbg_mma_d2")
    return out

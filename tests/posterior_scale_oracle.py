"""References for the posterior, its x-gradients and EI at the sizes the scoring path runs at (n up to a few thousand,
M up to tens of thousands), and a mirror of how the scoring call (boss.jl_b200/csrc/boss_b200.cu, `ScoreCall::setup`
and `score_slice`) cuts a call into chunks and picks a path for every (chunk, slice) pass.

- `reference(kernel)`: the FP64 oracle for every covariance function (oracle.boss_oracle for SE / Matern-3/2 /
  Matern-5/2, tests/kernels_more_oracle.py's copy for Matern-1/2 and RQ), with its posterior_fit, mean_and_var,
  mean_var_grad, ei_value_grad, ei_acquisition and posterior_cov.
- `adjudicator_post_grad_longdouble`: mu, sigma^2, d mu / dx and d sigma^2 / dx in x87 extended precision (numpy
  longdouble): direct distances, the column Cholesky written out, W = L^-1, u = W^T W k* = K^-1 k* and the derivative
  formulas of csrc/grad.cuh's header comment.
- `post_bounds`, `ratio`, `grad_ratio`: the comparisons a device result is held to (<= 1 passes).  Mean and variance use the
  rule of tests/test_gpu_parity_adversarial.py: 1e-9 relative, floored by the conditioning of K and the rounding of
  the scaled distances.  Gradients: per dimension j, max_m |g_jm - ref_jm| <= 1e-8 max_m |ref_jm|.
- `perturbed_post_grad`: the FP64 reference formed through W explicitly, with one deliberate defect (a zeroed tile of
  W, a zeroed ragged block of K*^T, a dropped block of W^T, a wrong 1/l in the derivative): the host tests show the
  comparisons reject each of them.
- `score_plan`: the chunks of a scoring call and the path of every (chunk, slice) pass.
"""
from __future__ import annotations

import numpy as np
import scipy.linalg as sl

from oracle import boss_oracle as OB
from tests.kernels_more_oracle import O as OK
from tests.loglik_scale_oracle import _kappa_ld

EPS = 2.0 ** -52
TOL_POST, TOL_GRAD = 1e-9, 1e-8
TM = 128                                     # csrc/common.cuh `TM`, rows of a block
NW_NB = 32                                   # csrc/score_narrow.cuh `NW_NB`, candidates of a narrow / quarter CTA
NSM = 148                                    # SMs of the B200 the cost model counts waves over
NQ_COST_CHAIN, NQ_COST_WORK, NQ_COST_FIXED = 0.085, 0.0019, 0.15   # csrc/boss_b200.cu, same names
PGRAD_SLOT_BYTES = 256 << 20                 # csrc/boss_b200.cu `PGRAD_SLOT_BYTES`
PATHS = ("wide_fused", "wide_split", "narrow", "quarter")


# ---- references ----------------------------------------------------------------------------------------------------

def reference(kernel):
    """The shared oracle for SE / Matern-3/2 / Matern-5/2, kernels_more_oracle's extended copy for the others."""
    return OB if kernel in (OB.KERNEL_SE, OB.KERNEL_MATERN32, OB.KERNEL_MATERN52) else OK


def _scaled(X, Xs, ls, mask):
    inv = 1.0 / ls
    return OB.discrete_round(mask, X) * inv[:, None], OB.discrete_round(mask, Xs) * inv[:, None], inv


def adjudicator_post_grad_longdouble(X, y_minus_mean, lengthscales, amplitude, noise_std, kernel, Xs, mask=None):
    """-> mu (M,), var (M,) (raw: before the clip at 0, with the 1e-18 jitter), dmu (d, M), dvar (d, M) as float64
    roundings of the extended-precision values.  Discrete dimensions have zero derivative; Matern-1/2 takes
    kappa'(r)/r = 0 at r = 0.  Cost ~ n^3 / 2 long-double multiply-adds plus 2 n^2 M (n = 1024: a few seconds)."""
    LD = np.longdouble
    X = OB.discrete_round(mask, np.asarray(X, dtype=np.float64)).astype(LD)
    Xs = OB.discrete_round(mask, np.asarray(Xs, dtype=np.float64)).astype(LD)
    d, n = X.shape
    ls = np.asarray(lengthscales, dtype=np.float64).astype(LD) + LD(OB.MIN_PARAM_VALUE)
    a = LD(float(amplitude)) + LD(OB.MIN_PARAM_VALUE)
    s = LD(float(noise_std)) + LD(OB.MIN_PARAM_VALUE)
    inv = 1 / ls
    Xa, Xb = X * inv[:, None], Xs * inv[:, None]

    def sqdist(A, B):
        D2 = np.zeros((A.shape[1], B.shape[1]), dtype=LD)
        for q in range(d):
            diff = A[q][:, None] - B[q][None, :]
            D2 += diff * diff
        return D2

    a2 = a * a
    K = a2 * _kappa_ld(sqdist(Xa, Xa), kernel)[0]
    K[np.diag_indices(n)] += s * s
    L = np.zeros((n, n), dtype=LD)
    for j in range(n):                                   # column Cholesky
        v = K[j:, j] - L[j:, :j] @ L[j, :j]
        L[j, j] = np.sqrt(v[0])
        L[j + 1:, j] = v[1:] / L[j, j]
    W = np.zeros((n, n), dtype=LD)                       # W = L^-1 (lower), row by row
    for i in range(n):
        W[i, i] = 1 / L[i, i]
        if i:
            W[i, :i] = -(L[i, :i] @ W[:i, :i]) / L[i, i]
    alpha = W.T @ (W @ np.asarray(y_minus_mean, dtype=np.float64).astype(LD))
    kap, g = _kappa_ld(sqdist(Xa, Xb), kernel)           # n x M
    Ks, G = a2 * kap, a2 * g
    V = W @ Ks
    u = W.T @ V                                          # K^-1 k*
    mu = Ks.T @ alpha
    var = a2 - np.sum(V * V, axis=0) + LD(OB.DEFAULT_JITTER)
    M = Xs.shape[1]
    dmu = np.zeros((d, M), dtype=LD)
    dvar = np.zeros((d, M), dtype=LD)
    for j in range(d):
        if mask is not None and mask[j]:
            continue
        dk = G * (Xb[j][None, :] - Xa[j][:, None]) * inv[j]
        dmu[j] = alpha @ dk
        dvar[j] = -2 * np.sum(u * dk, axis=0)
    return mu.astype(np.float64), var.astype(np.float64), dmu.astype(np.float64), dvar.astype(np.float64)


def mp_post_grad(X, y_minus_mean, lengthscales, amplitude, noise_std, kernel, Xs, mask=None, dps=40):
    """40-digit reference (n <~ 12): mu and var in mpmath, their x-gradients by mp.diff of mu and var in each coordinate
    of the candidate (discrete coordinates rounded inside the function, so their derivative is 0)."""
    import mpmath as mp
    from tests.kernels_more_oracle import _mp_kappa
    mp.mp.dps = dps
    X = OB.discrete_round(mask, np.asarray(X, dtype=np.float64))
    Xs = np.asarray(Xs, dtype=np.float64)
    d, n = X.shape
    eps = mp.mpf(OB.MIN_PARAM_VALUE)
    ls = [mp.mpf(float(v)) + eps for v in lengthscales]
    a2 = (mp.mpf(float(amplitude)) + eps) ** 2
    s2 = (mp.mpf(float(noise_std)) + eps) ** 2
    Xm = [[mp.mpf(float(X[q, i])) for i in range(n)] for q in range(d)]

    def k(p, i):
        d2 = sum(((p[q] - Xm[q][i]) / ls[q]) ** 2 for q in range(d))
        return a2 * _mp_kappa(mp, d2, kernel)

    K = mp.matrix(n, n)
    for i in range(n):
        for j in range(n):
            K[i, j] = k([Xm[q][i] for q in range(d)], j) + (s2 if i == j else 0)
    L = mp.cholesky(K)
    alpha = mp.lu_solve(L.T, mp.lu_solve(L, mp.matrix([mp.mpf(float(v)) for v in y_minus_mean])))

    def post(p):
        p = [mp.nint(p[q]) if mask is not None and mask[q] else p[q] for q in range(d)]
        ks = mp.matrix([k(p, i) for i in range(n)])
        v = mp.lu_solve(L, ks)
        return sum(ks[i] * alpha[i] for i in range(n)), a2 - sum(v[i] ** 2 for i in range(n)) + mp.mpf(OB.DEFAULT_JITTER)

    M = Xs.shape[1]
    mu, var = np.empty(M), np.empty(M)
    dmu, dvar = np.empty((d, M)), np.empty((d, M))
    for m in range(M):
        p0 = [mp.mpf(float(Xs[q, m])) for q in range(d)]
        mu_m, var_m = post(p0)
        mu[m], var[m] = float(mu_m), float(var_m)
        for j in range(d):
            def f(t, j=j, which=0):
                p = list(p0)
                p[j] = t
                return post(p)[which]
            dmu[j, m] = float(mp.diff(lambda t: f(t, which=0), p0[j]))
            dvar[j, m] = float(mp.diff(lambda t: f(t, which=1), p0[j]))
    return mu, var, dmu, dvar


def perturbed_post_grad(X, y_minus_mean, lengthscales, amplitude, noise_std, kernel, Xs, mask=None, zero_w_tile=None,
                        zero_ks_tail=None, drop_wt_last_rows=False, dinvl=None):
    """The FP64 posterior and its x-gradients formed through W = L^-1 (what the device stores), with at most one defect:
    zero_w_tile = (bi, bj): that 128 x 128 tile of W zeroed (V = W k* and u = W^T V both see it); zero_ks_tail = m: the
    live rows of the last row block of K*^T zeroed for candidate m; drop_wt_last_rows: u = W^T V without W^T's last row
    block; dinvl = (j, rel): 1/l_j multiplied by 1 + rel in the derivative's chain factor only.
    -> mu, var (raw), dmu (d, M), dvar (d, M)."""
    Om = reference(kernel)
    X = np.asarray(X, dtype=np.float64)
    ls, amp, noise = OB.condition_params(lengthscales, amplitude, noise_std)
    d, n = X.shape
    Xa, Xb, inv = _scaled(X, np.asarray(Xs, dtype=np.float64), ls, mask)
    K = amp * amp * Om._kappa(OB._pairwise_sqdist_direct(Xa, Xa), kernel)
    K[np.diag_indices(n)] += noise * noise
    Lc = np.linalg.cholesky(K)
    W = sl.solve_triangular(Lc, np.eye(n), lower=True, check_finite=False)
    alpha = W.T @ (W @ np.asarray(y_minus_mean, dtype=np.float64))
    D2 = OB._pairwise_sqdist_direct(Xa, Xb)
    Ks = amp * amp * Om._kappa(D2, kernel)
    G = amp * amp * Om._kappa_dr_over_r(D2, kernel)
    if zero_ks_tail is not None:
        r0 = (n - 1) // TM * TM
        Ks[r0:, zero_ks_tail] = 0.0
        G[r0:, zero_ks_tail] = 0.0
    Wp = W.copy()
    if zero_w_tile is not None:
        bi, bj = zero_w_tile
        Wp[bi * TM:(bi + 1) * TM, bj * TM:(bj + 1) * TM] = 0.0
    V = Wp @ Ks
    WT = Wp.T.copy()
    if drop_wt_last_rows:
        WT[(n - 1) // TM * TM:] = 0.0
    u = WT @ V
    mu = Ks.T @ alpha
    var = amp * amp - np.sum(V * V, axis=0) + OB.DEFAULT_JITTER
    M = Ks.shape[1]
    dmu, dvar = np.zeros((d, M)), np.zeros((d, M))
    for j in range(d):
        if mask is not None and mask[j]:
            continue
        f = inv[j] * (1.0 + dinvl[1] if dinvl is not None and dinvl[0] == j else 1.0)
        dk = G * (Xb[j][None, :] - Xa[j][:, None]) * f
        dmu[j] = alpha @ dk
        dvar[j] = -2.0 * np.sum(u * dk, axis=0)
    return mu, var, dmu, dvar


# ---- comparisons ---------------------------------------------------------------------------------------------------

def ratio(got, ref, rel, floor):
    """max |got - ref| / max(rel |ref|, floor): tests/test_gpu_parity_adversarial.py's comparison rule."""
    got = np.asarray(got, dtype=np.float64); ref = np.asarray(ref, dtype=np.float64)
    return float(np.max(np.abs(got - ref) / np.maximum(rel * np.abs(ref), floor))) if ref.size else 0.0


def floors(kappa, a2, y_absmax, alpha_l1, u1, x2):
    """The floors of the mean / variance rule (tests/test_gpu_parity_adversarial.py's module docstring):
    f_var = 4 kappa eps a^2 + 2 |u|_1 (1 + |u|_1) dk,  f_mu = 4 kappa eps max|y - m| + |alpha|_1 (1 + |u|_1) dk,
    kappa = cond_2(K), u1 = max over candidates of |K^-1 k*|_1, dk = 12 eps a^2 max|x~|^2.  -> (f_mu, f_var)."""
    dk = 12 * EPS * a2 * x2
    return 4 * kappa * EPS * y_absmax + alpha_l1 * (1 + u1) * dk, 4 * kappa * EPS * a2 + 2 * u1 * (1 + u1) * dk


def post_bounds(X, y_minus_mean, lengthscales, amplitude, noise_std, kernel, Xs, mask=None):
    """`floors` of one GP at the candidates Xs, with kappa = lambda_max / lambda_min of the symmetric eigenvalues
    (cond_2 of the positive definite K, at a fraction of the cost of an SVD).  -> (f_mu, f_var)."""
    Om = reference(kernel)
    X = np.asarray(X, dtype=np.float64); Xs = np.asarray(Xs, dtype=np.float64)
    ls, amp, noise = OB.condition_params(lengthscales, amplitude, noise_std)
    a2 = amp * amp
    Xa, Xb, _ = _scaled(X, Xs, ls, mask)
    K = a2 * Om._kappa(OB._pairwise_sqdist_direct(Xa, Xa), kernel)
    K[np.diag_indices(X.shape[1])] += noise * noise
    ev = sl.eigvalsh(K, check_finite=False)
    kappa = float(ev[-1] / ev[0])
    y = np.asarray(y_minus_mean, dtype=np.float64)
    cf = sl.cho_factor(K, check_finite=False)
    alpha = sl.cho_solve(cf, y, check_finite=False)
    U = sl.cho_solve(cf, a2 * Om._kappa(OB._pairwise_sqdist_direct(Xa, Xb), kernel), check_finite=False)
    u1 = float(np.max(np.sum(np.abs(U), axis=0)))
    x2 = max(float(np.max(np.sum(Xa ** 2, axis=0))), float(np.max(np.sum(Xb ** 2, axis=0))))
    return floors(kappa, a2, float(np.max(np.abs(y))), float(np.sum(np.abs(alpha))), u1, x2)


def grad_ratio(g, ref, tol=TOL_GRAD):
    """Per dimension (every leading index), max_m |g - ref| over tol max_m |ref| (1 where ref is all zero)."""
    g, ref = np.asarray(g, dtype=np.float64), np.asarray(ref, dtype=np.float64)
    scale = np.max(np.abs(ref), axis=-1, keepdims=True)
    scale = np.where(scale > 0, scale, 1.0)
    return float(np.max(np.abs(g - ref) / (tol * scale))) if ref.size else 0.0


def post_grad_ratios(got, ref, bounds):
    """got / ref = (mu, var, dmu, dvar); bounds = post_bounds(...) -> dict of the four ratios."""
    f_mu, f_var = bounds
    return dict(mu=ratio(got[0], ref[0], TOL_POST, f_mu), var=ratio(got[1], ref[1], TOL_POST, f_var),
                dmu=grad_ratio(got[2], ref[2]), dvar=grad_ratio(got[3], ref[3]))


# ---- chunks and paths ----------------------------------------------------------------------------------------------

def pick_row_splits(ncb, nblk):
    """pick_row_splits of csrc/boss_b200.cu -> (splits, cost in block-steps)."""
    cost = ((ncb + NSM - 1) // NSM) * (nblk * (nblk + 1) // 2 + 1.0)
    if ncb >= 4 * NSM or nblk < 2:
        return 1, cost
    best_t, best = 1e300, 1
    for ns in range(1, nblk + 1):
        maxw = 0
        for y in range(ns):
            w, j = 0, 0
            while True:
                i = (j >> 1) * 2 * ns + ((2 * ns - 1 - y) if (j & 1) else y)
                if i >= nblk:
                    break
                w += i + 1
                j += 1
            maxw = max(maxw, w)
        waves = (ncb * ns + NSM - 1) // NSM
        t = waves * (maxw + 1.0)
        if t < best_t * (1.0 - 1e-9):
            best_t, best = t, ns
    return best, best_t


def chunk_capacity(n_per_slice, M, d, xgrad, pgrad=False):
    """ScoreCall::setup's chunk leading dimension CH and have_vt (csrc/boss_b200.cu)."""
    max_npad = max((n + TM - 1) // TM * TM for n in n_per_slice)
    nsl = len(n_per_slice)
    ncb_max = min((4 << 30) // (1024 * max_npad), 592)                          # ScoreCall::setup's ncb_max
    if ncb_max >= NSM:
        ncb_max = ncb_max // NSM * NSM
    xgrad = xgrad or pgrad                                                       # ScoreArgs::xgrad
    if xgrad:
        ncb_max = max(1, min(ncb_max, 296))                                      # a.xgrad() cap
    if pgrad:
        per_block = 128 * nsl * (20 + 16 * d)                                    # a.pgrad(): per_block
        ncb_max = max(1, min(ncb_max, PGRAD_SLOT_BYTES // per_block))
    CH = min(ncb_max, (M + 127) // 128) * 128                                    # need_cb, ncb_cap, CH
    return CH, xgrad or CH <= 8192                                               # have_vt


def score_plan(n_per_slice, M, d, xgrad, pgrad=False, nsl=1, path=None, unfused=False):
    """The (chunk, slice) passes of an unscreened scoring call: n_per_slice is one n for all nsl slices or a list of
    one n per slice (sample-major, as the call takes them); path / unfused: BOSS_SCORE_PATH / BOSS_UNFUSED_SCORE.
    xgrad: the call computes x-gradients (boss_ei_value_grad); pgrad: boss_gp_predict_grad, which implies xgrad.
    -> dict(CH, have_vt, xgrad, passes=[dict(chunk, m0, ch, slice, nblk, path, nsp, nsp32)])."""
    ns = list(n_per_slice) if np.ndim(n_per_slice) else [int(n_per_slice)] * nsl
    nsl = len(ns)
    CH, have_vt = chunk_capacity(ns, M, d, xgrad, pgrad)
    passes = []
    for c, m0 in enumerate(range(0, M, CH)):                                     # score_core's chunk loop
        ch = min(CH, M - m0)
        ncb, ncb32 = (ch + 127) // 128, (ch + NW_NB - 1) // NW_NB               # score_slice's ncb, ncb32
        for q, n in enumerate(ns):
            nblk = (n + TM - 1) // TM
            nsp, cost_w = pick_row_splits(ncb, nblk)                             # score_slice's nsp
            nsp32, cost_n = pick_row_splits(ncb32, nblk)                         # score_slice's nsp32
            narrow = 0.32 * cost_n < cost_w                                      # score_slice's narrow
            cost_q = max(NQ_COST_CHAIN * nblk, NQ_COST_WORK * ncb32 * (nblk * (nblk + 1) // 2)) + NQ_COST_FIXED
            quarter = have_vt and cost_q < min(cost_w, 0.32 * cost_n if narrow else cost_w) and nblk >= 2   # score_slice's quarter
            if path == "wide":                                                   # score_slice's BOSS_SCORE_PATH switch
                narrow = quarter = False
            elif path == "narrow":
                narrow, quarter = True, False
            elif path == "quarter" and have_vt:
                quarter = True
            if quarter:
                narrow = False
            fuse = nsp == 1 and not narrow and not quarter and q == nsl - 1 and not unfused   # score_slice's fuse
            p = "quarter" if quarter else "narrow" if narrow else "wide_fused" if fuse else "wide_split"
            passes.append(dict(chunk=c, m0=m0, ch=ch, slice=q, nblk=nblk, path=p, nsp=nsp, nsp32=nsp32))
    return dict(CH=CH, have_vt=have_vt, xgrad=xgrad or pgrad, passes=passes)


def plan_counts(plan):
    """What boss_dbg_score_paths reports after the planned call (lib.dbg_score_paths' dict)."""
    out = {p: 0 for p in PATHS}
    for ps in plan["passes"]:
        out[ps["path"]] += 1
    out["xgrad"] = len(plan["passes"]) if plan["xgrad"] else 0
    return out


def chunk_edges(plan, M):
    """The candidates either side of every chunk boundary, and the first and last candidate."""
    out = {0, M - 1}
    for m0 in {ps["m0"] for ps in plan["passes"]}:
        if m0:
            out.update((m0 - 1, m0))
    return sorted(out)

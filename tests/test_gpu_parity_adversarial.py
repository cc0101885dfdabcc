"""Adversarial GPU parity: ill-conditioned kernel matrices, candidates ON training points, tile-boundary sizes.

The ordinary parity suite (tests/test_gpu_parity.py) uses the survey's well-conditioned family (noise 0.1,
l in [0.3, 1.5]).  Here: near-duplicate training points (|dx| 1e-6 .. 1e-3), noise_std in {0, 1e-6, 1e-3},
length-scales in {1e-2, 1, 1e2}, n in {127, 128, 129, 255, 257} (one below / on / above the 128-row tile), d = 1 and 3,
candidates exactly on training points.  Every case is compared with BOTH the restated reference path (oracle/, LAPACK
trsm order) and the x87 extended-precision adjudicator (oracle.adjudicator_longdouble, 64-bit mantissa).

THE COMPARISON RULE (SURVEY.md 7, hard part 1).  sigma^2 = a^2 - |L^-1 k*|^2 cancels catastrophically near training
points; the reference itself (any FP64 evaluation) is only accurate to about cond(K) eps a^2 there.  Separately, the
kernel VALUES are only defined up to the rounding of the scaled squared distance: Distances.jl's GEMM trick
(|a|^2 + |b|^2 - 2 a.b) and the direct form sum (a_i - b_i)^2 both carry an absolute error of a few eps |x~|^2, which for
small length-scales (x~ = x / l large) moves k by dk <= 12 eps a^2 max|x~|^2 (|d kappa / d d^2| <= 1.5 for all three
kernels) - and the posterior amplifies that by |K^-1 k*|_1, |alpha|_1.  So, with kappa = cond_2(K), eps = 2^-52,
a^2 = k(x, x), u = K^-1 k*, alpha = K^-1 (y - m):

    variance   |s2 - s2_ref| <= max(1e-9 |s2_ref|,  4 kappa eps a^2      + 2 |u|_1 (1 + |u|_1) dk)
    mean       |mu - mu_ref| <= max(1e-9 |mu_ref|,  4 kappa eps max|y-m| + |alpha|_1 (1 + |u|_1) dk)
    log-lik    |ll - ll_ref| <= max(1e-8 |ll_ref|,  4 kappa eps |ll_ref| + (sum|K^-1_ij| + |alpha|_1^2) dk / 2)

The first branch is the north star's tolerance; the second is the floor below which no FP64 evaluation order -
including the reference's own - is defined (first term: conditioning of the solve; second: rounding of the distances).
The test applies the rule to CUDA vs the oracle with the GEMM trick (Appendix A.3's guess at the reference), CUDA vs the
oracle with direct differences (what the CUDA kernels compute), CUDA vs the extended-precision truth, and records
oracle vs truth next to them: the CUDA path is as close to the truth as the restated reference is.  Every row also
keeps the fraction of the conditioning-only bound that was used (gpurun_out/parity_adversarial.json ->
profiles/r02_parity_report.json).
When kappa eps >= 1e-3 the matrix is numerically singular: LAPACK may or may not call it positive definite, and the
only requirement is that a failure is reported as BOSS_NOT_POSDEF / a variance below -1e-8 as status 2, never as a
silent wrong number.
"""
import json
import os

import numpy as np
import pytest

from oracle import boss_oracle as O
from tests.posterior_scale_oracle import floors, ratio as _ratio   # the rule, shared with the full-size tests

pytestmark = pytest.mark.gpu

EPS = 2.0 ** -52
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REPORT = os.path.join(ROOT, "gpurun_out", "parity_adversarial.json")
_rows = []


def _problem(n, d, dup_dist, seed):
    rng = np.random.default_rng(seed)
    X = rng.random((d, n))
    ndup = min(8, n // 4)
    if dup_dist is not None:
        delta = rng.standard_normal((d, ndup))
        delta *= dup_dist / np.linalg.norm(delta, axis=0)
        X[:, n - ndup:] = X[:, :ndup] + delta
    y = np.sin(3 * X).sum(0) + 0.05 * rng.standard_normal(n)
    Xs = np.concatenate([rng.random((d, 48)), X[:, :24], X[:, n - ndup:], 0.5 * (X[:, :ndup] + X[:, n - ndup:])], axis=1)
    return X, y, Xs


CASES = []
for _n in (127, 128, 129, 255, 257):
    for _d, _kid, _ell, _noise, _dup in [
        (1, 2, 1.0, 1e-3, 1e-3), (3, 2, 1.0, 1e-3, 1e-6), (3, 1, 1e-2, 0.0, None), (1, 0, 1.0, 1e-3, 1e-4),
        (3, 0, 1e2, 1e-3, None), (3, 2, 1e2, 1e-6, 1e-3), (1, 1, 1e-2, 1e-6, 1e-6), (3, 2, 1.0, 0.0, 1e-3),
    ]:
        CASES.append((_n, _d, _kid, _ell, _noise, _dup))


@pytest.mark.parametrize("n,d,kid,ell,noise,dup", CASES)
def test_adversarial_posterior_and_loglik(lib, n, d, kid, ell, noise, dup):
    X, y, Xs = _problem(n, d, dup, seed=n * 131 + d * 17 + kid)
    ls = np.full(d, ell)
    amp = 1.3
    a2 = (amp + 1e-8) ** 2
    K = O.kernel_matrix(X, None, ls + 1e-8, amp + 1e-8, kid) + (noise + 1e-8) ** 2 * np.eye(n)
    kappa = float(np.linalg.cond(K))
    singular = kappa * EPS >= 1e-3
    row = {"n": n, "d": d, "kernel": kid, "lengthscale": ell, "noise_std": noise, "dup_dist": dup, "cond_K": kappa}

    try:
        post = O.posterior_fit(X, y, ls, amp, noise, kid)
    except O.PosDefException:
        post = None
    gp = lib.gp_fit(X, y, ls, amp, noise, kid)
    if post is None or gp is None:
        # one side rejected the matrix: legitimate only when it is numerically singular
        row["outcome"] = f"not positive definite (oracle: {post is None}, cuda: {gp is None})"
        _rows.append(row)
        assert singular or (post is None) == (gp is None), row
        if gp is not None:
            gp.free()
        return

    mu_o, var_o = O.mean_and_var_raw(post, Xs)
    ll_o = O.gp_loglik(X, y, ls, amp, noise, kid)
    with O.variant(distances="direct"):
        post_d = O.posterior_fit(X, y, ls, amp, noise, kid)
        mu_d, var_d = O.mean_and_var_raw(post_d, Xs)
        ll_d = O.gp_loglik(X, y, ls, amp, noise, kid)
    mu_g, var_g, st_g = lib.gp_predict(gp, Xs)
    ll_g = gp.loglik
    _, st_o = O.clip_var_status(var_o)
    if singular:
        # numerically singular: only the failure semantics are defined
        row["outcome"] = "numerically singular: semantics only"
        assert np.all((st_g == 0) | (st_g == 2))
        assert np.all(np.isfinite(mu_g[st_g == 0]))
        _rows.append(row)
        gp.free()
        return
    # floors of the rule
    Kinv = np.linalg.inv(K)
    alpha = Kinv @ y
    U = Kinv @ O.kernel_matrix(X, Xs, ls + 1e-8, amp + 1e-8, kid)
    u1 = float(np.max(np.sum(np.abs(U), axis=0)))
    x2 = max(float(np.max(np.sum((X / (ls[:, None] + 1e-8)) ** 2, axis=0))),
             float(np.max(np.sum((Xs / (ls[:, None] + 1e-8)) ** 2, axis=0))))
    dk = 12 * EPS * a2 * x2
    c_var, c_mu = 4 * kappa * EPS * a2, 4 * kappa * EPS * float(np.max(np.abs(y)))
    f_mu, f_var = floors(kappa, a2, float(np.max(np.abs(y))), float(np.sum(np.abs(alpha))), u1, x2)
    f_ll_abs = 0.5 * dk * (float(np.sum(np.abs(Kinv))) + float(np.sum(np.abs(alpha))) ** 2)

    def clip(v):   # the [-1e-8, 0) -> 0 branch of _clip_var (status 2 leaves the raw value on both sides)
        return np.where((v < 0) & (v >= -1e-8), 0.0, v)

    def ll_ratio(a, b, with_dist=True):
        return abs(a - b) / max(1e-8 * abs(b), 4 * kappa * EPS * abs(b) + (f_ll_abs if with_dist else 0.0))

    mu_t, var_t, ll_t = O.adjudicator_longdouble(X, y, ls, amp, noise, kid, Xs)
    refs = {"oracle_gemm": (mu_o, clip(var_o), ll_o), "oracle_direct": (mu_d, clip(var_d), ll_d), "truth": (mu_t, clip(var_t), ll_t)}
    for name, (mu_r, var_r, ll_r) in refs.items():
        row[f"var_cuda_vs_{name}"] = _ratio(var_g, var_r, 1e-9, f_var)
        row[f"mean_cuda_vs_{name}"] = _ratio(mu_g, mu_r, 1e-9, f_mu)
        row[f"loglik_cuda_vs_{name}"] = ll_ratio(ll_g, ll_r)
    # informational: the same against the conditioning-only floor, and the restated reference against the truth
    row["var_cuda_vs_truth_cond_floor_only"] = _ratio(var_g, clip(var_t), 1e-9, c_var)
    row["mean_cuda_vs_truth_cond_floor_only"] = _ratio(mu_g, mu_t, 1e-9, c_mu)
    row["info_var_oracle_gemm_vs_truth"] = _ratio(clip(var_o), clip(var_t), 1e-9, f_var)
    row["info_mean_oracle_gemm_vs_truth"] = _ratio(mu_o, mu_t, 1e-9, f_mu)
    row["info_loglik_oracle_gemm_vs_truth"] = ll_ratio(ll_o, ll_t)
    row["min_var_over_a2"] = float(np.min(var_t) / a2)
    row["outcome"] = "compared"
    _rows.append(row)
    for k, v in row.items():
        if "_cuda_vs_" in k and not k.endswith("_only"):
            assert v <= 1.0, (k, row)
    # status agreement wherever the raw variance is clear of the -1e-8 boundary by more than the floor
    clear = np.abs(var_d + 1e-8) > f_var
    _, st_d = O.clip_var_status(var_d)
    assert np.array_equal(st_g[clear], st_d[clear])
    gp.free()


def test_candidates_on_training_points_interpolate(lib):
    """The reference's own property test (test/unit/test/models/gaussian_process.jl:94-96: mean(x_i) ~ y_i, atol 0.01)
    at tight noise, plus the exact statement: at a training point the posterior variance is s^2 (1 - s^2 [K^-1]_ii)."""
    rng = np.random.default_rng(7)
    n, d = 200, 2
    X = rng.random((d, n)); y = np.sin(3 * X).sum(0)
    ls, amp, noise = np.array([0.4, 0.6]), 1.0, 1e-3
    gp = lib.gp_fit(X, y, ls, amp, noise, 2)
    mu, var, st = lib.gp_predict(gp, X)
    assert np.all(st == 0)
    assert np.max(np.abs(mu - y)) < 0.01
    K = O.kernel_matrix(X, None, ls + 1e-8, amp + 1e-8, 2) + (noise + 1e-8) ** 2 * np.eye(n)
    kappa = np.linalg.cond(K)
    s2 = (noise + 1e-8) ** 2
    exact = s2 * (1.0 - s2 * np.diag(np.linalg.inv(K).astype(np.longdouble)).astype(np.float64))
    assert np.max(np.abs(var - exact)) <= max(1e-9 * np.max(exact), 4 * kappa * EPS * (amp + 1e-8) ** 2)
    gp.free()


def test_zz_write_report():
    """Last in the file: dump the per-case ratios (fraction of the rule's bound that was used)."""
    os.makedirs(os.path.dirname(REPORT), exist_ok=True)
    compared = [r for r in _rows if r.get("outcome") == "compared"]
    keys = [k for k in (compared[0] if compared else {}) if "_vs_" in k]
    summary = {k: max(r[k] for r in compared) for k in keys}
    with open(REPORT, "w") as f:
        json.dump({"rule": "see tests/test_gpu_parity_adversarial.py docstring; values are |diff| / bound (<= 1 passes)",
                   "cases": len(_rows), "compared": len(compared), "max_fraction_of_bound": summary, "rows": _rows}, f, indent=1)
    assert len(_rows) == 0 or len(compared) >= len(_rows) // 3

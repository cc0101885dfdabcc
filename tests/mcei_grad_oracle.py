"""numpy reference of the x-gradient of the Monte-Carlo EI (DESIGN.md 2.11, include/boss_b200.h boss_mcei_value_grad),
built on the oracle's mean_var_grad.  Plain vectorised numpy, no device code: the CPU tests check it against central
differences of O.mc_ei_acquisition, the GPU tests check the device against it."""
import numpy as np

from oracle import boss_oracle as O


def _coefs(y_dim, c, q, t):
    z = np.zeros(y_dim)
    return (z.copy() if c is None else np.asarray(c, dtype=np.float64),
            z.copy() if q is None else np.asarray(q, dtype=np.float64),
            z.copy() if t is None else np.asarray(t, dtype=np.float64))


def fitness(kind, c0, c, q, t):
    """The expression of fit_kind as a closure of one y_dim vector (what O.mc_ei_acquisition takes)."""
    c, q, t = (np.asarray(v, dtype=np.float64) for v in _coefs(len(c), c, q, t))

    def f(y):
        y = np.asarray(y, dtype=np.float64)
        if kind == 1:
            return c0 + float(c @ y)
        if kind == 2:
            return c0 + float(c @ y) + float(np.sum(q * (y - t) ** 2))
        v = (c * y + t)[c != 0]
        return c0 + float(v.max() if kind == 3 else v.min())
    return f


def _fit_and_grad(kind, c0, c, q, t, Y):
    """f(Y) and df/dy for Y (y_dim, ...): the branch the device's value takes (max / min: the first extreme output)."""
    if kind == 1:
        f = c0 + np.tensordot(c, Y, axes=1)
        G = np.broadcast_to(c.reshape((-1,) + (1,) * (Y.ndim - 1)), Y.shape).copy()
        return f, G
    shp = (-1,) + (1,) * (Y.ndim - 1)
    if kind == 2:
        dv = Y - t.reshape(shp)
        f = c0 + np.tensordot(c, Y, axes=1) + np.tensordot(q, dv * dv, axes=1)
        return f, c.reshape(shp) + 2.0 * q.reshape(shp) * dv
    live = np.flatnonzero(c != 0)
    V = (c.reshape(shp) * Y + t.reshape(shp))[live]
    pick = np.argmax(V, axis=0) if kind == 3 else np.argmin(V, axis=0)     # first extreme in index order
    f = c0 + np.take_along_axis(V, pick[None], axis=0)[0]
    G = np.zeros_like(Y)
    for a, i in enumerate(live):
        G[i] = np.where(pick == a, c[i], 0.0)
    return f, G


def kink_margin(posts_per_sample, Xs, kind, c0, c, q, t, eps, best, prior_mean_s=None):
    """Per candidate, the smallest |imp_k| and (max / min) the smallest gap between the extreme term and the next one
    over every eps column the candidate uses: how close it is to a point where the MC-EI is not differentiable."""
    Xs = np.asarray(Xs, dtype=np.float64)
    S, y_dim, M = len(posts_per_sample), len(posts_per_sample[0]), Xs.shape[1]
    c, q, t = _coefs(y_dim, c, q, t)
    eps = np.asarray(eps, dtype=np.float64).reshape(y_dim, -1)
    out = np.full(M, np.inf)
    for s in range(S):
        mu = np.empty((y_dim, M)); var = np.empty((y_dim, M))
        for i in range(y_dim):
            pm = None if prior_mean_s is None else np.asarray(prior_mean_s)[i]
            mu[i], var[i], _ = O.mean_and_var(posts_per_sample[s][i], Xs, pm)
        e = eps if S == 1 else eps[:, s:s + 1]
        Y = mu[:, :, None] + np.sqrt(var)[:, :, None] * e[:, None, :]
        f, _ = _fit_and_grad(kind, c0, c, q, t, Y)
        out = np.minimum(out, np.min(np.abs(f - best), axis=1))
        if kind in (3, 4) and np.count_nonzero(c) > 1:
            live = np.flatnonzero(c != 0)
            V = np.sort((c[:, None, None] * Y + t[:, None, None])[live], axis=0)
            gap = V[-1] - V[-2] if kind == 3 else V[1] - V[0]
            out = np.minimum(out, np.min(gap, axis=1))
    return out


def mc_ei_value_grad(posts_per_sample, Xs, fitness_kind, c0, c, q, t, eps, best, y_max, prior_mean_s=None,
                     prior_mean_grad_s=None):
    """Value and x-gradient of the MC-EI (x PoF) for in-domain points.  posts_per_sample[s][i] = posterior of BI sample
    s, output i; eps (y_dim, K): one posterior uses every column, S > 1 posteriors take column s each.

      y_k = mu + sd .* eps_k,  imp_k = f(y_k) - best,  EI_s = 1/|K_s| sum_k max(0, imp_k)
      d EI_s = sum_i A_i d mu_i + B_i d sd_i,  A_i = 1/|K_s| sum_{imp_k > 0} g_i(y_k),  B_i = ... g_i(y_k) eps_ik
      d sd_i = d var_i / (2 sd_i) when sd_i > 0 (mean_var_grad already zeroes d var where the variance was clipped)

    Returns val (M,) (-inf where a variance failed), grad (d, M)."""
    Xs = np.asarray(Xs, dtype=np.float64)
    d, M = Xs.shape
    S, y_dim = len(posts_per_sample), len(posts_per_sample[0])
    c, q, t = _coefs(y_dim, c, q, t)
    eps = np.asarray(eps, dtype=np.float64).reshape(y_dim, -1)
    acc = np.zeros(M)
    gacc = np.zeros((d, M))
    failed = np.zeros(M, dtype=bool)
    for s in range(S):
        posts = posts_per_sample[s]
        pm = [None if prior_mean_s is None else np.asarray(prior_mean_s)[i] for i in range(y_dim)]
        pmg = [None if prior_mean_grad_s is None else np.asarray(prior_mean_grad_s)[i] for i in range(y_dim)]
        mus = np.empty((y_dim, M)); vs = np.empty((y_dim, M))
        dmus = np.empty((y_dim, d, M)); dvs = np.empty((y_dim, d, M))
        for i in range(y_dim):
            mus[i], vs[i], dmus[i], dvs[i], st = O.mean_var_grad(posts[i], Xs, pm[i], pmg[i])
            failed |= st != 0
        if best is None and y_max is None:
            continue
        if y_max is not None:                      # PoF and its gradient: the closed-form oracle with best = None
            pof, dpof = O.ei_value_grad(posts, Xs, np.ones(y_dim), None, y_max, prior_mean_s=prior_mean_s,
                                        prior_mean_grad_s=prior_mean_grad_s)
        if best is None:
            acc += pof
            gacc += dpof
            continue
        sd = np.sqrt(vs)
        with np.errstate(divide="ignore", invalid="ignore"):
            dsd = np.where(sd[:, None, :] > 0, dvs / (2.0 * sd[:, None, :]), 0.0)
        e = eps if S == 1 else eps[:, s:s + 1]
        K = e.shape[1]
        Y = mus[:, :, None] + sd[:, :, None] * e[:, None, :]              # y_dim x M x K
        f, G = _fit_and_grad(fitness_kind, c0, c, q, t, Y)
        imp = f - best                                                     # M x K
        pos = imp > 0.0
        ei = np.where(pos, imp, 0.0).sum(axis=1) / K
        A = (G * pos[None]).sum(axis=2) / K                                # y_dim x M
        B = (G * pos[None] * e[:, None, :]).sum(axis=2) / K
        nan = np.isnan(imp).any(axis=1)
        ei = np.where(nan, np.nan, ei)
        A = np.where(nan[None], np.nan, A)
        dei = np.einsum("im,idm->dm", A, dmus) + np.einsum("im,idm->dm", B, dsd)
        if y_max is None:
            acc += ei
            gacc += dei
        else:
            acc += ei * pof
            gacc += dei * pof + ei * dpof
    val = np.where(failed, -np.inf, acc / S)
    grad = np.where(failed[None], 0.0, gacc / S)
    return val, grad

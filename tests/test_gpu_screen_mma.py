"""The tensor-core distances of the FP32 mean tier (DESIGN.md 2.9).

- The MMA's d2 = |u|^2 + |t|^2 - 2 u.t stays within the error model the bound E rests on, over adversarial magnitudes,
  for the 8-, 16- and 32-wide k-steps of every padded input dimension.
- On the bench problem: max |mu~ - mu64| / E (DESIGN.md 2.9 lists it beside the SIMT kernel's), the ambiguous count
  and the re-seeded pool, and the screened pair equal to the unscreened one.
"""
import numpy as np
import pytest

from tests.util_problems import make_problem

pytestmark = pytest.mark.gpu

EPS = 2.0**-24


def _kp(dp):
    return 8 * ((dp + 7) // 8) if dp <= 16 else 32


def _model(u, t, kp):
    """The per-pair bound of DESIGN.md 2.9 for FP32 inputs and norms rounded to FP32 once: the TF32 split
    (3 * 2^-22 per product), the MMA chain (3 kp / 8 mma of <= 10 * 2^-23 * the largest addend each), the assembly
    (two FP32 additions) and the rounding of the norms.  eps ((29 + 15 kp) |u| |t| + 3 (|u|^2 + |t|^2))."""
    nu = np.sum(u.astype(np.float64) ** 2, axis=1)
    nt = np.sum(t.astype(np.float64) ** 2, axis=1)
    P = np.sqrt(nu)[:, None] * np.sqrt(nt)[None, :]
    S = nu[:, None] + nt[None, :]
    return EPS * ((29 + 15 * kp) * P + 3 * S), S


def _cases(rng, m, n, kp, dp):
    def pad(a):
        out = np.zeros((a.shape[0], kp), np.float32)
        out[:, :dp] = a
        return out
    g = lambda r, c: rng.standard_normal((r, c))   # noqa: E731
    mag = 10.0 ** rng.uniform(-3, 3, dp)
    yield "normal", pad(g(m, dp)), pad(g(n, dp))
    yield "per-dim magnitudes 1e-3..1e3", pad(g(m, dp) * mag), pad(g(n, dp) * mag)
    u = g(m, dp) * 300.0
    t = u[rng.integers(0, m, n)] * (1 + 1e-6 * g(n, dp)) + 1e-3 * g(n, dp)
    yield "near-cancellation, |u| ~ 1e3", pad(u), pad(t)
    # every value a TF32 rounding tie (bit 12 set, bits 0-11 clear) or one bit below / above it
    b = (rng.integers(0x3F000000, 0x41000000, (m + n, dp)) & ~0x1FFF) | 0x1000
    b = b + rng.integers(-1, 2, b.shape)
    v = b.astype(np.uint32).view(np.float32) * np.where(rng.random(b.shape) < 0.5, -1.0, 1.0).astype(np.float32)
    yield "TF32 ties", pad(v[:m]), pad(v[m:])
    yield "one large coordinate", pad(g(m, dp) * np.r_[1e4, np.ones(dp - 1)]), pad(g(n, dp))


@pytest.mark.parametrize("dp", [2, 4, 6, 8, 12, 16, 32])
def test_mma_d2_within_model(lib, dp):
    rng = np.random.default_rng(dp)
    kp, m, n = _kp(dp), 16 * 32, 8 * 64
    worst = 0.0
    for name, u, t in _cases(rng, m, n, kp, dp):
        u32, t32 = u.astype(np.float32), t.astype(np.float32)
        nu = np.sum(u32.astype(np.float64) ** 2, axis=1)
        nt = np.sum(t32.astype(np.float64) ** 2, axis=1)
        got = lib.dbg_mma_d2(dp, u32, t32, nu.astype(np.float32), nt.astype(np.float32)).astype(np.float64)
        ref = np.sum((u32.astype(np.float64)[:, None, :] - t32.astype(np.float64)[None, :, :]) ** 2, axis=2)
        bound, S = _model(u32, t32, kp)
        err = np.abs(got - ref)
        ratio = float(np.max(err / bound))
        k_seen = float(np.max(err / (EPS * S)))
        worst = max(worst, ratio)
        print(f"dp {dp} {name}: max err / model {ratio:.3e}, max err / (2^-24 (|u|^2 + |t|^2)) {k_seen:.2f}")
        assert ratio <= 1.0, (name, ratio)
    print(f"dp {dp}: worst err / model {worst:.3e}")


def test_bench_problem_band_and_pool(lib, monkeypatch):
    X, Y, ls, amp, ns = make_problem(2048, 8, seed=1002)
    gp = lib.gp_fit(X, Y[0], ls[0], amp[0], ns[0], lib.KERNEL_MATERN52)
    mu32, E, mu64 = lib.dbg_screen_mean(gp, np.random.default_rng(7).random((8, 65_536)))
    ratio = float(np.max(np.abs(mu32 - mu64) / E))
    print(f"bench problem: max |mu~ - mu64| / E = {ratio:.3e}, median E = {np.median(E):.3e}")
    assert ratio <= 1.0
    import torch
    for k in ("BOSS_NO_SCREEN", "BOSS_SCREEN_F64", "BOSS_SCREEN_NO_RESEED"):
        monkeypatch.delenv(k, raising=False)
    M = 1 << 21
    gen = torch.Generator(device="cuda")
    gen.manual_seed(2002)
    Xs = torch.rand((M, 8), dtype=torch.float64, device="cuda", generator=gen)   # bench.py's candidates
    torch.cuda.synchronize()
    best = float(np.max(Y[0]))
    r = lib.ei_score_dev([gp], 1, 1, Xs.data_ptr(), M, [1.0], best, None)
    st, amb = lib.dbg_screen_stats(), lib.dbg_screen_ambiguous()
    print(f"bench call: ambiguous {amb[0]}, pool before re-seed {amb[1]}, after re-seed {st[2]}")
    assert st[0] == 1 and st[2] >= 1
    monkeypatch.setenv("BOSS_NO_SCREEN", "1")
    ref = lib.ei_score_dev([gp], 1, 1, Xs.data_ptr(), M, [1.0], best, None)
    assert (np.float64(r[0]).view(np.int64), r[1]) == (np.float64(ref[0]).view(np.int64), ref[1])
    gp.free()

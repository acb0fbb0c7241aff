"""The chain layout of the fixed-point register kernel (ssf_kernel<int32_t, int32_t, NPL, false, false>; csrc/ssf.cu,
ssf_run_device): up to 28 chains per CTA and no producer warp, so that up to 148 x 28 replicas run in one wave, and one
chain per CTA when R <= 148.  At each layout boundary the kernel, forced with ISB_SSF_MODE=1, must equal the oracle and
the cold kernel (ISB_SSF_MODE=0) bit for bit: spins, flip counts and exact-fallback counts, and the cached fields it
leaves behind (a second run continues on them and must equal the same run on fields rebuilt from the spins)."""
import numpy as np
import pytest

from cases import commensurate_J

pytestmark = pytest.mark.gpu
SMS, CHAINS = 148, 28
# 4096: C2, one wave of 28 chains per CTA (147 CTAs); 148 x 28 + 1: the first R that takes a second wave; 149: just above
# one chain per SM; 5: one chain per CTA
RS = [4096, SMS * CHAINS + 1, SMS + 1, 5]
SEED = 515


def _layout(R):
    """(chains per CTA, CTAs) as the launcher picks them for the fixed-point kernel."""
    if R <= SMS:
        return 1, R
    waves = -(-R // (SMS * CHAINS))
    nw = -(-R // (SMS * waves))
    return nw, -(-R // nw)


def _samples(R):
    """First replicas of the first two CTAs, the last chain of the first CTA, the middle, the first chain of the last
    CTA and the last replica."""
    nw, ctas = _layout(R)
    return sorted({r for r in (0, nw - 1, nw, R // 2, (ctas - 1) * nw, R - 1) if 0 <= r < R})


def _model(synth, kind, N):
    """(J, h, rule, T) of one coupling set."""
    if kind == "continuum":      # SK couplings: Glauber at a temperature where about a fifth of the attempts flip
        return synth.sk_J(N, SEED + N), synth.gaussian(SEED + 1, N) * 0.3, 1, 0.8
    if kind == "ties":           # +-0.1 / +-0.3, h = 0, T = 0: exact ties recur, and each one falls back
        return commensurate_J(synth, N, SEED + 2 + N), np.zeros(N), 1, 0.0
    g = synth.gaussian(SEED + 4 + N, N * N).reshape(N, N)   # integers and a dyadic h: nothing falls back
    J = np.triu(np.where(g > 0.5, 1.0, np.where(g < -0.5, -1.0, 0.0)), 1)
    return J + J.T, np.where(synth.gaussian(SEED + 5, N) > 0, 0.5, -0.5), 2, 1.5


@pytest.mark.parametrize("kind", ["continuum", "ties", "integer"])
@pytest.mark.parametrize("N", [1024, 256])
@pytest.mark.parametrize("R", RS)
def test_fixed_register_kernel_layouts(ctx, orc, synth, monkeypatch, R, N, kind):
    from isingmodel_jl_b200 import _lib as L
    J, h, rule, T = _model(synth, kind, N)
    S0 = synth.spins(SEED + 6 + N, R, N)
    start, n1, n2 = 19, 2 * N + N // 3 + 5, N + 45            # ragged: both runs start and end inside a 32-site window
    Ta = np.array([T])
    e = L.Ensemble(L.Model.dense(ctx, J, h, L.PREC_F64), R)

    def second(mode, S=None):
        monkeypatch.setenv("ISB_SSF_MODE", str(mode))
        if S is not None:
            e.set_spins(S)                                      # drops the cached fields: rebuilt from S
        out = e.ssf_run(rule, n2, start=(start + n1) % N, seed=SEED, step_offset=n1, T=Ta, steps_per_T=n2)
        return e.get_spins(), out["flips"], e.last_stats()["exact_fallbacks"]

    def two_runs(mode):
        monkeypatch.setenv("ISB_SSF_MODE", str(mode))
        e.set_spins(S0)
        out = e.ssf_run(rule, n1, start=start, seed=SEED, T=Ta, steps_per_T=n1)
        first = e.get_spins(), out["flips"], e.last_stats()["exact_fallbacks"]
        return first, second(mode)                              # the second run continues on the cached fields

    runs = {"plain": two_runs(1), "cold": two_runs(0)}
    (S1, f1, fb1), (S2, f2, fb2) = runs["plain"]
    for part, (S, f, fb) in enumerate(runs["cold"]):
        ref = runs["plain"][part]
        assert np.array_equal(S, ref[0]), f"run {part + 1}: spins differ between the plain and the cold kernel"
        assert np.array_equal(f, ref[1]), f"run {part + 1}: flip counts differ between the plain and the cold kernel"
        assert fb == ref[2], f"run {part + 1}: {fb} exact fallbacks on the cold kernel, {ref[2]} on the plain one"
    rebuilt = second(1, S1)
    assert np.array_equal(rebuilt[0], S2) and np.array_equal(rebuilt[1], f2) and rebuilt[2] == fb2, \
        "the run on the plain kernel's cached fields differs from the run on fields rebuilt from its spins"
    assert f1.sum() > 0 and f2.sum() > 0
    if kind == "ties":
        assert fb1 + fb2 > 0
    elif kind == "integer":
        assert fb1 + fb2 == 0
    for r in _samples(R):
        fl = ctx.philox_fluct(rule, SEED, 0, r, 1, n1 + n2)[0]
        s, nf, _, _ = orc.ssf_run(rule, J, h, S0[r], n1, start=start, fluct=fl[:n1], T=Ta, steps_per_T=n1)
        assert np.array_equal(s, S1[r]) and nf == f1[r], f"replica {r}: first run differs from the oracle"
        s, nf, _, _ = orc.ssf_run(rule, J, h, s, n2, start=(start + n1) % N, fluct=fl[n1:], T=Ta, steps_per_T=n2)
        assert np.array_equal(s, S2[r]) and nf == f2[r], f"replica {r}: second run differs from the oracle"


def test_fixed_segmented_anneal_alternating_kernels_equals_one_launch(ctx, synth, monkeypatch):
    """C2's size (SK N = 1024, 4096 replicas).  Four sweeps at T = 3 and four at T = 0.05, three times over, cut into
    segments of two sweeps: each segment's kernel follows the previous segment's acceptance (above 10 %: plain, below:
    cold), so the run alternates between the plain and the cold kernel.  Every replica must equal one launch of either."""
    from isingmodel_jl_b200 import _lib as L
    N, R = 1024, 4096
    J, h = synth.sk_J(N, SEED + 7), np.zeros(N)
    S0 = synth.spins(SEED + 8, R, N)
    T = np.array([3.0] * 4 + [0.05] * 4 + [3.0] * 4 + [0.05] * 4 + [3.0] * 4 + [0.05] * 4)
    nsteps = T.size * N
    e = L.Ensemble(L.Model.dense(ctx, J, h, L.PREC_F64), R)

    def run(env):
        for k in ("ISB_SSF_MODE", "ISB_SSF_SEG_MIN", "ISB_SSF_COLD_THR"):
            monkeypatch.delenv(k, raising=False)
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        e.set_spins(S0)
        out = e.ssf_run(L.RULE_GLAUBER, nsteps, seed=SEED, T=T, steps_per_T=N)
        return e.get_spins(), out["flips"], e.last_stats()

    seg = run({"ISB_SSF_SEG_MIN": str(2 * N), "ISB_SSF_COLD_THR": "0.1"})
    assert seg[2]["launches"] >= T.size // 2                  # one launch per segment (plus the field initialisation)
    for mode in ("1", "0"):
        one = run({"ISB_SSF_MODE": mode})
        assert one[2]["launches"] <= 2
        assert np.array_equal(seg[0], one[0]), f"spins differ from one launch with ISB_SSF_MODE={mode}"
        assert np.array_equal(seg[1], one[1]), f"flip counts differ from one launch with ISB_SSF_MODE={mode}"
        assert seg[2]["exact_fallbacks"] == one[2]["exact_fallbacks"]

"""GPU tests of the fixed-point dense sweep kernels (DESIGN §3): int32 couplings and cached fields, integer decision
thresholds, and the reference's fresh Float64 row dot for every decision the thresholds cannot settle.  Untraced
sequential runs of Float64 dense models take this path by default; every decision must equal the oracle's (spins and flip
counts bit for bit), whatever kernel (plain or cold) runs each segment."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _lib():
    from isingmodel_jl_b200 import _lib
    return _lib


def _oracle_check(orc, J, h, S0, S, flips, rule, nsteps, fl, per_rep, T, N, replicas, start=0, tscale=None):
    for r in replicas:
        Tr = T if tscale is None else T * tscale[r]
        f = None if fl is None else (fl[r] if per_rep else fl)
        s, nf, _, _ = orc.ssf_run(rule, J, h, S0[r], nsteps, start=start, fluct=f, T=Tr, steps_per_T=N)
        assert np.array_equal(s, S[r]) and nf == flips[r], f"replica {r}"


@pytest.mark.parametrize("mode", ["plain", "cold", "mixed"])
@pytest.mark.parametrize("N", [96, 500, 1024])
@pytest.mark.parametrize("rule", [0, 1, 2])
def test_fixed_point_equals_oracle(ctx, orc, synth, monkeypatch, rule, N, mode):
    """h != 0, per-replica temperature factors, ragged runs; the plain kernel, the cold kernel, or both alternating by
    segment.  Sampled replicas equal the oracle, and every replica equals the Float64 kernels' run."""
    L = _lib()
    R, sweeps = 40, 9
    nsteps = sweeps * N + 37                                      # ragged: the run ends inside a 32-site window
    J, h = synth.sk_J(N, 101 + N), synth.gaussian(102, N) * 0.3
    S0 = synth.spins(103, R, N)
    per_rep = rule == 1
    gen = synth.logistic if rule == 1 else synth.exponential
    fl = None if rule == 0 else gen(104, (R, nsteps) if per_rep else nsteps)
    T = synth.geometric_schedule(3.0, 0.05, sweeps + 1)
    tscale = None if rule == 0 else 0.5 + synth.gaussian(105, R) ** 2
    if mode == "mixed":                                           # short segments: plain and cold launches alternate
        monkeypatch.setenv("ISB_SSF_SEG_MIN", str(N + 13))
        monkeypatch.setenv("ISB_SSF_SEG_THR", "0.15")
        monkeypatch.setenv("ISB_SSF_COLD_THR", "0.05")
    else:
        monkeypatch.setenv("ISB_SSF_MODE", {"plain": "1", "cold": "0"}[mode])
    e = L.Ensemble(L.Model.dense(ctx, J, h, L.PREC_F64), R)
    e.set_spins(S0)
    if tscale is not None:
        e.set_temperature_scale(tscale)
    out = e.ssf_run(rule, nsteps, start=3, fluct=fl, fluct_per_replica=per_rep, T=T, steps_per_T=N)
    S = e.get_spins()
    _oracle_check(orc, J, h, S0, S, out["flips"], rule, nsteps, fl, per_rep, T, N, (0, 1, R // 2, R - 1), start=3,
                  tscale=tscale)
    # the Float64 kernels reach the same state
    monkeypatch.setenv("ISB_SSF_FIXED", "0")
    e.set_spins(S0)
    out64 = e.ssf_run(rule, nsteps, start=3, fluct=fl, fluct_per_replica=per_rep, T=T, steps_per_T=N)
    assert np.array_equal(e.get_spins(), S) and np.array_equal(out64["flips"], out["flips"])
    assert e.last_stats()["exact_fallbacks"] == 0


def test_fixed_point_continuation_and_traced_runs(ctx, orc, synth):
    """Untraced (fixed-point) and traced (Float64) runs alternate on one ensemble: each path rebuilds its own field cache
    when the other one ran, and the chain continues as one run of the reference."""
    L = _lib()
    N, R, n1, n2, n3 = 200, 16, 2100, 1300, 1700
    nt = n1 + n2 + n3
    J, h = synth.sk_J(N, 111), synth.gaussian(112, N) * 0.2
    S0 = synth.spins(113, R, N)
    fl = synth.logistic(114, (R, nt))
    T = synth.geometric_schedule(2.0, 0.2, nt)                  # one temperature per step
    e = L.Ensemble(L.Model.dense(ctx, J, h, L.PREC_F64), R)
    e.set_spins(S0)
    e.ssf_run(1, n1, fluct=fl[:, :n1].copy(), fluct_per_replica=True, T=T[:n1])
    out = e.ssf_run(1, n2, start=n1 % N, fluct=fl[:, n1:n1 + n2].copy(), fluct_per_replica=True, T=T[n1:n1 + n2],
                    trace_every=100)
    S_mid = e.get_spins()
    e.ssf_run(1, n3, start=(n1 + n2) % N, fluct=fl[:, n1 + n2:].copy(), fluct_per_replica=True, T=T[n1 + n2:])
    S_end = e.get_spins()
    for r in (0, 7, R - 1):
        s, _, E, _ = orc.ssf_run(1, J, h, S0[r], n1 + n2, fluct=fl[r, :n1 + n2], T=T)
        assert np.array_equal(s, S_mid[r])
        s, *_ = orc.ssf_run(1, J, h, S0[r], nt, fluct=fl[r], T=T)
        assert np.array_equal(s, S_end[r])
    assert out["E"] is not None and out["E"].shape == (n2 // 100, R)
    e.set_spins(S0)                                               # drops both caches
    e.ssf_run(1, 300, fluct=fl[:, :300].copy(), fluct_per_replica=True, T=T[:300])
    S = e.get_spins()
    for r in (0, R - 1):
        s, *_ = orc.ssf_run(1, J, h, S0[r], 300, fluct=fl[r, :300], T=T)
        assert np.array_equal(s, S[r])


@pytest.mark.parametrize("hmag", [0.05, 0.0])
def test_fixed_point_commensurate_couplings_at_zero_temperature(ctx, orc, synth, hmag):
    """Couplings +-0.1 / +-0.3 at T = 0 without the tie audit: exact ties and one-ulp cancellations of the reference
    again and again (h = 0).  Every one of them lies in the fallback band and is decided on the reference's row dot;
    |h| = 0.05 keeps every field at least 0.05 away from zero, and nothing needs to fall back."""
    L = _lib()
    n, R, sweeps, per = 96, 12, 300, 75
    g = synth.gaussian(91, n * n).reshape(n, n)
    J = np.where(g > 0.8, 0.3, np.where(g > 0.0, 0.1, np.where(g > -0.8, -0.1, -0.3)))
    J = np.where(np.abs(synth.gaussian(92, n * n).reshape(n, n)) < 0.25, J, 0.0)
    J = np.triu(J, 1)
    J = J + J.T
    h = np.where(synth.gaussian(93, n) > 0, hmag, -hmag)
    S0 = synth.spins(94, R, n)
    e = L.Ensemble(L.Model.dense(ctx, J, h, L.PREC_F64), R)
    e.set_spins(S0)
    fallbacks = 0
    for c in range(sweeps // per):
        e.ssf_run(L.RULE_GLAUBER, per * n, fluct=np.zeros(per * n), T=np.zeros(1), steps_per_T=per * n)
        fallbacks += e.last_stats()["exact_fallbacks"]
    S = e.get_spins()
    for r in range(R):
        s, *_ = orc.ssf_run(orc.GLAUBER, J, h, S0[r], sweeps * n, fluct=np.zeros(sweeps * n), T=np.zeros(1),
                            steps_per_T=sweeps * n)
        assert np.array_equal(s, S[r]), f"replica {r}"
    assert (fallbacks > 0) == (hmag == 0.0)


@pytest.mark.parametrize("rule", [0, 1, 2])
def test_fixed_point_integer_couplings_never_fall_back(ctx, orc, synth, rule):
    """Couplings that are exact multiples of the quantum (integers, h on a dyadic grid): the thresholds are exact, nothing
    falls back, and the zero-field ties of Hopfield dynamics resolve as the reference's heaviside(0) = 1."""
    L = _lib()
    N, R, sweeps = 128, 24, 20
    g = synth.gaussian(121, N * N).reshape(N, N)
    J = np.triu(np.where(g > 0.5, 1.0, np.where(g < -0.5, -1.0, 0.0)), 1)
    J = J + J.T
    h = np.where(synth.gaussian(122, N) > 0, 0.5, -0.5) * (rule != 0)
    S0 = synth.spins(123, R, N)
    nsteps = sweeps * N
    fl = None if rule == 0 else synth.logistic(124, nsteps)
    T = synth.geometric_schedule(4.0, 0.1, sweeps)
    e = L.Ensemble(L.Model.dense(ctx, J, h, L.PREC_F64), R)
    e.set_spins(S0)
    out = e.ssf_run(rule, nsteps, fluct=fl, T=T, steps_per_T=N)
    assert e.last_stats()["exact_fallbacks"] == 0
    _oracle_check(orc, J, h, S0, e.get_spins(), out["flips"], rule, nsteps, fl, False, T, N, range(R))


def test_fixed_point_refused_for_a_huge_dynamic_range(ctx, orc, synth):
    """One coupling 10^4 times the others sets the quantum; the other rows would sit in a fallback band wider than 2^-20
    of their field scale, so the model keeps the Float64 kernels (no decision is counted as a fallback)."""
    L = _lib()
    N, R, sweeps = 96, 12, 50
    J = synth.sk_J(N, 131)
    J[3, 70] = J[70, 3] = 1e4
    h = synth.gaussian(132, N) * 0.1
    S0 = synth.spins(133, R, N)
    nsteps = sweeps * N
    fl = synth.logistic(134, (R, nsteps))
    T = synth.geometric_schedule(3.0, 0.1, sweeps)
    e = L.Ensemble(L.Model.dense(ctx, J, h, L.PREC_F64), R)
    e.set_spins(S0)
    out = e.ssf_run(1, nsteps, fluct=fl, fluct_per_replica=True, T=T, steps_per_T=N)
    assert e.last_stats()["exact_fallbacks"] == 0
    _oracle_check(orc, J, h, S0, e.get_spins(), out["flips"], 1, nsteps, fl, True, T, N, range(R))


def test_fixed_point_full_size(ctx, orc, synth, monkeypatch):
    """The benchmark's model and ensemble size (SK N = 1024, 4096 replicas, Philox noise): 24 untraced sweeps equal the
    Float64 kernels for every replica and the oracle on sampled ones."""
    L = _lib()
    N, R, sweeps = 1024, 4096, 24
    nsteps = sweeps * N
    J, h = synth.sk_J(N, 1234), np.zeros(N)
    S0 = synth.spins(1235, R, N)
    T = synth.geometric_schedule(3.0, 0.05, sweeps)
    e = L.Ensemble(L.Model.dense(ctx, J, h, L.PREC_F64), R)
    e.set_spins(S0)
    out = e.ssf_run(L.RULE_GLAUBER, nsteps, seed=77, T=T, steps_per_T=N)
    S, fb = e.get_spins(), e.last_stats()["exact_fallbacks"]
    monkeypatch.setenv("ISB_SSF_FIXED", "0")
    e.set_spins(S0)
    out64 = e.ssf_run(L.RULE_GLAUBER, nsteps, seed=77, T=T, steps_per_T=N)
    assert np.array_equal(e.get_spins(), S) and np.array_equal(out64["flips"], out["flips"])
    print(f"\n[C2 size, {sweeps} sweeps] {fb} exact fallbacks")
    for r in (0, R - 1):
        fl = ctx.philox_fluct(L.RULE_GLAUBER, 77, 0, r, 1, nsteps)[0]
        s, nf, _, _ = orc.ssf_run(orc.GLAUBER, J, h, S0[r], nsteps, fluct=fl, T=T, steps_per_T=N)
        assert np.array_equal(s, S[r]) and nf == out["flips"][r], f"replica {r}"

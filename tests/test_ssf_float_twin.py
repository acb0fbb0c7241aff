"""CPU checks of the cached-field twin (tests/ssf_float_twin.py), the reference of the Float32 dense sweeps: where the
cached fields are exact it must reproduce the C oracle bit for bit, and where they are not it must leave it."""
import numpy as np
import pytest

from cases import GUARD_PER, GUARD_SWEEPS, guard_case
from ssf_float_twin import FieldTwin


def _integer_model(synth, n, seed, scale):
    g = synth.gaussian(seed, n * n).reshape(n, n)
    J = np.triu(np.round(g * 1.5) * scale, 1)
    h = np.round(synth.gaussian(seed + 1, n) * 2.0) * 0.25
    return J + J.T, h


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("rule", [0, 1, 2])
@pytest.mark.parametrize("order", ["seq", "list"])
def test_twin_equals_the_oracle_on_exact_couplings(orc, synth, dtype, rule, order):
    """Integer couplings (x 1/8 for Float64 storage: dyadic) and h on a 1/4 grid: every field sum is exact in the storage
    type, so the cached fields are the reference's fresh row dots and the dynamics are the reference's.  Per-replica
    temperature factors, a schedule that changes inside 32-site windows, a start inside a window, shared and per-replica
    noise, traces, and a second run that continues from the cached fields."""
    n, R = 45, 5
    J, h = _integer_model(synth, n, 7 + rule, 0.125 if dtype == np.float64 else 1.0)
    S0 = synth.spins(9, R, n)
    spT, tr = 19, 23                                            # neither is a multiple of 32
    n1, n2 = 17 * spT, 3 * n + 4                                # the second run starts at a schedule boundary
    nsteps = n1 + n2
    nodes = synth.nodes(10, n, nsteps) if order == "list" else None
    per_rep = rule == 1
    gen = synth.logistic if rule == 1 else synth.exponential
    fl = gen(11, (R, nsteps) if per_rep else nsteps) * 3.0
    T = synth.geometric_schedule(4.0, 0.2, 30)
    tscale = 0.5 + synth.uniform01(12, R)
    tw = FieldTwin(J, h, S0, dtype)
    o1 = tw.run(rule, n1, nodes=None if nodes is None else nodes[:n1], start=13, fluct=fl[..., :n1],
                fluct_per_replica=per_rep, T=T, steps_per_T=spT, tscale=tscale, trace_every=tr)
    S1 = tw.S.copy()
    o2 = tw.run(rule, n2, nodes=None if nodes is None else nodes[n1:], start=(13 + n1) % n, fluct=fl[..., n1:],
                fluct_per_replica=per_rep, T=T[n1 // spT:], steps_per_T=spT, tscale=tscale)
    assert o1["flips"].sum() > 0 and (o2["flips"].sum() > 0 or rule == 0)   # (Hopfield runs reach a fixed point)
    for r in range(R):
        f = fl[r] if per_rep else fl
        s, flips, E, M = orc.ssf_run(rule, J, h, S0[r], n1, nodes=None if nodes is None else nodes[:n1], start=13,
                                     fluct=f[:n1], T=T * tscale[r], steps_per_T=spT, trace_every=tr)
        assert np.array_equal(s, S1[r]) and flips == o1["flips"][r], f"replica {r}"
        assert np.array_equal(M, o1["M"][:, r]) and np.allclose(E, o1["E"][:, r], rtol=1e-12, atol=1e-12)
        s, flips, _, _ = orc.ssf_run(rule, J, h, S1[r], n2, nodes=None if nodes is None else nodes[n1:],
                                     start=(13 + n1) % n, fluct=f[n1:], T=T[n1 // spT:] * tscale[r], steps_per_T=spT)
        assert np.array_equal(s, tw.S[r]) and flips == o2["flips"][r], f"replica {r}"


def test_twin_leaves_the_oracle_on_continuum_couplings(orc, synth):
    """Gaussian couplings in Float32 storage: the first decision of every chain is put exactly on the reference's
    tie (F T = 2 x its fresh Float64 field, up by heaviside(0) = 1).  The twin decides on the rounded float field: down
    exactly where float rounding lowered the field, so it leaves the oracle in those chains and follows it elsewhere."""
    n, R, site = 64, 24, 5
    J, h = synth.sk_J(n, 31), synth.gaussian(32, n) * 0.3
    S0 = synth.spins(33, R, n)
    f64 = np.array([orc.local_field(J, h, S0[r])[site] for r in range(R)])
    fl = np.zeros((R, 40))
    fl[:, 0] = 2.0 * f64                                        # T = 1: x = 2 f - F T = 0 in the reference
    tw = FieldTwin(J, h, S0, np.float32)
    tw.run(1, 40, start=site, fluct=fl, fluct_per_replica=True, T=np.ones(1), steps_per_T=40)
    lowered = FieldTwin(J, h, S0, np.float32).fresh_fields(+1)[:, site].astype(np.float64) < f64
    differ = np.array([not np.array_equal(orc.ssf_run(1, J, h, S0[r], 40, start=site, fluct=fl[r], T=np.ones(1),
                                                      steps_per_T=40)[0], tw.S[r]) for r in range(R)])
    assert 0 < lowered.sum() < R
    assert np.array_equal(differ, lowered)


@pytest.mark.parametrize("order", ["seq", "list"])
@pytest.mark.parametrize("n", [20, 50, 100, 200, 400, 1000])
def test_guard_cases_need_the_guard(orc, synth, n, order):
    """The near-tie guard cases of the GPU variant matrix are strong enough: the incremental Float64 dynamics *without*
    the guard (the twin in Float64 storage, with the library's refresh rule) leaves the reference in some chain."""
    J, h, S0 = guard_case(synth, n)
    nsteps, per = GUARD_SWEEPS * n, GUARD_PER * n
    nodes = synth.nodes(95 + n, n, nsteps) if order == "list" else None
    tw = FieldTwin(J, h, S0, np.float64)
    for t0 in range(0, nsteps, per):
        tw.run(1, per, nodes=None if nodes is None else nodes[t0:t0 + per], start=t0 % n, fluct=np.zeros(per),
               T=np.zeros(1), steps_per_T=per)
    S, _ = orc.ssf_run_batch(1, J, h, S0, nsteps, nodes=nodes, fluct=np.zeros(nsteps), T=np.zeros(1), steps_per_T=nsteps,
                             nthreads=4)
    assert any(not np.array_equal(S[r], tw.S[r]) for r in range(len(S0)))

"""GPU tests of the Swendsen-Wang sweeps (isb_sw_run, cluster.SwendsenWang).

The core check is a replay: tests/sw_reference.py restates the documented rule in numpy (bond list, Philox words, CPU
labelling with root = smallest site, field grid) and must reproduce the final spins, traced E / M / sum |C|^2 and the flip
counts bit for bit.  The physics tests compare with exact results (Kaufman's solution of the torus, enumeration)
independently of the RNG."""
import numpy as np
import pytest
import scipy.sparse as sp

from exact_ising import mean_energy
from sw_reference import sw_replay

pytestmark = pytest.mark.gpu


def _lib():
    from isingmodel_jl_b200 import _lib
    return _lib


def _torus(L, coupling=1.0):
    from isingmodel_jl_b200 import synth
    return sp.csc_matrix(synth.lattice_J(L, coupling))


def _pm_torus(L, seed):
    """L x L torus with +-1 couplings."""
    from isingmodel_jl_b200 import synth
    A = sp.triu(_torus(L), 1).tocoo()
    v = np.where(synth.uniform01(seed, A.nnz) < 0.5, -1.0, 1.0)
    U = sp.coo_matrix((v, (A.row, A.col)), shape=A.shape)
    return (U + U.T).tocsc()


def _gauss_torus(L, seed):
    from isingmodel_jl_b200 import synth
    A = sp.triu(_torus(L), 1).tocoo()
    U = sp.coo_matrix((synth.gaussian(seed, A.nnz), (A.row, A.col)), shape=A.shape)
    return (U + U.T).tocsc()


def _regular3(n, seed):
    """Random 3-regular graph (configuration model, loops and multi-edges dropped) with Gaussian couplings."""
    rng = np.random.default_rng(seed)
    stubs = rng.permutation(np.repeat(np.arange(n), 3))
    i, j = stubs[0::2], stubs[1::2]
    keep = i != j
    i, j = np.minimum(i[keep], j[keep]), np.maximum(i[keep], j[keep])
    ij = np.unique(np.stack([i, j], 1), axis=0)
    U = sp.coo_matrix((rng.standard_normal(len(ij)), (ij[:, 0], ij[:, 1])), shape=(n, n))
    return (U + U.T).tocsc()


def _demo3x3():
    return sp.csc_matrix(np.load(__import__("os").path.join(__import__("os").path.dirname(__file__), "golden",
                                                              "ssf_3x3_glauber.npz"))["J"])


def _spins(seed, R, n):
    return np.where(np.random.default_rng(seed).random((R, n)) < 0.5, -1, 1).astype(np.int8)


def _run_and_replay(ctx, J, h, R, nsweeps, T, *, seed=5, sweeps_per_T=None, scale=None, replicas=None, trace_every=1,
                    dyadic=True, want_csq=True):
    L = _lib()
    n = J.shape[0]
    T = np.atleast_1d(np.asarray(T, dtype=np.float64))
    spT = nsweeps if (sweeps_per_T is None and T.size == 1) else (sweeps_per_T or 1)
    ens = L.Ensemble(L.Model.sparse(ctx, J, h), R)
    S0 = _spins(seed + 100, R, n)
    ens.set_spins(S0)
    if scale is not None:
        ens.set_temperature_scale(scale)
    out = ens.sw_run(nsweeps, T, sweeps_per_T=spT, trace_every=trace_every, seed=seed, want_csq=want_csq)
    S = ens.get_spins()
    ref = sw_replay(J, h, S0, nsweeps, T, seed, sweeps_per_T=spT, scale=scale, replicas=replicas, trace_every=trace_every)
    reps = np.arange(R) if replicas is None else np.asarray(replicas)
    assert np.array_equal(S[reps], ref["S"]), "final spins differ from the replay"
    assert np.array_equal(out["flips"][reps], ref["flips"])
    if trace_every > 0:
        assert np.array_equal(out["M"][:, reps], ref["M"])
        if want_csq:
            assert np.array_equal(out["csq"][:, reps], ref["csq"])
        else:
            assert out["csq"] is None
        if dyadic:
            assert np.array_equal(out["E"][:, reps], ref["E"])
        else:
            assert np.allclose(out["E"][:, reps], ref["E"], rtol=1e-12, atol=1e-12 * n)
    else:
        assert out["E"] is None and out["M"] is None and out["csq"] is None
    st = ens.last_stats()
    assert st["launches"] == 1 and st["flips"] == int(out["flips"].sum())
    return ens, out, S0


@pytest.mark.parametrize("T", [1.5, 2.269, 5.0])
def test_ferromagnet_32x32_matches_replay(ctx, T):
    _run_and_replay(ctx, _torus(32), np.zeros(1024), 16, 6, T)


def test_pm_j_64x64_matches_replay(ctx):
    _run_and_replay(ctx, _pm_torus(64, 3), np.zeros(4096), 7, 5, 1.0)


def test_gaussian_with_non_dyadic_field_matches_replay(ctx):
    from isingmodel_jl_b200 import synth
    _run_and_replay(ctx, _gauss_torus(32, 4), synth.gaussian(6, 1024) * 0.3, 8, 6, 1.2, dyadic=False)


def test_random_3_regular_graph_matches_replay(ctx):
    from isingmodel_jl_b200 import synth
    _run_and_replay(ctx, _regular3(500, 8), synth.gaussian(9, 500) * 0.2, 9, 8, 0.8, dyadic=False)


def test_demo_3x3_antiferromagnet_matches_replay(ctx):
    _run_and_replay(ctx, _demo3x3(), np.array([0.25, -0.5, 0, 0, 0.125, 0, 0, 0, 1.0]), 33, 20, 1.0)


def test_schedule_and_temperature_factors_match_replay(ctx):
    T = np.array([3.0, 2.5, 2.2, 2.0])
    _run_and_replay(ctx, _torus(32), np.zeros(1024), 12, 8, T, sweeps_per_T=2, trace_every=2)
    scale = np.linspace(0.6, 1.6, 12)
    _run_and_replay(ctx, _torus(32), np.zeros(1024), 12, 8, T, sweeps_per_T=2, trace_every=3, scale=scale)


@pytest.mark.parametrize("R", [1, 7, 4096])
def test_replica_counts_match_replay(ctx, R):
    reps = None if R < 100 else np.array([0, 1, 2, 1000, 2047, 2048, 3333, 4095])
    _run_and_replay(ctx, _torus(32), np.zeros(1024), R, 4, 2.269, replicas=reps)


def test_largest_supported_size_matches_replay(ctx):
    """n = 16384 (a 128 x 128 torus) with a field and every output requested."""
    from isingmodel_jl_b200 import synth
    h = np.round(synth.gaussian(21, 16384) * 8) / 64
    _run_and_replay(ctx, _torus(128), h, 3, 3, 2.269)


def test_untraced_without_field_matches_replay(ctx):
    """h = 0 and no trace: the kernel keeps no sum words (labels first in shared memory); small models pack several
    replicas per CTA, with idle groups in the last one (R = 33 of 9 sites, R = 9 of 500 sites)."""
    _run_and_replay(ctx, _torus(32), np.zeros(1024), 12, 7, 2.269, trace_every=0)
    _run_and_replay(ctx, _demo3x3(), np.zeros(9), 33, 15, 1.0, trace_every=0)
    _run_and_replay(ctx, _regular3(500, 8), np.zeros(500), 9, 6, 0.8, trace_every=0, dyadic=False)


def test_trace_without_cluster_sizes_matches_replay(ctx):
    """E and M traced without sum |C|^2, with and without a field."""
    _run_and_replay(ctx, _torus(32), np.zeros(1024), 10, 8, 2.269, trace_every=2, want_csq=False)
    _run_and_replay(ctx, _demo3x3(), np.array([0.25, -0.5, 0, 0, 0.125, 0, 0, 0, 1.0]), 17, 9, 1.0, trace_every=3,
                    want_csq=False)


def test_long_run_matches_replay_and_repeats(ctx):
    """300 sweeps at T_c (large clusters, deep union-find trees every sweep): replayed bit for bit on a subset of the
    replicas, and identical in a second run."""
    from isingmodel_jl_b200 import synth
    h = np.round(synth.gaussian(23, 1024) * 4) / 256
    ens, out, S0 = _run_and_replay(ctx, _torus(32), h, 64, 300, 2.269, trace_every=50, replicas=[0, 17, 40, 63])
    L = _lib()
    again = L.Ensemble(L.Model.sparse(ctx, _torus(32), h), 64)
    again.set_spins(S0)
    out2 = again.sw_run(300, 2.269, sweeps_per_T=300, trace_every=50, seed=5)
    assert np.array_equal(again.get_spins(), ens.get_spins())
    for key in ("E", "M", "csq", "flips"):
        assert np.array_equal(out[key], out2[key]), key


def test_deterministic_and_two_calls_equal_one(ctx):
    L = _lib()
    J, R, T = _torus(32), 64, np.array([2.6, 2.4, 2.269])
    S0 = _spins(31, R, 1024)
    res = []
    for _ in range(2):
        ens = L.Ensemble(L.Model.sparse(ctx, J, np.zeros(1024)), R)
        ens.set_spins(S0)
        out = ens.sw_run(9, T, sweeps_per_T=3, trace_every=1, seed=77)
        res.append((ens.get_spins(), out))
    assert np.array_equal(res[0][0], res[1][0])
    for key in ("E", "M", "csq", "flips"):
        assert np.array_equal(res[0][1][key], res[1][1][key]), key
    T9 = np.repeat(T, 3)
    one = res[0][1]
    ens = L.Ensemble(L.Model.sparse(ctx, J, np.zeros(1024)), R)
    ens.set_spins(S0)
    a = ens.sw_run(4, T9[:4], trace_every=1, seed=77)
    b = ens.sw_run(5, T9[4:], trace_every=1, seed=77, sweep_offset=4)
    assert np.array_equal(ens.get_spins(), res[0][0])
    assert np.array_equal(np.concatenate([a["E"], b["E"]]), one["E"])
    assert np.array_equal(np.concatenate([a["csq"], b["csq"]]), one["csq"])
    assert np.array_equal(a["flips"] + b["flips"], one["flips"])


def test_swendsen_wang_class_continues_the_chain(ctx):
    from isingmodel_jl_b200 import SwendsenWang
    from isingmodel_jl_b200.SpinSystems import SpinSystem
    J, R = _torus(32), 6
    S0 = _spins(41, R, 1024)
    ss = SpinSystem(S0, J, np.zeros(1024))
    sw = SwendsenWang(ss, seed=3)
    sw.temperatureScale = np.linspace(0.9, 1.1, R)
    sw.run(4, 2.3)
    out = sw.run(3, [2.3, 2.2, 2.1])
    ref = sw_replay(J, np.zeros(1024), S0, 4, [2.3], 3, sweeps_per_T=4, scale=sw.temperatureScale)
    ref = sw_replay(J, np.zeros(1024), ref["S"], 3, [2.3, 2.2, 2.1], 3, sweep_offset=4, scale=sw.temperatureScale,
                    trace_every=1)
    assert np.array_equal(ss.spinConfiguration, ref["S"]) and sw.offset == 7
    assert np.array_equal(out["E"], ref["E"]) and np.array_equal(out["csq"], ref["csq"])


# ------------------------------------------------------------------ physics
def _means(ens, nburn, nmeas, T, seed):
    ens.sw_run(nburn, T, sweeps_per_T=nburn, seed=seed)
    out = ens.sw_run(nmeas, T, sweeps_per_T=nmeas, trace_every=1, seed=seed, sweep_offset=nburn)
    return out


@pytest.mark.parametrize("T", [2.0, 2.269, 3.0])
def test_mean_energy_of_the_torus_matches_kaufman(ctx, T):
    L = _lib()
    R = 256
    ens = L.Ensemble(L.Model.sparse(ctx, _torus(32), np.zeros(1024)), R)
    ens.set_spins(_spins(51, R, 1024))
    out = _means(ens, 100, 200, T, 13)
    per = out["E"].mean(axis=0)                         # one mean per independent replica
    err = per.std(ddof=1) / np.sqrt(R)
    assert abs(per.mean() - mean_energy(32, T)) < 5 * err, (per.mean(), mean_energy(32, T), err)


def test_improved_susceptibility_estimator_matches_m2(ctx):
    L = _lib()
    R, N = 256, 1024
    ens = L.Ensemble(L.Model.sparse(ctx, _torus(32), np.zeros(N)), R)
    ens.set_spins(_spins(52, R, N))
    out = _means(ens, 100, 200, 2.269, 17)
    a, b = out["csq"].mean(axis=0) / N, (out["M"] ** 2).mean(axis=0) / N
    d = a - b
    assert abs(d.mean()) < 5 * d.std(ddof=1) / np.sqrt(R)


def _enumerate(J, h, T):
    from sw_reference import bonds
    I, Jc, V = bonds(J)
    n = J.shape[0]
    st = ((np.arange(1 << n)[:, None] >> np.arange(n)[None, :]) & 1) * 2 - 1
    E = -(st[:, I] * st[:, Jc]) @ V - st @ h
    w = np.exp(-(E - E.min()) / T)
    return st, E, w / w.sum()


def test_field_4x4_torus_mean_energy_and_magnetisation(ctx):
    L = _lib()
    J, h, T, R = _torus(4), np.full(16, 0.3), 2.5, 2048
    st, Ex, p = _enumerate(J, h, T)
    ens = L.Ensemble(L.Model.sparse(ctx, J, h), R)
    ens.set_spins(_spins(53, R, 16))
    out = _means(ens, 50, 100, T, 19)
    for obs, exact in ((out["E"], Ex @ p), (out["M"], st.sum(1) @ p)):
        per = obs.mean(axis=0)
        assert abs(per.mean() - exact) < 5 * per.std(ddof=1) / np.sqrt(R), (per.mean(), exact)


def test_demo_3x3_histogram_with_a_field(ctx):
    L = _lib()
    J, h, T, R = _demo3x3(), np.array([0.3, -0.2, 0.1, 0.0, 0.25, -0.1, 0.05, 0.0, 0.15]), 1.0, 4096
    st, _, p = _enumerate(J, h, T)
    ens = L.Ensemble(L.Model.sparse(ctx, J, h), R)
    ens.set_spins(_spins(54, R, 9))
    ens.sw_run(50, T, sweeps_per_T=50, seed=23)
    counts = np.zeros(512)
    for c in range(4):                                   # configurations 25 sweeps apart, one per replica
        ens.sw_run(25, T, sweeps_per_T=25, seed=23, sweep_offset=50 + 25 * c)
        s = ens.get_spins()
        idx = ((s > 0).astype(np.int64) << np.arange(9)).sum(1)
        counts += np.bincount(idx, minlength=512)
    exp_ = p * counts.sum()
    keep = exp_ > 5
    chi2 = float((((counts - exp_) ** 2) / exp_)[keep].sum())
    dof = int(keep.sum()) - 1
    assert chi2 < dof + 6 * np.sqrt(2 * dof), (chi2, dof)


# ------------------------------------------------------------------ composition
def test_single_spin_run_after_swendsen_wang(ctx):
    """The cached fields of the neighbour-list kernel are rebuilt after an SW call: a random-order isb_ssf_run continues
    bit for bit like one on a fresh ensemble given the same spins; replica selection moves the SW chains."""
    L = _lib()
    from isingmodel_jl_b200 import synth
    J, h, R = _regular3(300, 61), synth.gaussian(62, 300) * 0.2, 8
    m = L.Model.sparse(ctx, J, h)
    ens = L.Ensemble(m, R)
    ens.set_spins(_spins(63, R, 300))
    ens.ssf_run(L.RULE_GLAUBER, 600, order=L.ORDER_RANDOM, T=[1.0], steps_per_T=600, seed=1)   # fields cached
    ens.sw_run(5, 1.0, sweeps_per_T=5, seed=2)
    S = ens.get_spins()
    fresh = L.Ensemble(m, R)
    fresh.set_spins(S)
    a = ens.ssf_run(L.RULE_GLAUBER, 900, order=L.ORDER_RANDOM, T=[1.0], steps_per_T=900, seed=3, trace_every=300)
    b = fresh.ssf_run(L.RULE_GLAUBER, 900, order=L.ORDER_RANDOM, T=[1.0], steps_per_T=900, seed=3, trace_every=300)
    assert np.array_equal(ens.get_spins(), fresh.get_spins()) and np.array_equal(a["E"], b["E"])
    src = np.array([3, 3, 0, 7, 1, 2, 6, 5], dtype=np.int32)
    before = ens.get_spins()
    ens.select_replicas(src)
    assert np.array_equal(ens.get_spins(), before[src])
    ens.sw_run(2, 1.0, sweeps_per_T=2, seed=4, sweep_offset=5)
    ref = sw_replay(J, h, before[src], 2, [1.0], 4, sweep_offset=5, sweeps_per_T=2)
    assert np.array_equal(ens.get_spins(), ref["S"])


# ------------------------------------------------------------------ errors
def test_errors_leave_the_spins_unchanged(ctx):
    L = _lib()
    from isingmodel_jl_b200 import synth

    def code(ens, *a, **k):
        with pytest.raises(L.IsbError) as ei:
            ens.sw_run(*a, **k)
        return ei.value.code

    dense = L.Ensemble(L.Model.dense(ctx, synth.sk_J(16, 1), None, L.PREC_F64), 2)
    assert code(dense, 2, 1.0) == L.ERR_STATE
    W, hv, bh = synth.bipartite_W(8, 4, 2)
    assert code(L.Ensemble(L.Model.bipartite(ctx, W, hv, bh), 2), 2, 1.0) == L.ERR_STATE
    n = 16385
    ring = sp.coo_matrix((np.ones(n), (np.arange(n), (np.arange(n) + 1) % n)), shape=(n, n))
    big = L.Ensemble(L.Model.sparse(ctx, (ring + ring.T).tocsc(), np.zeros(n)), 1)
    assert code(big, 1, 1.0) == L.ERR_UNSUPPORTED
    ens = L.Ensemble(L.Model.sparse(ctx, _torus(16), np.zeros(256)), 4)
    S0 = _spins(71, 4, 256)
    ens.set_spins(S0)
    assert code(ens, -1, 1.0) == L.ERR_ARG
    assert code(ens, 2, 1.0, sweeps_per_T=0) == L.ERR_ARG
    assert code(ens, 2, 1.0, trace_every=-1) == L.ERR_ARG
    assert code(ens, 3, [1.0], sweeps_per_T=2) == L.ERR_ARG          # schedule too short
    assert code(ens, 2, np.zeros(0)) == L.ERR_ARG                      # no schedule
    assert code(ens, 2, [1.0, -1.0]) == L.ERR_ARG
    assert code(ens, 2, [0.0], sweeps_per_T=2) == L.ERR_ARG
    assert code(ens, 2, [np.inf], sweeps_per_T=2) == L.ERR_NONFINITE
    assert code(ens, 2, [np.nan], sweeps_per_T=2) == L.ERR_NONFINITE
    ens.set_temperature_scale(np.array([1.0, -1.0, 1.0, 1.0]))
    assert code(ens, 2, 1.0, sweeps_per_T=2) == L.ERR_ARG
    ens.set_temperature_scale(None)
    assert np.array_equal(ens.get_spins(), S0)
    out = ens.sw_run(0, np.zeros(0))                                   # nsweeps = 0: a no-op
    assert np.array_equal(ens.get_spins(), S0) and not out["flips"].any()

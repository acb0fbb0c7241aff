"""GPU tests of the int8 digit-plane mode of the tcgen05 block-Gibbs path (ISB_PREC_I8X2 / _I8X3 / _I8X4).

The couplings are rounded ONCE to a fixed-point grid (isb_model_effective_couplings returns them) and the contraction
runs in exact int32 arithmetic, so — unlike the bf16 / fp16 term modes with their fp32 accumulators — the tensor path
must reproduce the Float64 reference (src/OnBipartiteGraph.jl:30-43,53-66) BIT FOR BIT on the grid couplings, for any
contraction depth: every sum the oracle forms over multiples of the quantum is exact in Float64 as well."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _lib():
    from isingmodel_jl_b200 import _lib
    return _lib


def _prec(L, name):
    return {"i8x2": L.PREC_I8X2, "i8x3": L.PREC_I8X3, "i8x4": L.PREC_I8X4}[name]


def _bits(name):
    return {"i8x2": 16, "i8x3": 24, "i8x4": 32}[name]


def _check_grid(W, Weff, bits, diag_split):
    """|W - Weff| <= quantum / 2 with quantum = 2^e <= 2^-(bits-2) max|W_offdiag| ... (a power of two)."""
    D = np.abs(W - Weff)
    off = np.abs(W - np.diag(np.diag(W))) if diag_split else np.abs(W)
    amax = off.max()
    q0 = 2.0 ** (np.ceil(np.log2(amax)) - (bits - 1))
    assert D.max() <= q0 + 1e-300, (D.max(), q0)          # within one quantum (half, unless the top digit clamped)
    k = Weff / (q0 / 2)                                     # on the grid (q0 or 2 q0 when the range was bumped)
    assert np.array_equal(k, np.rint(k))


I8_CASES = [  # nv, nh, rule, R, nsteps, prec, persist
    (96, 40, 0, 64, 4, "i8x3", None), (96, 40, 1, 64, 4, "i8x3", None),
    (300, 77, 0, 140, 3, "i8x3", None), (300, 77, 1, 140, 3, "i8x2", None),
    (784, 512, 0, 300, 2, "i8x3", None), (784, 512, 1, 130, 2, "i8x4", None),
    (200, 1000, 0, 257, 2, "i8x3", None), (24, 17, 0, 1, 5, "i8x3", None),
    (160, 96, 0, 300, 4, "i8x3", "1"), (160, 96, 1, 300, 4, "i8x3", "1"), (784, 512, 0, 1000, 3, "i8x3", "1"),
    (96, 80, 0, 19500, 2, "i8x3", None),       # chain-resident by default (>= 96 replicas per SM)
]


@pytest.mark.parametrize("nv,nh,rule,R,nsteps,prec,persist", I8_CASES)
def test_i8_trajectories_bit_exact(ctx, orc, synth, monkeypatch, nv, nh, rule, R, nsteps, prec, persist):
    L = _lib()
    if persist is not None:
        monkeypatch.setenv("ISB_TC_PERSIST", persist)
    W, h, b = synth.bipartite_W(nv, nh, 201, 0.1)
    m = L.Model.bipartite(ctx, W, h, b, _prec(L, prec))
    Weff = m.effective_couplings()
    _check_grid(W, Weff, _bits(prec), False)
    S0, T0 = synth.spins(202, R, nv), synth.spins(203, R, nh)
    gen = synth.logistic if rule == 0 else synth.exponential
    shared = R > 2000                      # keep the fluctuation arrays small for the many-replica case
    Fv = gen(204, (nsteps, nv) if shared else (R, nsteps, nv), 1)
    Fh = gen(204, (nsteps, nh) if shared else (R, nsteps, nh), 2)
    T = synth.geometric_schedule(2.0, 0.4, nsteps)
    e = L.Ensemble(m, R)
    e.set_spins(S0)
    e.set_hidden(T0)
    e.bip_run(rule, nsteps, Fv=Fv, Fh=Fh, fluct_per_replica=not shared, T=T)
    S, Tm = e.get_spins(), e.get_hidden()
    rows = range(R) if R <= 300 else list(range(0, R, 97)) + [R - 1]
    for r in rows:
        s, t, _ = orc.bip_run(rule, Weff, h, b, S0[r], T0[r], nsteps, Fv if shared else Fv[r], Fh if shared else Fh[r], T)
        assert np.array_equal(s, S[r]) and np.array_equal(t, Tm[r]), f"replica {r}"
    # both launch modes give the same bits
    for ps in ("0", "1"):
        monkeypatch.setenv("ISB_TC_PERSIST", ps)
        e2 = L.Ensemble(m, R)
        e2.set_spins(S0)
        e2.set_hidden(T0)
        e2.bip_run(rule, nsteps, Fv=Fv, Fh=Fh, fluct_per_replica=not shared, T=T)
        assert np.array_equal(e2.get_spins(), S) and np.array_equal(e2.get_hidden(), Tm), ps


@pytest.mark.parametrize("rule", [0, 1])
def test_i8_square_model_with_dominant_diagonal(ctx, orc, synth, rule):
    """The MultiSpinFlip embedding W = (J + qI)/2 (demo.jl:82-90): the diagonal is 64x the couplings; it is split off
    and added from the unit's own input spin, so the grid resolves the off-diagonal couplings to 2^-23 of THEIR maximum."""
    L = _lib()
    n, R, nsteps = 384, 150, 4
    J = synth.sk_J(n, 211)
    q = 0.5 * float(np.linalg.eigvalsh(J)[-1])
    W = 0.5 * (J + q * np.eye(n))
    hb = synth.gaussian(212, n) * 0.05
    m = L.Model.bipartite(ctx, W, hb, hb, L.PREC_I8X3)
    Weff = m.effective_couplings()
    _check_grid(W, Weff, 24, True)
    assert np.abs(W - Weff).max() < 2.0 ** -23 * np.abs(J).max()      # scaled to the couplings, not to q / 2
    S0 = synth.spins(213, R, n)
    gen = synth.logistic if rule == 0 else synth.exponential
    Fv, Fh = gen(214, (R, nsteps, n), 1), gen(214, (R, nsteps, n), 2)
    T = synth.geometric_schedule(1.0, 0.1, nsteps)
    e = L.Ensemble(m, R)
    e.set_spins(S0)
    e.set_hidden(S0)
    e.bip_run(rule, nsteps, Fv=Fv, Fh=Fh, fluct_per_replica=True, T=T)
    S, Tm = e.get_spins(), e.get_hidden()
    for r in range(R):
        s, t, _ = orc.bip_run(rule, Weff, hb, hb, S0[r], S0[r], nsteps, Fv[r], Fh[r], T)
        assert np.array_equal(s, S[r]) and np.array_equal(t, Tm[r]), f"replica {r}"


def test_i8_philox_mode_follows_the_f64_path(ctx, synth):
    """In-kernel noise: the same Philox words on both paths; the int8 path decides in fp32 on an exact field, the
    Float64 path in double on the original couplings: T = 0 with integer couplings must agree exactly (every step),
    Gaussian couplings almost always."""
    L = _lib()
    nv, nh, R = 192, 128, 512
    W = np.round(synth.gaussian(221, nv * nh).reshape(nv, nh) * 1.5)
    h, b = np.round(synth.gaussian(222, nv)), np.round(synth.gaussian(223, nh))
    S0, T0 = synth.spins(224, R, nv), synth.spins(225, R, nh)
    out = {}
    for prec in (L.PREC_F64, L.PREC_I8X3, L.PREC_I8X2):
        m = L.Model.bipartite(ctx, W, h, b, prec)
        if prec != L.PREC_F64:
            assert np.array_equal(m.effective_couplings(), W)      # small integers are on every grid
        e = L.Ensemble(m, R)
        e.set_spins(S0)
        e.set_hidden(T0)
        e.bip_run(0, 3, seed=5, T=np.zeros(3))
        out[prec] = (e.get_spins(), e.get_hidden())
    for prec in (L.PREC_I8X3, L.PREC_I8X2):
        assert np.array_equal(out[L.PREC_F64][0], out[prec][0]) and np.array_equal(out[L.PREC_F64][1], out[prec][1])
    W, h, b = synth.bipartite_W(nv, nh, 226, 0.1)
    En = {}
    for prec in (L.PREC_F64, L.PREC_I8X3):
        e = L.Ensemble(L.Model.bipartite(ctx, W, h, b, prec), R)
        e.set_spins(S0)
        e.set_hidden(T0)
        e.bip_run(0, 30, seed=6, T=np.full(30, 1.0))
        En[prec] = e.energy()
    a, c = En[L.PREC_F64], En[L.PREC_I8X3]
    assert np.mean(np.abs(a - c) < 1e-9 * np.maximum(1, np.abs(a))) > 0.9
    assert abs(a.mean() - c.mean()) < 4 * a.std() / np.sqrt(R)


@pytest.mark.parametrize("prec", ["i8x3", "bf16x3", "fp16x2"])
@pytest.mark.parametrize("rule", [0, 1])
def test_tensor_path_samples_the_boltzmann_distribution(ctx, synth, prec, rule):
    """Exact-enumeration check of the IN-KERNEL-NOISE tensor path (fp32 decisions, ex2.approx, 32-bit uniforms): block
    Gibbs (SCA) and the per-unit Metropolis of MomentumAnnealing both leave exp(-E(sigma, tau) / T) / Z invariant,
    E = -sigma' W tau - h' sigma - b' tau (src/SpinSystems.jl:139-145).  6 x 5 units = 2048 joint states, enumerated."""
    L = _lib()
    P = {"i8x3": L.PREC_I8X3, "bf16x3": L.PREC_BF16X3, "fp16x2": L.PREC_FP16X2}[prec]
    nv, nh, R, burn, keep, T = 6, 5, 8192, 40, 120, 1.3
    W, h, b = synth.bipartite_W(nv, nh, 231, 0.6)
    e = L.Ensemble(L.Model.bipartite(ctx, W, h, b, P), R)
    e.set_spins(synth.spins(232, R, nv))
    e.set_hidden(synth.spins(233, R, nh))
    e.bip_run(rule, burn, seed=17, T=np.full(burn, T))
    _, Sv, Sh = e.bip_run(rule, keep, seed=17, step_offset=burn, T=np.full(keep, T), trace_every=1, want_S=True)
    code = ((Sv.reshape(-1, nv) < 0) @ (1 << np.arange(nv))) | (((Sh.reshape(-1, nh) < 0) @ (1 << np.arange(nh))) << nv)
    hist = np.bincount(code, minlength=1 << (nv + nh)).astype(float)
    st = np.arange(1 << (nv + nh))
    sig = 1.0 - 2.0 * ((st[:, None] >> np.arange(nv)) & 1)
    tau = 1.0 - 2.0 * ((st[:, None] >> (nv + np.arange(nh))) & 1)
    E = -np.einsum("ki,ij,kj->k", sig, W, tau) - sig @ h - tau @ b
    p = np.exp(-E / T)
    p /= p.sum()
    tv = 0.5 * np.abs(hist / hist.sum() - p).sum()
    # 9.8e5 samples over 2048 states: the sampling noise of TV is ~ 0.5 sqrt(2 K / (pi n)) = 0.018 (chains decorrelate
    # within a few steps at this temperature); a wrong acceptance rule shows up as TV > 0.1
    assert tv < 0.04, tv
    assert 0.5 * np.abs(1.0 / len(p) - p).sum() > 0.3       # the target is far from uniform
    # per-unit marginals are a sharper check of the acceptance probabilities
    mv = (Sv.reshape(-1, nv) > 0).mean(0)
    assert np.abs(mv - ((sig > 0) * p[:, None]).sum(0)).max() < 0.01


def test_i8_row_sharded_blocks_equal_the_unsharded_path(pkg, ctx, synth):
    from isingmodel_jl_b200 import _lib as L, rowshard
    n, R, nsteps, seed = 512, 150, 4, 11
    J = synth.sk_J(n, 241)
    q = 1.5
    W = 0.5 * (J + q * np.eye(n))
    h = synth.gaussian(242, n) * 0.1
    S0 = synth.spins(243, R, n)
    T = synth.geometric_schedule(2.0, 0.3, nsteps)
    for rule in (0, 1):
        e = L.Ensemble(L.Model.bipartite(ctx, W, 0.5 * h, 0.5 * h, L.PREC_I8X3), R)
        e.set_spins(S0)
        e.set_hidden(S0)
        e.bip_run(rule, nsteps, seed=seed, T=T)
        ref_v, ref_h = e.get_spins(), e.get_hidden()
        for G in (1, 2, 4):
            sca = rowshard.RowShardedSCA(n, R, W=W, h=h, rule=rule, prec=L.PREC_I8X3, emulate_blocks=G)
            sca.set_spins(S0)
            sca.run(nsteps, T, seed=seed)
            assert np.array_equal(sca.get_spins(), ref_v), f"rule {rule} G={G}"
            assert np.array_equal(sca.get_hidden(), ref_h), f"rule {rule} G={G}"
    # the device-generated synthetic instance (a priori grid) against the same rows passed in with that grid
    a = rowshard.RowShardedSCA(n, R, seed=99, q=1.0, prec=L.PREC_I8X3, emulate_blocks=4)
    a.set_spins(S0)
    a.run(3, np.array([1.0, 0.7, 0.4]), seed=5)
    b = rowshard.RowShardedSCA(n, R, seed=99, q=1.0, prec=L.PREC_I8X3, emulate_blocks=2)
    b.set_spins(S0)
    b.run(3, np.array([1.0, 0.7, 0.4]), seed=5)
    assert np.array_equal(a.get_spins(), b.get_spins())

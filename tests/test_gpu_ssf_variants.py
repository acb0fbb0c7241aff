"""Every dense single-spin sweep kernel the launcher can pick (csrc/ssf.cu, ssf_run_device) meets a reference once, at
every chain layout: N = 20, 50, 100, 200, 400, 1000 give NPL = 1, 2, 4, 8, 16, 32 (ragged: padding and partial last
windows).  Each kernel is forced with ISB_SSF_MODE (2 streaming, 1 plain, 0 cold), which fails when the run cannot take
the kernel, so a case cannot pass on a substitute.

| family                       | kernels                                         | reference                     |
|------------------------------|-------------------------------------------------|-------------------------------|
| Float64                      | ssf_kernel<double, double, NPL, LIST, TMA>       | C oracle (bit-exact, E 1e-9)  |
| Float64, near-tie guard      | ssf_kernel<double, double, NPL, LIST, TMA, true> | C oracle                      |
| Float32                      | ssf_kernel<float, float, NPL, LIST, TMA>         | tests/ssf_float_twin.py       |
| int32 fixed point            | ssf_kernel<int32_t, int32_t, NPL, false, false>  | C oracle                      |
| cold, Float64 / int32        | ssf_cold_kernel<false> / <true>                  | C oracle                      |

Beyond the samples checked against the reference, every replica of one arithmetic must agree across its kernels:
Float64 streaming, plain, cold, fixed point and fixed-point cold; Float32 streaming and plain.

Combinations the launcher cannot launch, each shown to raise under ISB_SSF_MODE:
* cold Float64 at NPL 1 (Npad = 32 is not a multiple of 64) and cold int32 at NPL 1, 2 (Npad not a multiple of 128);
* cold Float32, cold with the near-tie guard, cold in list or random order or in a traced run (no such kernel);
* streaming int32 fixed point (the fixed-point path has no streaming kernel);
* fixed point in list or random order, in traced runs or with the tie audit, and for Float32 models (those runs take
  the Float64 or Float32 kernels instead: nothing to force)."""
import numpy as np
import pytest

from cases import GUARD_PER, GUARD_R, GUARD_SWEEPS, guard_case
from ssf_float_twin import FieldTwin

pytestmark = pytest.mark.gpu
E_RTOL = 1e-9
NS = [20, 50, 100, 200, 400, 1000]          # NPL = next_pow2(ceil(N / 32)) = 1, 2, 4, 8, 16, 32
# per N, rotated across the cases: (rule, noise, replicas, per-replica temperature factors, first site)
#   replicas: <= 148 -> one chain per CTA; 301, 157 -> several chains per CTA with a ragged last CTA; 2100 at NPL 32 -> two
#   waves of 14 Float64 chains per SM
CASES = {20: (1, "replica", 7, True, 5), 50: (2, "shared", 301, False, 17), 100: (0, None, 40, True, 33),
         200: (1, "philox", 157, True, 70), 400: (2, "replica", 148, False, 250), 1000: (1, "philox", 2100, True, 999)}
RANDOM_N = 200                              # the one random-order case of each family with list kernels
SEED = 4242


def _lib():
    from isingmodel_jl_b200 import _lib
    return _lib


def _npad(N):
    return 32 * (1 << max(0, int(np.ceil(N / 32)) - 1).bit_length())


def _samples(R, field_regs):
    """First, second, middle and last replica, and the first chain of the last CTA (the launcher's layout)."""
    chains = 14 if field_regs > 32 else (20 if field_regs > 16 else 28)
    if R <= 148:
        nw, ctas = 1, R
    else:
        waves = -(-R // (148 * chains))
        nw = -(-R // (148 * waves))
        ctas = -(-R // nw)
    return sorted({0, 1, R // 2, (ctas - 1) * nw, R - 1})


def _close(a, b, rtol=E_RTOL):
    return np.all(np.abs(a - b) <= rtol * np.maximum(1.0, np.abs(b)))


class Case:
    """The inputs of one (family, N) case: a ragged run, a schedule whose period is not a multiple of 32, traces at an
    odd period, the first site inside a window."""

    def __init__(self, ctx, synth, N, order, J=None, h=None):
        L = _lib()
        self.N = N
        self.rule, self.noise, self.R, tsc, self.start = CASES[N]
        self.order = order
        self.J = synth.sk_J(N, SEED + N) if J is None else J
        self.h = synth.gaussian(SEED + 1, N) * 0.3 if h is None else h
        self.S0 = synth.spins(SEED + 2 + N, self.R, N)
        sweeps = max(2, 600 // N)
        self.nsteps = sweeps * N + N // 3 + 7
        self.spT = (self.nsteps // 7) | 1
        self.trace_every = (self.nsteps // 4) | 1
        self.T = synth.geometric_schedule(3.0, 0.1, -(-self.nsteps // self.spT))
        self.tscale = 0.5 + synth.uniform01(SEED + 3, self.R) if tsc else None
        self.per_rep = self.noise == "replica"
        shape = (self.R, self.nsteps) if self.per_rep else self.nsteps
        gen = synth.logistic if self.rule == 1 else synth.exponential
        self.fl = gen(SEED + 4, shape) if self.noise in ("shared", "replica") else None
        self.nodes = None
        if order == "list":
            self.nodes = synth.nodes(SEED + 5, N, self.nsteps)
        elif order == "random":
            self.nodes = ctx.philox_nodes(N, SEED, 0, self.nsteps)
        self.ctx = ctx
        self.L = L

    def fluct_of(self, r):
        if self.rule == 0:
            return None
        if self.noise == "philox":
            return self.ctx.philox_fluct(self.rule, SEED, 0, r, 1, self.nsteps)[0]
        return self.fl[r] if self.per_rep else self.fl

    def T_of(self, r):
        return self.T if self.tscale is None else self.T * self.tscale[r]

    def run(self, e, monkeypatch, mode, fixed=False, trace=False):
        """One run from S0 (set_spins: the fields are rebuilt) with the kernel forced; (spins, run output, stats)."""
        L = self.L
        monkeypatch.setenv("ISB_SSF_MODE", str(mode))
        if fixed:
            monkeypatch.delenv("ISB_SSF_FIXED", raising=False)
        else:
            monkeypatch.setenv("ISB_SSF_FIXED", "0")
        e.set_spins(self.S0)
        order = {"seq": L.ORDER_SEQUENTIAL, "list": L.ORDER_LIST, "random": L.ORDER_RANDOM}[self.order]
        out = e.ssf_run(self.rule, self.nsteps, order=order, nodes=self.nodes if self.order == "list" else None,
                        start=self.start if self.order == "seq" else 0, fluct=None if self.rule == 0 else self.fl,
                        fluct_per_replica=self.per_rep, seed=SEED, T=self.T, steps_per_T=self.spT,
                        trace_every=self.trace_every if trace else 0)
        return e.get_spins(), out, e.last_stats()

    def refuses(self, e, monkeypatch, mode, fixed=False, trace=False):
        with pytest.raises(self.L.IsbError) as ei:
            self.run(e, monkeypatch, mode, fixed, trace)
        assert ei.value.code == self.L.ERR_ARG and "ISB_SSF_MODE" in str(ei.value)

    def check_oracle(self, orc, S, out, samples, traced):
        for r in samples:
            s, flips, E, M = orc.ssf_run(self.rule, self.J, self.h, self.S0[r], self.nsteps,
                                         nodes=None if self.order == "seq" else self.nodes,
                                         start=self.start if self.order == "seq" else 0, fluct=self.fluct_of(r),
                                         T=self.T_of(r), steps_per_T=self.spT,
                                         trace_every=self.trace_every if traced else 0)
            assert np.array_equal(s, S[r]) and flips == out["flips"][r], f"replica {r}"
            if traced:
                assert np.array_equal(M, out["M"][:, r]) and _close(out["E"][:, r], E), f"replica {r}"


def _same(a, b, what):
    assert np.array_equal(a[0], b[0]), f"{what}: spins differ"
    assert np.array_equal(a[1]["flips"], b[1]["flips"]), f"{what}: flip counts differ"


def _ensemble(L, ctx, c, prec):
    e = L.Ensemble(L.Model.dense(ctx, c.J, c.h, prec), c.R)
    if c.tscale is not None:
        e.set_temperature_scale(c.tscale)
    return e


@pytest.mark.parametrize("N", NS)
def test_float64_sequential_kernels(ctx, orc, synth, monkeypatch, N):
    """Sequential order on Float64 models: streaming and plain (traced: E and M against the oracle), cold, fixed point and
    fixed-point cold on the same inputs; all replicas agree, sampled ones equal the oracle."""
    L = _lib()
    c = Case(ctx, synth, N, "seq")
    e = _ensemble(L, ctx, c, L.PREC_F64)
    runs = {"streaming": c.run(e, monkeypatch, 2, trace=True), "plain": c.run(e, monkeypatch, 1, trace=True)}
    if _npad(N) % 64 == 0:
        runs["cold"] = c.run(e, monkeypatch, 0)
    else:
        c.refuses(e, monkeypatch, 0)
    c.refuses(e, monkeypatch, 0, trace=True)                    # traced: no cold kernel
    for k, v in runs.items():
        assert v[2]["exact_fallbacks"] == 0, k                  # the Float64 kernels never fall back
    runs["fixed"] = c.run(e, monkeypatch, 1, fixed=True)
    if _npad(N) % 128 == 0:
        runs["fixed cold"] = c.run(e, monkeypatch, 0, fixed=True)
    else:
        c.refuses(e, monkeypatch, 0, fixed=True)
    c.refuses(e, monkeypatch, 2, fixed=True)
    ref = runs["streaming"]
    for k, v in runs.items():
        _same(v, ref, k)
    assert np.array_equal(runs["plain"][1]["E"], ref[1]["E"]) and np.array_equal(runs["plain"][1]["M"], ref[1]["M"])
    assert ref[1]["flips"].sum() > 0
    c.check_oracle(orc, ref[0], ref[1], _samples(c.R, 2 * (_npad(N) // 32)), traced=True)


@pytest.mark.parametrize("N,order", [(N, "list") for N in NS] + [(RANDOM_N, "random")])
def test_float64_list_kernels(ctx, orc, synth, monkeypatch, N, order):
    """List and random order on Float64 models: streaming (traced) and plain; no cold kernel."""
    L = _lib()
    c = Case(ctx, synth, N, order)
    e = _ensemble(L, ctx, c, L.PREC_F64)
    st, pl = c.run(e, monkeypatch, 2, trace=True), c.run(e, monkeypatch, 1)
    _same(pl, st, "plain")
    c.refuses(e, monkeypatch, 0)
    assert st[1]["flips"].sum() > 0
    c.check_oracle(orc, st[0], st[1], _samples(c.R, 2 * (_npad(N) // 32)), traced=True)


@pytest.mark.parametrize("N", NS)
def test_float32_kernels(ctx, synth, monkeypatch, N):
    """Float32 models (float couplings and fields, Float64 decisions) against the Float32 twin: sequential, list and (one N)
    random order, streaming and plain; traced E against the twin's energy of its own float fields, M exact."""
    L = _lib()
    orders = ["seq", "list"] + (["random"] if N == RANDOM_N else [])
    for order in orders:
        c = Case(ctx, synth, N, order)
        e = _ensemble(L, ctx, c, L.PREC_F32)
        st, pl = c.run(e, monkeypatch, 2, trace=True), c.run(e, monkeypatch, 1)
        _same(pl, st, f"{order}: plain")
        c.refuses(e, monkeypatch, 0)                            # no Float32 cold kernel
        assert st[1]["flips"].sum() > 0
        sm = _samples(c.R, _npad(N) // 32)
        tw = FieldTwin(c.J, c.h, c.S0[sm], np.float32)
        fl = None if c.rule == 0 else np.stack([c.fluct_of(r) for r in sm])
        o = tw.run(c.rule, c.nsteps, nodes=None if order == "seq" else c.nodes, start=c.start if order == "seq" else 0,
                   fluct=fl, fluct_per_replica=True, T=c.T, steps_per_T=c.spT,
                   tscale=None if c.tscale is None else c.tscale[sm], trace_every=c.trace_every)
        assert np.array_equal(tw.S, st[0][sm]), f"{order}: spins differ from the Float32 twin"
        assert np.array_equal(o["flips"], st[1]["flips"][sm]), f"{order}: flip counts differ from the Float32 twin"
        assert np.array_equal(o["M"], st[1]["M"][:, sm])
        assert _close(st[1]["E"][:, sm], o["E"], 1e-12)


@pytest.mark.parametrize("N", NS)
def test_guard_kernels(ctx, orc, synth, monkeypatch, N):
    """Couplings +-0.1 / +-0.3 and h = 0 at T = 0 (tests/cases.py guard_case): exact ties and one-ulp cancellations of the
    reference again and again, in 300 sweeps run as four runs of 75 (each run after the first refreshes the fields).  On
    these inputs the incremental dynamics without the guard leave the reference (tests/test_ssf_float_twin.py).  The
    guarded Float64 kernels (streaming and plain, sequential, list and, for one N, random order) and the fixed-point
    kernels with their exact fallback must follow the oracle in every chain."""
    L = _lib()
    J, h, S0 = guard_case(synth, N)
    rule = CASES[N][0]
    nsteps, per = GUARD_SWEEPS * N, GUARD_PER * N
    e = L.Ensemble(L.Model.dense(ctx, J, h, L.PREC_F64), GUARD_R)
    lists = {"list": synth.nodes(95 + N, N, nsteps)}
    if N == RANDOM_N:
        lists["random"] = ctx.philox_nodes(N, SEED, 0, nsteps)

    def run(order, mode, fixed=False):
        monkeypatch.setenv("ISB_SSF_MODE", str(mode))
        if fixed:
            monkeypatch.delenv("ISB_SSF_FIXED", raising=False)
        else:
            monkeypatch.setenv("ISB_SSF_FIXED", "0")
        e.set_spins(S0)
        flips, fallbacks = np.zeros(GUARD_R, dtype=np.int64), 0
        for t0 in range(0, nsteps, per):
            kw = {"start": t0 % N} if order == "seq" else (
                {"nodes": lists["list"][t0:t0 + per]} if order == "list" else
                {"order": L.ORDER_RANDOM, "seed": SEED, "step_offset": t0})
            out = e.ssf_run(rule, per, fluct=np.zeros(per), T=np.zeros(1), steps_per_T=per, **kw)
            flips += out["flips"]
            fallbacks += e.last_stats()["exact_fallbacks"]
        return e.get_spins(), flips, fallbacks

    for order in ["seq"] + list(lists):
        nodes = lists.get(order)
        want = [orc.ssf_run(rule, J, h, S0[r], nsteps, nodes=nodes, fluct=np.zeros(nsteps), T=np.zeros(1),
                            steps_per_T=nsteps)[:2] for r in range(GUARD_R)]
        got = {"streaming": run(order, 2), "plain": run(order, 1)}
        if order == "seq":
            got["fixed"] = run(order, 1, fixed=True)
            if _npad(N) % 128 == 0:
                got["fixed cold"] = run(order, 0, fixed=True)
        for k, (S, flips, fallbacks) in got.items():
            for r in range(GUARD_R):
                assert np.array_equal(S[r], want[r][0]) and flips[r] == want[r][1], f"{order} {k}: replica {r}"
            # route evidence: the fixed-point kernels decide the ties on the exact path, the Float64 ones never do
            assert (fallbacks > 0) == k.startswith("fixed"), f"{order} {k}: {fallbacks} exact fallbacks"
        with pytest.raises(L.IsbError):                         # no cold kernel with the near-tie guard
            run(order, 0)


@pytest.mark.parametrize("mode", [2, 1])
def test_float32_fields_drift_within_a_run_and_are_rebuilt_after_64_sweeps(ctx, monkeypatch, mode):
    """Site 0 (h = 0) couples with J = 1 to sites 1 and 2, which their own fields flip in turn, and with J = 2^-30 to site 3,
    which stays down.  Its fresh field is -2^-30 throughout; in float, the first flip takes it to -2 - 2^-30 = -2 and the
    second to 0, so at T = 0 the cached field turns site 0 up where the reference keeps it down.  The library (and the
    twin) follows the drifted field until a run starts at least 64 N steps after the last rebuild, and the rebuilt one
    from then on."""
    L = _lib()
    monkeypatch.setenv("ISB_SSF_MODE", str(mode))
    n, R = 4, 3
    J = np.zeros((n, n))
    J[0, 1] = J[1, 0] = J[0, 2] = J[2, 0] = 1.0
    J[0, 3] = J[3, 0] = 2.0 ** -30
    h = np.array([0.0, -10.0, 10.0, -10.0])
    S0 = np.tile(np.array([-1, 1, -1, -1], dtype=np.int8), (R, 1))
    e = L.Ensemble(L.Model.dense(ctx, J, h, L.PREC_F32), R)
    tw = FieldTwin(J, h, S0, np.float32)
    e.set_spins(S0)
    seen, done = [], 0
    for nsteps in (n, 64 * n - n - 1, 1, n, 64 * n, n):
        kw = dict(start=(1 + done) % n, fluct=np.zeros(nsteps), T=np.zeros(1), steps_per_T=nsteps)
        out = e.ssf_run(L.RULE_GLAUBER, nsteps, **kw)
        o = tw.run(L.RULE_GLAUBER, nsteps, **kw)
        S = e.get_spins()
        assert np.array_equal(S, tw.S) and np.array_equal(out["flips"], o["flips"]), f"after {done + nsteps} steps"
        seen.append(int(S[0, 0]))
        done += nsteps
    # drifted up in the first run; no rebuild before a run that starts 64 N steps after the first; rebuilt there: down
    assert seen == [1, 1, 1, -1, -1, -1]

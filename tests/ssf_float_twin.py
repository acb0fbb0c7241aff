"""A numpy restatement of the library's dense single-spin dynamics with cached fields in a given storage type — TEST
INFRASTRUCTURE, not the reference algorithm (that is ``oracle``).

The reference takes every decision on a fresh Float64 row dot.  The sweep kernels keep cached local fields instead and
update them by +-2 J[i, :] per accepted flip.  With ``ISB_PREC_F32`` the couplings and fields are floats, so the
library's trajectories are *not* the reference's; this twin states what they are, operation by operation:

* couplings ``Jf = dtype(J)`` (J symmetric with a zero diagonal, as the model stores it);
* a (re)built field ``f_i = dtype(fl64(sum_j (double) Jf_ij s_j, sequentially over ascending j) +- h_i)``, + for Glauber
  and Metropolis, - for Hopfield (``field_init_kernel<float, true>``, ``csrc/ssf.cu``);
* the decision ``x = fl64(2 (double) f_i - fts)`` with ``fts = fl64(F Tl)``, negated for Metropolis when the spin is
  down, ``Tl = fl64(T[k // steps_per_T] tscale[r])``; the spin is up iff ``!(x < 0)``;
* an accepted flip of site i with d = +-2: ``f_j = dtype(f_j + d Jf_ij)`` for every j (the product is exact);
* the fields are rebuilt at the start of a run when the rule's h sign changed, after ``set_spins``, or once at least
  ``64 N`` steps have run since the last rebuild (``ssf_ensure_fields``); never inside a run;
* traced ``E = -1/2 sum_i s_i (double) f_i - ecoef sum_i h_i s_i``, ecoef 1.5 for Hopfield and 0.5 otherwise.

With ``dtype=np.float64`` and couplings whose sums are exact (integers, dyadic values) it is the reference's dynamics;
tests/test_ssf_float_twin.py checks that against the C oracle."""
import numpy as np

HOPFIELD, GLAUBER, METROPOLIS = 0, 1, 2
FIELD_REFRESH_SWEEPS = 64   # ISB_FIELD_REFRESH_SWEEPS, csrc/handles.hpp


class FieldTwin:
    """R chains of one dense model, vectorised over the chains; one Python iteration per step."""

    def __init__(self, J, h, S, dtype=np.float32):
        J = np.asarray(J, dtype=np.float64)
        assert np.array_equal(J, J.T) and not np.any(np.diag(J)), "give the twin a symmetric J with a zero diagonal"
        self.dtype = np.dtype(dtype)
        self.Jf = J.astype(self.dtype)
        self.Jd = self.Jf.astype(np.float64)
        self.n = J.shape[0]
        self.h = np.zeros(self.n) if h is None else np.asarray(h, dtype=np.float64).copy()
        self.set_spins(S)

    def set_spins(self, S):
        self.S = np.array(S, dtype=np.int8, copy=True).reshape(-1, self.n)
        self.F = None
        self.sign = 0               # 0: no valid fields (rebuilt by the next run)
        self.since = 0              # steps run since the last rebuild

    def fresh_fields(self, sign):
        """The fields a rebuild computes now (double accumulation over ascending j, then +- h, then one rounding)."""
        acc = np.zeros(self.S.shape, dtype=np.float64)
        s = self.S.astype(np.float64)
        for j in range(self.n):
            acc += self.Jd[j][None, :] * s[:, j:j + 1]      # J symmetric: column j of row i is row j of column i
        return (acc + self.h[None, :] if sign > 0 else acc - self.h[None, :]).astype(self.dtype)

    def energy(self, rule):
        """The traced energy of the kernels: computed from the cached fields, not from a fresh row dot."""
        s = self.S.astype(np.float64)
        ecoef = 1.5 if rule == HOPFIELD else 0.5
        return -0.5 * np.sum(s * self.F.astype(np.float64), axis=1) - ecoef * (s @ self.h)

    def run(self, rule, nsteps, *, nodes=None, start=0, fluct=None, fluct_per_replica=False, T=None, steps_per_T=1,
            tscale=None, trace_every=0):
        """One library run (isb_ssf_run); returns dict(flips[R], E[ntr][R], M[ntr][R]).  ``fluct`` is shared [nsteps] or,
        with ``fluct_per_replica``, [R][nsteps] (pass the Philox variates of the chains for in-kernel noise)."""
        R, n = self.S.shape
        sign = -1 if rule == HOPFIELD else 1
        if self.since >= FIELD_REFRESH_SWEEPS * n:
            self.sign = 0
        if self.sign != sign:
            self.F = self.fresh_fields(sign)
            self.sign = sign
            self.since = 0
        T = np.atleast_1d(np.asarray(T, dtype=np.float64))
        tsc = np.ones(R) if tscale is None else np.asarray(tscale, dtype=np.float64)
        fl = None if (rule == HOPFIELD or fluct is None) else np.asarray(fluct, dtype=np.float64)
        flips = np.zeros(R, dtype=np.int64)
        ntr = nsteps // trace_every if trace_every > 0 else 0
        E, M = np.zeros((ntr, R)), np.zeros((ntr, R))
        two = self.dtype.type(2)
        for k in range(nsteps):
            i = int(nodes[k]) if nodes is not None else (start + k) % n
            if fl is None:
                ft = np.zeros(R)
            else:
                ft = (fl[:, k] if fluct_per_replica else fl[k]) * (T[k // steps_per_T] * tsc)
            s = self.S[:, i]
            fts = np.where(s > 0, ft, -ft) if rule == METROPOLIS else ft
            x = 2.0 * self.F[:, i].astype(np.float64) - fts
            up = ~(x < 0.0)
            flip = up != (s > 0)
            if flip.any():
                rs = np.nonzero(flip)[0]
                d = np.where(up[rs], two, -two).astype(self.dtype)
                self.F[rs] = self.F[rs] + d[:, None] * self.Jf[i][None, :]
                self.S[rs, i] = np.where(up[rs], 1, -1)
                flips[rs] += 1
            if ntr and (k + 1) % trace_every == 0:
                E[(k + 1) // trace_every - 1] = self.energy(rule)
                M[(k + 1) // trace_every - 1] = self.S.sum(axis=1)
        self.since += nsteps
        return {"flips": flips, "E": E, "M": M}

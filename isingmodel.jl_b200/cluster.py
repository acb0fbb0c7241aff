"""Swendsen-Wang cluster sweeps (isb_sw_run) for spin systems with sparse couplings.

Near a critical point single-spin dynamics decorrelate in about L^2.17 sweeps on a 2D lattice; a Swendsen-Wang sweep
(bonds between aligned neighbours activated with probability 1 - exp(-2|J|/T), every cluster of active bonds flipped as a
whole) decorrelates in about L^0.2-0.35.  What a user near T_c pays for is an independent sample, not a spin update.
"""
from __future__ import annotations

import numpy as np

__all__ = ["SwendsenWang"]


class SwendsenWang:
    """Swendsen-Wang sweeps of every replica of ``ss`` (a ``SpinSystem`` built from a scipy.sparse coupling matrix, at
    most 16384 sites; an updating algorithm with a ``spinSystem`` field is accepted too).

    The sweeps draw from the library's counter RNG (``seed``) indexed by the absolute sweep, which ``run`` keeps in
    ``offset``: consecutive calls continue one chain, bit for bit the same as one longer call.
    ``temperatureScale``: optional per-replica temperature factors ([replicas], None = 1); replica r runs sweep k at
    T[k] * temperatureScale[r].  They are pushed to the device before every call."""

    def __init__(self, ss, *, seed=0):
        self.ss = ss.spinSystem if hasattr(ss, "spinSystem") else ss
        self.seed = int(seed)
        self.offset = 0              # sweeps run so far (the absolute index of the next one)
        self.temperatureScale = None

    def run(self, sweeps, T, *, trace_every=1):
        """``sweeps`` sweeps; ``T`` is a scalar or one temperature per sweep.  Returns dict(E, M [ntr][R] | None, csq
        [ntr][R] int64 | None (sum of |C|^2 over the clusters of the traced sweep; <csq> / N is the susceptibility at
        h = 0), flips [R]); ntr = sweeps // trace_every (trace_every = 0: no traces)."""
        sweeps = int(sweeps)
        Ta = np.asarray(T, dtype=np.float64).reshape(-1)
        if Ta.size != 1 and Ta.size != sweeps:
            raise ValueError(f"T must be a scalar or one temperature per sweep ({Ta.size} values for {sweeps} sweeps)")
        spT = sweeps if Ta.size == 1 else 1
        ens = self.ss._ensemble()
        # (the ensemble may have been rebuilt since the last call, which drops factors set on it earlier)
        ens.set_temperature_scale(None if self.temperatureScale is None
                                  else np.asarray(self.temperatureScale, dtype=np.float64).reshape(-1))
        out = ens.sw_run(sweeps, Ta, sweeps_per_T=max(spT, 1), trace_every=int(trace_every), seed=self.seed,
                         sweep_offset=self.offset)
        self.ss._dev_newer = True
        self.offset += sweeps
        return out

"""Replica axis utilities (SURVEY §8f rank 4): temperature ladders and replica exchange (parallel tempering) on
top of an ensemble, using per-replica temperature factors (isb_ens_set_temperature_scale).

The reference has one chain per object and a scalar ``temperature``; R reference objects that differ only in
their temperature are one ensemble here.  A swap exchanges the *temperatures* of two replicas (the spins stay
where they are), accepted with probability min(1, exp((1/T_a - 1/T_b)(E_a - E_b))).
"""
from __future__ import annotations

import numpy as np

from . import SamplingHelper, _lib
from .SpinSystems import calcEnergy


def set_temperatures(ua, temperatures):
    """Give replica r the temperature ``temperatures[r]`` for all later runs: the algorithm's scalar temperature
    (or schedule) becomes a common factor, ``temperatures / ua.temperature`` the per-replica scale."""
    ss = ua.spinSystem
    t = np.asarray(temperatures, dtype=np.float64)
    if t.shape != (ss.replicas,):
        raise ValueError("one temperature per replica is required")
    ua.temperatureScale = t / float(ua.temperature)
    ss._ensemble().set_temperature_scale(ua.temperatureScale)


def configurationIndex(spins):
    """The demo's labelling of a configuration (demo.jl:161-165): the integer whose binary digits are (1 - s_i)/2,
    first site most significant.  ``spins``: [..., N] of +-1."""
    s = np.asarray(spins)
    bits = ((1 - s) // 2).astype(np.int64)
    w = 1 << np.arange(s.shape[-1] - 1, -1, -1, dtype=np.int64)
    return bits @ w


def configurationHistogram(ua, maxMCSteps, *, stride=1, burn_in=0, seed=0, order="random", chunk=1 << 16):
    """Counts of the configurations visited by every replica (the histogram cell of demo.jl:159-168, which maps
    all states of ``makeSampler!(GlauberDynamics(ss, T), 50000)`` through ``configurationIndex``), taken every
    ``stride`` steps after ``burn_in`` steps, accumulated on the device (isb_ssf_run_hist).  Returns int64[2^N]."""
    n = ua.spinSystem._host_spins.shape[1]
    hist = np.zeros(1 << n, dtype=np.int64)
    off = 0
    if burn_in:
        SamplingHelper.run_(ua, burn_in, seed=seed, order=order, temperatures=np.array([ua.temperature]),
                            steps_per_T=burn_in)
        off = burn_in
    chunk = max(stride, chunk // stride * stride)
    done = 0
    while done < maxMCSteps:
        m = min(chunk, maxMCSteps - done)
        SamplingHelper.run_(ua, m, seed=seed, step_offset=off + done, order=order, start=(done % n) if order == "sequential" else 0,
                            temperatures=np.array([ua.temperature]), steps_per_T=m, trace_every=stride, hist=hist)
        done += m
    return hist


class ParallelTempering:
    """``ladders`` independent temperature ladders of ``len(levels)`` replicas each (replica index =
    ladder * len(levels) + slot).  ``run`` alternates ``sweeps`` sequential sweeps of every replica at its current
    temperature with one round of neighbour swaps inside each ladder."""

    def __init__(self, ua, levels, *, seed=0):
        self.ua, self.ss = ua, ua.spinSystem
        self.levels = np.asarray(levels, dtype=np.float64)
        L = len(self.levels)
        if self.ss.replicas % L:
            raise ValueError("the number of replicas must be a multiple of the number of temperature levels")
        self.nlad = self.ss.replicas // L
        # level[l, s] = index into `levels` currently held by slot s of ladder l
        self.level = np.tile(np.arange(L), (self.nlad, 1))
        self.rng = np.random.default_rng(seed)
        self.seed, self.offset = int(seed), 0
        self.accepted = np.zeros(L - 1, dtype=np.int64)
        self.proposed = np.zeros(L - 1, dtype=np.int64)
        ua.temperature = 1.0
        self._push()

    def _push(self):
        self.ua.temperatureScale = self.levels[self.level].reshape(-1)
        self.ss._ensemble().set_temperature_scale(self.ua.temperatureScale)

    def run(self, rounds, sweeps=1):
        """Returns E[rounds][levels][ladders]: the energy found at each temperature level after each round."""
        n = self.ss._host_spins.shape[1]
        L = len(self.levels)
        out = np.zeros((rounds, L, self.nlad))
        for k in range(rounds):
            SamplingHelper.run_(self.ua, sweeps * n, order="sequential", seed=self.seed, step_offset=self.offset,
                                temperatures=np.array([1.0]), steps_per_T=sweeps * n)
            self.offset += sweeps * n
            E = np.asarray(calcEnergy(self.ua)).reshape(self.nlad, L)
            # the state sampled at each level during this round = the slot that held the level BEFORE the swaps
            slot_of = np.argsort(self.level, axis=1)            # slot_of[l, level] = slot holding that level
            lad = np.arange(self.nlad)
            out[k] = E[lad[None, :], slot_of.T]
            # neighbour swaps: even pairs on even rounds, odd pairs on odd rounds
            for lo in range(k & 1, L - 1, 2):
                a, b = slot_of[:, lo], slot_of[:, lo + 1]
                d = (1.0 / self.levels[lo] - 1.0 / self.levels[lo + 1]) * (E[lad, a] - E[lad, b])
                acc = self.rng.random(self.nlad) < np.exp(np.minimum(0.0, d))
                self.proposed[lo] += self.nlad
                self.accepted[lo] += int(acc.sum())
                la = lad[acc]
                self.level[la, a[acc]], self.level[la, b[acc]] = lo + 1, lo
            self._push()
        return out


class DeviceParallelTempering:
    """``ParallelTempering`` with the whole round loop on the device (isb_ssf_run_pt): the same ladder layout (replica =
    ladder * len(levels) + slot), the same ``level[ladder, slot]``, ``accepted`` and ``proposed`` attributes and the same
    ``run`` result, without a host round trip per round.  The swaps draw from the library's counter RNG (``seed``), so
    the trajectory is a pure function of the seed and the absolute round; consecutive ``run`` calls continue it.
    ``order``: "sequential", "random" or "checkerboard" (periodic lattices)."""

    _ORDERS = {"sequential": _lib.ORDER_SEQUENTIAL, "random": _lib.ORDER_RANDOM, "checkerboard": _lib.ORDER_CHECKERBOARD}

    def __init__(self, ua, levels, *, seed=0, order="sequential"):
        self.ua, self.ss = ua, ua.spinSystem
        self.levels = np.asarray(levels, dtype=np.float64)
        L = len(self.levels)
        if L < 1 or self.ss.replicas % L:
            raise ValueError("the number of replicas must be a multiple of the number of temperature levels")
        if order not in self._ORDERS:
            raise ValueError(f"order must be one of {sorted(self._ORDERS)}")
        self.nlad = self.ss.replicas // L
        self.level = np.tile(np.arange(L), (self.nlad, 1))
        self.seed, self.order = int(seed), order
        self.offset = 0          # steps run so far (the Philox step offset of the next round)
        self.round = 0           # rounds run so far (the absolute round index of the next exchange)
        self.accepted = np.zeros(L - 1, dtype=np.int64)
        self.proposed = np.zeros(L - 1, dtype=np.int64)
        ua.temperature = 1.0
        ua.temperatureScale = self.levels[self.level].reshape(-1)

    def run(self, rounds, sweeps=1, *, overlaps=False):
        """Returns E[rounds][levels][ladders]: the energy traced at each temperature level at the end of each round; with
        ``overlaps`` also Q[rounds][levels][ladders/2], the overlap of ladders 2p and 2p+1 at each level."""
        n = self.ss._host_spins.shape[1]
        L = len(self.levels)
        ens = self.ss._ensemble()
        out = ens.ssf_run_pt(self.ua._rule, self.levels, rounds, sweeps * n, order=self._ORDERS[self.order],
                             start=self.offset % n if self.order != "random" else 0, seed=self.seed,
                             step_offset=self.offset, round_offset=self.round, level_of=self.level.reshape(-1),
                             want_Q=overlaps)
        self.ss._dev_newer = True
        K = self.round + np.arange(rounds)
        for lo in range(L - 1):
            self.proposed[lo] += self.nlad * int(np.count_nonzero((K & 1) == (lo & 1)))
        self.accepted += out["accepted"]
        self.level = out["level_of"].reshape(self.nlad, L).astype(np.int64)
        self.offset += rounds * sweeps * n
        self.round += rounds
        self.ua.temperatureScale = self.levels[self.level].reshape(-1)
        return (out["E"], out["Q"]) if overlaps else out["E"]


class PopulationAnnealing:
    """Population annealing with the whole temperature loop on the device (isb_ssf_run_pa).  The replicas of ``ua``'s
    spin system form ``populations`` independent populations of P = replicas / populations slots (population p = replicas
    p*P .. p*P + P - 1).  After the sweeps at each temperature every population is resampled in proportion to
    exp(-(1/T_next - 1/T) E), so that it stays an (approximately) equilibrium sample of the next temperature.

    Bookkeeping kept across ``run`` calls, so that consecutive calls continue one anneal:
      ``family``   [replicas] int32: the slot each replica's family started in (labels follow the resampling);
      ``lnZ``      [populations]: ln Z(T_current) / Z(T_first), from ln Z_{k+1}/Z_k = ln <exp(-(1/T_{k+1} - 1/T_k) E)>;
      ``lnZ_run``  [nT][populations]: ln Z(T[k]) / Z(T_first) at every temperature of the last run;
      ``temperature`` the temperature the populations are at (the last one run, or ``next_temperature``);
      ``offset`` / ``step``: the Philox step offset and the absolute temperature-step index of the next run.
    The resampling draws from the library's counter RNG (``seed``), so the anneal is a pure function of the seed.
    ``order``: "sequential", "random" or "checkerboard" (periodic lattices)."""

    _ORDERS = {"sequential": _lib.ORDER_SEQUENTIAL, "random": _lib.ORDER_RANDOM, "checkerboard": _lib.ORDER_CHECKERBOARD}

    def __init__(self, ua, *, populations=1, seed=0, order="sequential"):
        self.ua, self.ss = ua, ua.spinSystem
        R = self.ss.replicas
        if populations < 1 or R % populations:
            raise ValueError("the number of replicas must be a multiple of the number of populations")
        if order not in self._ORDERS:
            raise ValueError(f"order must be one of {sorted(self._ORDERS)}")
        self.populations, self.P = int(populations), R // int(populations)
        self.seed, self.order = int(seed), order
        self.family = np.arange(R, dtype=np.int32)
        self.lnZ = np.zeros(self.populations)
        self.lnZ_run = np.zeros((0, self.populations))
        self.temperature = None
        self.offset = 0          # steps run so far (the Philox step offset of the next temperature step)
        self.step = 0            # temperature steps run so far (the absolute index of the next one)
        ua.temperatureScale = None    # every replica runs at the schedule's temperature

    def run(self, temperatures, sweeps=1, *, next_temperature=None):
        """``sweeps`` sweeps at each of ``temperatures``, each followed by a resampling towards the next temperature
        (after the last one towards ``next_temperature``, if given).  Returns E[nT][populations][P]: the energy of every
        slot at the end of the sweeps at each temperature, before that step's resampling."""
        T = np.asarray(temperatures, dtype=np.float64).reshape(-1)
        if T.size == 0:
            return np.zeros((0, self.populations, self.P))
        if self.temperature is not None and T[0] != self.temperature:
            raise ValueError(f"the populations are at T = {self.temperature}, not T = {T[0]}: pass next_temperature "
                             "to the previous run to continue at another temperature")
        n = self.ss._host_spins.shape[1]
        ens = self.ss._ensemble()
        ens.set_temperature_scale(None)
        self.ua.temperatureScale = None
        Tn = 0.0 if next_temperature is None else float(next_temperature)
        out = ens.ssf_run_pa(self.ua._rule, self.populations, T, sweeps * n, T_next=Tn, order=self._ORDERS[self.order],
                             start=self.offset % n if self.order != "random" else 0, seed=self.seed,
                             step_offset=self.offset, T_offset=self.step, family=self.family)
        self.ss._dev_newer = True
        self.family = out["family"]
        path = self.lnZ + np.concatenate([np.zeros((1, self.populations)), np.cumsum(out["lnQ"], axis=0)])
        self.lnZ_run = path[:T.size]
        self.lnZ = path[-1]
        self.temperature = T[-1] if next_temperature is None else Tn
        self.offset += T.size * sweeps * n
        self.step += T.size
        return out["E"].reshape(T.size, self.populations, self.P)

    def family_statistics(self):
        """Per population: the number of surviving families, rho_t = P * sum(nu^2) and the family entropy
        -sum(nu ln nu), where nu is the fraction of the population that descends from one initial replica."""
        fams, rho, ent = (np.zeros(self.populations, dtype=np.int64), np.zeros(self.populations),
                          np.zeros(self.populations))
        for p, labels in enumerate(self.family.reshape(self.populations, self.P)):
            nu = np.unique(labels, return_counts=True)[1] / self.P
            fams[p], rho[p], ent[p] = nu.size, self.P * float((nu * nu).sum()), float(-(nu * np.log(nu)).sum())
        return {"families": fams, "rho_t": rho, "entropy": ent}

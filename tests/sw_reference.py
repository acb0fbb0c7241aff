"""numpy replay of the Swendsen-Wang rule of isb_sw_run (include/ising_b200.h) — test infrastructure.

Bond list with the constructor's symmetrise / drop-zero rule, Philox words from oracle_np.philox4x32_10, a CPU labelling
(connected components, root = smallest site), the field grid hq / q, and E, M, sum |C|^2 and flips.  Replicas are
independent, so any subset of an ensemble's replicas can be replayed on its own."""
import numpy as np
import scipy.sparse as sp
from scipy.sparse.csgraph import connected_components

from oracle.oracle_np import philox4x32_10

DOM_SW_BOND, DOM_SW_FLIP = 7, 8
TWO_M32 = 1.0 / 4294967296.0


def bonds(J):
    """(I, Jc, V): the pairs i < j with J_ij != 0, ordered by i then j, as isb_model_sparse stores them (the upper
    triangle defines J_ij; the diagonal and zeros are dropped)."""
    A = sp.csc_matrix(J, dtype=np.float64)
    A.sum_duplicates()
    U = sp.triu(A, 1).tocoo()
    keep = U.data != 0.0
    I, Jc, V = U.row[keep].astype(np.int64), U.col[keep].astype(np.int64), U.data[keep]
    o = np.lexsort((Jc, I))
    return I[o], Jc[o], V[o]


def field_grid(h):
    """(hq int64 [n], q): q = 2^(e_h - 30), e_h the smallest integer with max|h| <= 2^e_h, hq = rint(h / q)."""
    h = np.asarray(h, dtype=np.float64).reshape(-1)
    hmax = float(np.max(np.abs(h))) if h.size else 0.0
    if hmax == 0.0:
        return np.zeros(h.size, dtype=np.int64), 1.0
    f, ex = np.frexp(hmax)
    eh = int(ex) - 1 if f == 0.5 else int(ex)
    q = float(np.ldexp(1.0, eh - 30))
    return np.rint(h / q).astype(np.int64), q


def bond_probability(V, T):
    """1 - exp(-2|J| / T), in the device's operation order."""
    return 1.0 - np.exp((-2.0 * np.abs(V)) / T)


def flip_probability(S, q, T):
    """P = 1 / (1 + exp(2 q S / T)) for the exact cluster sums S."""
    return 1.0 / (1.0 + np.exp((2.0 * q * np.asarray(S, dtype=np.float64)) / T))


def _philox_words(seed, K, reps, dom, count):
    nq = (count + 3) // 4
    c3 = (np.uint32(dom) << np.uint32(28)) | np.arange(nq, dtype=np.uint32)
    w = philox4x32_10(np.uint32(K & 0xFFFFFFFF), np.uint32((K >> 32) & 0xFFFFFFFF),
                      np.asarray(reps, dtype=np.uint32)[:, None], c3[None, :], seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF)
    return np.stack(w, axis=-1).reshape(len(reps), 4 * nq)[:, :count]


def energy(I, Jc, V, h, S):
    """E = -sum_bonds J s_i s_j - sum h s for every row of S."""
    S = S.astype(np.float64)
    return -(S[:, I] * S[:, Jc]) @ V - S @ np.asarray(h, dtype=np.float64)


def sw_replay(J, h, S0, nsweeps, T, seed, *, sweep_offset=0, sweeps_per_T=1, scale=None, replicas=None, trace_every=0):
    """Replay isb_sw_run on the replicas `replicas` (default: all rows of S0).  T: the schedule; scale: the per-replica
    factors of the whole ensemble (or None).  Returns dict(S, E, M, csq [ntr][nr], flips [nr])."""
    S0 = np.asarray(S0, dtype=np.int8)
    reps = np.arange(S0.shape[0]) if replicas is None else np.asarray(replicas, dtype=np.int64)
    s = S0[reps].astype(np.int64)
    nr, n = s.shape
    I, Jc, V = bonds(J)
    hq, q = field_grid(h)
    has_h = bool(np.any(hq != 0))
    T = np.asarray(T, dtype=np.float64).reshape(-1)
    tsc = np.ones(nr) if scale is None else np.asarray(scale, dtype=np.float64)[reps]
    ntr = nsweeps // trace_every if trace_every > 0 else 0
    E, M, csq = np.zeros((ntr, nr)), np.zeros((ntr, nr)), np.zeros((ntr, nr), dtype=np.int64)
    flips = np.zeros(nr, dtype=np.int64)
    node = np.arange(nr * n)
    for k in range(nsweeps):
        K = sweep_offset + k
        Tr = T[k // sweeps_per_T] * tsc                                   # [nr]
        w = _philox_words(seed, K, reps, DOM_SW_BOND, V.size)            # [nr][nb]
        u = (w.astype(np.float64) + 0.5) * TWO_M32
        same = s[:, I] == s[:, Jc]
        active = ((V[None, :] > 0.0) == same) & (u < bond_probability(V[None, :], Tr[:, None]))
        rr, ee = np.nonzero(active)
        G = sp.coo_matrix((np.ones(rr.size), (rr * n + I[ee], rr * n + Jc[ee])), shape=(nr * n, nr * n)).tocsr()
        ncomp, lab = connected_components(G, directed=False)
        root = np.full(ncomp, nr * n, dtype=np.int64)
        np.minimum.at(root, lab, node)
        z = _philox_words(seed, K, reps, DOM_SW_FLIP, n)                 # word of site rho, used at roots
        uz = (z.astype(np.float64) + 0.5) * TWO_M32
        if has_h:
            Ssum = np.zeros(ncomp, dtype=np.int64)
            np.add.at(Ssum, lab, (hq[None, :] * s).reshape(-1))
            comp_rep = root // n
            P = flip_probability(Ssum, q, Tr[comp_rep])
        else:
            P = np.full(ncomp, 0.5)
        flip_comp = uz.reshape(-1)[root] < P
        f = flip_comp[lab].reshape(nr, n)
        s = np.where(f, -s, s)
        flips += f.sum(axis=1)
        if trace_every > 0 and (k + 1) % trace_every == 0:
            t = (k + 1) // trace_every - 1
            E[t] = energy(I, Jc, V, h, s)
            M[t] = s.sum(axis=1)
            sizes = np.bincount(lab, minlength=ncomp).astype(np.float64)
            csq[t] = np.bincount(root // n, weights=sizes * sizes, minlength=nr).astype(np.int64)   # (exact below 2^53)
    return {"S": s.astype(np.int8), "E": E, "M": M, "csq": csq, "flips": flips}


def transition_matrix(J, h, T):
    """The full SW transition matrix of a tiny model (n <= ~8) by enumeration: every subset of the bonds that may be active
    (J_ij s_i s_j > 0) with its probability, every cluster-flip outcome with its heat-bath probability.  Also returns the
    Boltzmann weights of the grid fields q hq."""
    I, Jc, V = bonds(J)
    hq, q = field_grid(h)
    n = hq.size
    states = ((np.arange(1 << n)[:, None] >> np.arange(n)[None, :]) & 1) * 2 - 1
    index = lambda st: int(((st > 0).astype(np.int64) << np.arange(n)).sum())   # noqa: E731
    P = np.zeros((1 << n, 1 << n))
    pb = bond_probability(V, T)
    for a, s in enumerate(states):
        cand = np.nonzero((V > 0.0) == (s[I] == s[Jc]))[0]
        for mask in range(1 << cand.size):
            on = np.array([(mask >> b) & 1 for b in range(cand.size)], dtype=bool)
            pr = float(np.prod(np.where(on, pb[cand], 1.0 - pb[cand]))) if cand.size else 1.0
            if pr == 0.0:
                continue
            act = cand[on]
            G = sp.coo_matrix((np.ones(act.size), (I[act], Jc[act])), shape=(n, n)).tocsr()
            nc, lab = connected_components(G, directed=False)
            Sc = np.zeros(nc, dtype=np.int64)
            np.add.at(Sc, lab, hq * s)
            pf = flip_probability(Sc, q, T)
            for fm in range(1 << nc):
                fl = np.array([(fm >> c) & 1 for c in range(nc)], dtype=bool)
                pc = float(np.prod(np.where(fl, pf, 1.0 - pf)))
                t = np.where(fl[lab], -s, s)
                P[a, index(t)] += pr * pc
    Eg = -(states[:, I] * states[:, Jc]) @ V - states @ (q * hq.astype(np.float64))
    w = np.exp(-(Eg - Eg.min()) / T)
    return P, w / w.sum()

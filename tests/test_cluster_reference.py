"""CPU checks of the Swendsen-Wang rule of isb_sw_run (tests/sw_reference.py): the full transition matrix of three tiny
models leaves the Boltzmann distribution of the grid fields invariant, which pins down the rule's field and sign handling
independently of the device; and the field grid on its edge cases."""
import numpy as np
import pytest
import scipy.sparse as sp

from sw_reference import bonds, field_grid, sw_replay, transition_matrix


def _sym(n, entries):
    A = np.zeros((n, n))
    for i, j, v in entries:
        A[i, j] = A[j, i] = v
    return sp.csc_matrix(A)


CASES = {
    # 4-cycle ferromagnet, no field
    "cycle4": (_sym(4, [(0, 1, 1.0), (1, 2, 1.0), (2, 3, 1.0), (0, 3, 1.0)]), np.zeros(4), 1.3),
    # 2 x 3 grid with mixed-sign couplings and non-dyadic fields
    "grid2x3": (_sym(6, [(0, 1, 0.7), (1, 2, -1.1), (3, 4, 0.45), (4, 5, 1.3), (0, 3, -0.6), (1, 4, 0.9), (2, 5, 0.35)]),
                np.array([0.3, -0.17, 0.0, 0.55, -0.41, 0.123]), 0.9),
    # frustrated antiferromagnetic triangle in a field
    "triangle": (_sym(3, [(0, 1, -1.0), (1, 2, -1.0), (0, 2, -1.0)]), np.array([0.4, 0.4, 0.4]), 0.7),
}


@pytest.mark.parametrize("name", sorted(CASES))
def test_transition_matrix_keeps_the_boltzmann_distribution(name):
    J, h, T = CASES[name]
    P, pi = transition_matrix(J, h, T)
    assert np.allclose(P.sum(axis=1), 1.0, rtol=0, atol=1e-12)
    assert np.max(np.abs(pi @ P - pi)) < 1e-12
    # and the chain is not the identity: it moves between configurations
    assert np.max(np.diag(P)) < 1.0


def test_field_grid_edge_cases():
    hq, q = field_grid(np.array([0.5, -0.25, 0.1]))          # max|h| an exact power of two: e_h = -1
    assert q == 2.0 ** -31 and hq[0] == 1 << 30 and hq[1] == -(1 << 29)
    assert abs(hq[2] * q - 0.1) <= q / 2
    hq, q = field_grid(np.zeros(5))                            # h = 0: every hq_i is 0
    assert not hq.any()
    hq, q = field_grid(np.array([0.0, 0.0, -3.0, 0.0]))       # a single non-zero field: e_h = 2
    assert q == 2.0 ** -28 and list(hq) == [0, 0, -3 * (1 << 28), 0]
    assert np.abs(field_grid(np.array([0.3, -0.7]))[0]).max() <= 1 << 30


def test_bond_order_follows_the_constructor():
    # a non-symmetric input: the upper triangle defines J; the diagonal and explicit zeros are dropped
    A = sp.csc_matrix(np.array([[5.0, 0.0, 2.0], [9.0, 0.0, -1.0], [0.0, 0.0, 1.0]]))
    I, Jc, V = bonds(A)
    assert list(zip(I, Jc, V)) == [(0, 2, 2.0), (1, 2, -1.0)]


def test_replay_continues_and_subsets():
    """Two replay calls with the sweep offset continued equal one; a subset of replicas replays on its own."""
    J = _sym(6, [(0, 1, 0.7), (1, 2, -1.1), (3, 4, 0.45), (4, 5, 1.3), (0, 3, -0.6), (1, 4, 0.9), (2, 5, 0.35)])
    h = np.array([0.3, -0.17, 0.0, 0.55, -0.41, 0.123])
    S0 = np.where(np.random.default_rng(1).random((5, 6)) < 0.5, -1, 1).astype(np.int8)
    one = sw_replay(J, h, S0, 8, [1.1], 7, sweeps_per_T=8, trace_every=1)
    a = sw_replay(J, h, S0, 3, [1.1], 7, sweeps_per_T=3)
    b = sw_replay(J, h, a["S"], 5, [1.1], 7, sweep_offset=3, sweeps_per_T=5)
    assert np.array_equal(one["S"], b["S"]) and np.array_equal(one["flips"], a["flips"] + b["flips"])
    sub = sw_replay(J, h, S0, 8, [1.1], 7, sweeps_per_T=8, replicas=[3, 1])
    assert np.array_equal(sub["S"], one["S"][[3, 1]])
    assert np.all(one["csq"] >= 6) and np.all(one["csq"] <= 36)

"""Inputs of the golden cases whose big matrices are regenerated from seeds (see tests/golden/make_golden.py)."""
import numpy as np


def golden_J(name, g, synth):
    if "J" in g:
        return g["J"]
    if name == "ssf_c1_32x32_metropolis":
        J = synth.lattice_J(32)
    elif name == "ssf_c2_sk1024_glauber":
        J = synth.sk_J(1024, 2)
    else:
        raise KeyError(name)
    from conftest import sha
    assert sha(J) == str(g["J_sha"]), "synthetic J drifted from the one the golden file was made with"
    return J


def golden_W(name, g, synth):
    if "W" in g:
        return g["W"]
    if name.startswith("bip_c4_784x512"):
        W, _, _ = synth.bipartite_W(784, 512, 4)
    else:
        raise KeyError(name)
    from conftest import sha
    assert sha(W) == str(g["W_sha"]), "synthetic W drifted from the one the golden file was made with"
    return W


SSF_GOLDEN = ["ssf_2spin_hopfield", "ssf_2spin_glauber", "ssf_2spin_metropolis", "ssf_3x3_glauber",
              "ssf_3x3_metropolis", "ssf_c1_32x32_metropolis", "ssf_sk64_glauber", "ssf_sk64_hopfield",
              "ssf_c2_sk1024_glauber"]
BIP_GOLDEN = ["bip_2x3_sca", "bip_2x3_ma", "bip_24x17_sca", "bip_24x17_ma", "bip_c4_784x512_sca",
              "bip_c4_784x512_ma"]


def commensurate_J(synth, n, seed):
    """Couplings +-0.1 / +-0.3 on about a fifth of the pairs (symmetric, zero diagonal): sums that round and cancel
    exactly, so that an incrementally maintained Float64 field and the reference's fresh row dot disagree at exact ties.
    The model runs the sweep kernels' near-tie guard (GUARD) and the fixed-point exact fallback on it."""
    g = synth.gaussian(seed, n * n).reshape(n, n)
    J = np.where(g > 0.8, 0.3, np.where(g > 0.0, 0.1, np.where(g > -0.8, -0.1, -0.3)))
    J = np.where(np.abs(synth.gaussian(seed + 1, n * n).reshape(n, n)) < 0.25, J, 0.0)
    J = np.triu(J, 1)
    return J + J.T


# The near-tie guard cases of tests/test_gpu_ssf_variants.py: T = 0 dynamics, h = 0, GUARD_SWEEPS sweeps in runs of
# GUARD_PER sweeps (each run after the first starts with a field refresh).  tests/test_ssf_float_twin.py checks on the CPU
# that on these inputs the unguarded incremental Float64 dynamics leaves the reference.
GUARD_R, GUARD_SWEEPS, GUARD_PER = 12, 300, 75


def guard_case(synth, n):
    return commensurate_J(synth, n, 91 + n), np.zeros(n), synth.spins(94 + n, GUARD_R, n)


def nodes_of(g):
    return None if g["nodes"].size == 0 else g["nodes"].astype(np.int32)

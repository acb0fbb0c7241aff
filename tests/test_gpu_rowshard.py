"""GPU tests of the row-sharded synchronous SCA (BASELINE config 5): the result must not depend on the number of
row blocks, must equal the unsharded tensor-core path (itself checked against the oracle), and the NCCL
all-gather variants (2, 4 and 8 processes, one per GPU) must equal the single-process emulation."""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _unsharded(L, ctx, W, hhalf, S0, nsteps, T, seed, prec, rule=0):
    R, n = S0.shape
    e = L.Ensemble(L.Model.bipartite(ctx, W, hhalf, hhalf, prec), R)
    e.set_spins(S0)
    e.set_hidden(S0)
    e.bip_run(rule, nsteps, seed=seed, T=T)
    return e.get_spins(), e.get_hidden()


@pytest.mark.parametrize("kind", ["int", "gauss"])
def test_blocks_do_not_change_the_trajectory(pkg, ctx, synth, kind):
    from isingmodel_jl_b200 import _lib as L, rowshard
    n, R, nsteps, seed = 256, 150, 5, 11
    if kind == "int":
        J = np.round(synth.sk_J(n, 5) * 30.0)
        prec = L.PREC_BF16X1
    else:
        J = synth.sk_J(n, 5)
        prec = L.PREC_BF16X3
    h = np.round(synth.gaussian(6, n)) if kind == "int" else synth.gaussian(6, n) * 0.1
    q = 2.0
    W = 0.5 * (J + q * np.eye(n))
    S0 = synth.spins(7, R, n)
    T = synth.geometric_schedule(2.0, 0.3, nsteps)
    ref_v, ref_h = _unsharded(L, ctx, W, 0.5 * h, S0, nsteps, T, seed, prec)
    for G in (1, 2, 4):
        sca = rowshard.RowShardedSCA(n, R, W=W, h=h, prec=prec, emulate_blocks=G)
        sca.set_spins(S0)
        sca.run(nsteps, T, seed=seed)
        assert np.array_equal(sca.get_spins(), ref_v), f"G={G}"
        assert np.array_equal(sca.get_hidden(), ref_h), f"G={G}"


def test_momentum_annealing_rule_sharded(pkg, ctx, synth):
    from isingmodel_jl_b200 import _lib as L, rowshard
    n, R, nsteps, seed = 128, 64, 4, 3
    J = np.round(synth.sk_J(n, 8) * 20.0)
    W = 0.5 * (J + 2.0 * np.eye(n))
    S0 = synth.spins(9, R, n)
    T = np.full(nsteps, 1.5)
    ref_v, ref_h = _unsharded(L, ctx, W, np.zeros(n), S0, nsteps, T, seed, L.PREC_BF16X1, rule=1)
    sca = rowshard.RowShardedSCA(n, R, W=W, rule=L.BIP_MA, prec=L.PREC_BF16X1, emulate_blocks=2)
    sca.set_spins(S0)
    sca.run(nsteps, T, seed=seed)
    assert np.array_equal(sca.get_spins(), ref_v) and np.array_equal(sca.get_hidden(), ref_h)


def test_synthetic_sk_rows_and_generated_model(pkg, ctx, synth):
    from isingmodel_jl_b200 import _lib as L, rowshard
    n, R, seed = 512, 40, 99
    J = ctx.sk_rows(n, seed, 0, n)
    assert np.array_equal(J, J.T) and not np.diag(J).any()
    assert abs(J.std() * np.sqrt(n) - 1.0) < 0.02 and abs(J.mean()) < 3.0 / n
    assert np.array_equal(ctx.sk_rows(n, seed, 100, 7), J[100:107])
    q = 1.0
    S0 = synth.spins(1, R, n)
    T = np.array([1.0, 0.7, 0.4])
    a = rowshard.RowShardedSCA(n, R, seed=seed, q=q, emulate_blocks=4)       # generated on the device per block
    b = rowshard.RowShardedSCA(n, R, W=0.5 * (J + q * np.eye(n)), emulate_blocks=2)  # same matrix passed in
    for s in (a, b):
        s.set_spins(S0)
        s.run(3, T, seed=5)
    assert np.array_equal(a.get_spins(), b.get_spins())
    # the energy of the embedded model decreases under annealing (sanity of the dynamics)
    E0 = -0.5 * np.einsum("ri,ij,rj->r", S0.astype(float), J, S0.astype(float))
    S1 = a.get_spins().astype(float)
    E1 = -0.5 * np.einsum("ri,ij,rj->r", S1, J, S1)
    assert E1.mean() < E0.mean()


@pytest.mark.parametrize("prec_name,rule", [("i8x3", 0), ("bf16x3", 0), ("i8x3", 1)])
def test_step_loop_inside_the_library_single_block(pkg, ctx, synth, prec_name, rule):
    """isb_shard_run_* with one block (ISB_EXCH_LOCAL): the C step loop equals the Python-driven half-steps."""
    from isingmodel_jl_b200 import _lib as L, rowshard
    prec = {"i8x3": L.PREC_I8X3, "bf16x3": L.PREC_BF16X3}[prec_name]
    n, R, nsteps = 256, 300, 5
    S0 = synth.spins(21, R, n)
    T = synth.geometric_schedule(1.5, 0.3, nsteps)
    emu = rowshard.RowShardedSCA(n, R, seed=31, q=1.0, prec=prec, rule=rule, emulate_blocks=2)
    emu.set_spins(S0)
    emu.run(nsteps, T, seed=9, step_offset=3)
    abi = rowshard.ShardRunSCA(n, R, seed=31, q=1.0, prec=prec, rule=rule)
    assert abi.exchange == "local"
    abi.set_spins(S0)
    st = abi.run(nsteps, T, seed=9, step_offset=3)
    assert st["launches"] == 2 * nsteps
    assert np.array_equal(abi.get_spins(), emu.get_spins()) and np.array_equal(abi.get_hidden(), emu.get_hidden())
    abi.run(2, T[-1:], seed=9, step_offset=3 + nsteps)          # continues from the device state
    emu.run(2, T[-1:], seed=9, step_offset=3 + nsteps)
    assert np.array_equal(abi.get_spins(), emu.get_spins())


@pytest.mark.parametrize("ranks", [2, 4, 8])
def test_nccl_all_gather_ranks(pkg, ctx, ranks):
    """One process per GPU under torchrun: every exchange mode (NCCL all-gather, the two-group pipeline, copy-engine pushes,
    peer stores in the epilogue, and the library's own isb_shard_run_* loops) against the single-process emulation."""
    import torch
    if torch.cuda.device_count() < ranks:
        pytest.skip(f"needs {ranks} GPUs")
    res = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={ranks}",
                          "--master-addr", "127.0.0.1", "--master-port", str(29671 + ranks),
                          os.path.join(ROOT, "tests", "rowshard_worker.py")], capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    assert "ROWSHARD-OK" in res.stdout

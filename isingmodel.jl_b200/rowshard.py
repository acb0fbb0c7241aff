"""Row-sharded synchronous SCA over the GPUs of one box (BASELINE config 5, SURVEY §8e).

The MultiSpinFlip SCA of an N-spin model is the bipartite SCA (reference: src/OnBipartiteGraph.jl:30-43) on the
embedding W = (J + qI)/2, sigma = tau = s (demo.jl:82-90).  When W does not fit one GPU, rank g owns the output
units [g*nb, (g+1)*nb) of both half-steps and W[block rows, :]; after every half-step the freshly sampled
[R][nb] blocks are exchanged into the block-major [G][R][nb] matrix that is the next half-step's K operand.

Multi-GPU runs go through ``ShardRunSCA``, whose step loop and exchange live in the library (isb_shard_run_*).
``RowShardedSCA`` plays all G row blocks in turn in one process on one GPU: the library's noise is indexed by global
(replica, step, unit), so the trajectory does not depend on G, and the tests use it as the reference for G > 1.
"""
from __future__ import annotations

import numpy as np

from . import _lib


class RowShardedSCA:
    def __init__(self, n: int, R: int, *, emulate_blocks: int, seed: int | None = None, q: float = 1.0, W=None, h=None,
                 rule=_lib.BIP_SCA, prec=_lib.PREC_BF16X3, device: int | None = None):
        import torch

        self.torch = torch
        self.n, self.R, self.rule = int(n), int(R), rule
        self.G = int(emulate_blocks)
        if self.n % self.G:
            raise ValueError("n must be divisible by the number of blocks")
        self.nb = self.n // self.G
        self.ctx = _lib.context(device)
        self.dev = torch.device("cuda", self.ctx.device)
        torch.cuda.set_device(self.dev)
        self.ctx.set_stream(torch.cuda.current_stream(self.dev).cuda_stream)
        # operand format of the spin matrices: int8 +-1 for the int8 digit-plane models, else bf16
        self.dtype = torch.int8 if prec in _lib.I8_PRECS else torch.bfloat16
        self.models = []
        wmax = 0.0
        if W is not None and prec in _lib.I8_PRECS:
            # the fixed-point grid must be the same for every block: the largest off-diagonal |W| of the whole matrix
            Wa = np.abs(np.asarray(W, dtype=np.float64))
            wmax = float((Wa - np.diag(np.diag(Wa))).max())
        for g in range(self.G):
            if W is not None:
                Wg = np.asarray(W, dtype=np.float64)[g * self.nb:(g + 1) * self.nb, :]
                hb = None if h is None else 0.5 * np.asarray(h, dtype=np.float64)[g * self.nb:(g + 1) * self.nb]
                self.models.append(_lib.Model.shard_rows(self.ctx, self.n, self.G, g, Wg, hb, hb, prec, wmax=wmax))
            else:
                self.models.append(_lib.Model.shard_sk(self.ctx, self.n, self.G, g, int(seed), q, prec))
        # the visible and hidden layers, block-major [G][R][nb]; block g samples in place into its slab
        self.full_v = torch.zeros((self.G, self.R, self.nb), dtype=self.dtype, device=self.dev)
        self.full_h = torch.zeros((self.G, self.R, self.nb), dtype=self.dtype, device=self.dev)

    def set_spins(self, S):
        """S: (R, n) int8 +-1; the embedding starts from sigma = tau = s."""
        S = self.torch.as_tensor(np.ascontiguousarray(S, dtype=np.int8), device=self.dev)
        full = S.view(self.R, self.G, self.nb).permute(1, 0, 2).to(self.dtype)
        self.full_v.copy_(full)
        self.full_h.copy_(full)

    def _layer(self, full):
        s = (full > 0).to(self.torch.int8) * 2 - 1
        return s.permute(1, 0, 2).reshape(self.R, self.n).cpu().numpy()

    def get_spins(self):
        """(R, n) int8 visible layer."""
        return self._layer(self.full_v)

    def get_hidden(self):
        return self._layer(self.full_h)

    def run(self, nsteps, T, *, seed=0, step_offset=0):
        """nsteps synchronous SCA steps; T: array of nsteps temperatures (T[k] applies to step k)."""
        T = np.atleast_1d(np.asarray(T, dtype=np.float64))
        for k in range(int(nsteps)):
            Tk = float(T[min(k, len(T) - 1)])
            for layer in (1, 0):   # hidden from the visible layer, then visible from the hidden layer
                src, dst = (self.full_v, self.full_h) if layer == 1 else (self.full_h, self.full_v)
                # a half-step reads only src and its own slab of dst (MomentumAnnealing's previous values)
                for g, m in enumerate(self.models):
                    m.shard_halfstep(self.R, layer, self.rule, src.data_ptr(), dst[g].data_ptr(), seed, step_offset + k, Tk)


class ShardRunSCA:
    """The row-sharded SCA, one process per GPU, with the step loop inside the library (isb_shard_run_*,
    include/ising_b200.h): the two replica groups, the exchange after every half-step (``exchange="nccl"``:
    ncclAllGather through the library's own communicator; ``"copy"``: copy-engine pushes into IPC-mapped peer matrices
    + stream memory operations) and their ordering run in C; torch.distributed only carries the 128-byte NCCL id / the
    64-byte IPC handles between the ranks at construction.  What a C or Julia caller of the row-sharded path executes,
    step for step."""

    def __init__(self, n: int, R: int, *, seed: int | None = None, q: float = 1.0, W=None, h=None, rule=_lib.BIP_SCA,
                 prec=_lib.PREC_I8X3, device: int | None = None, group=None, exchange: str = "copy"):
        import torch.distributed as dist
        self.n, self.R, self.rule = int(n), int(R), rule
        self.distributed = dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1
        self.G = dist.get_world_size(group) if self.distributed else 1
        g = dist.get_rank(group) if self.distributed else 0
        if self.n % self.G:
            raise ValueError("n must be divisible by the number of blocks")
        self.nb = self.n // self.G
        self.ctx = _lib.context(device)
        if W is not None:
            Wa = np.asarray(W, dtype=np.float64)
            wmax = float((np.abs(Wa) - np.diag(np.abs(np.diag(Wa)))).max()) if prec in _lib.I8_PRECS else 0.0
            hb = None if h is None else 0.5 * np.asarray(h, dtype=np.float64)[g * self.nb:(g + 1) * self.nb]
            self.model = _lib.Model.shard_rows(self.ctx, self.n, self.G, g, Wa[g * self.nb:(g + 1) * self.nb, :], hb, hb, prec, wmax=wmax)
        else:
            self.model = _lib.Model.shard_sk(self.ctx, self.n, self.G, g, int(seed), q, prec)
        code = {"nccl": _lib.EXCH_NCCL, "copy": _lib.EXCH_COPY}[exchange] if self.distributed else _lib.EXCH_LOCAL
        self.exchange = "abi-" + exchange if self.distributed else "local"
        self.run_obj = _lib.ShardRun(self.model, self.R, code)
        if self.distributed:
            self.run_obj.wire(dist, group)
        self.launches = 0

    def set_spins(self, S):
        self.run_obj.set_spins(S)

    def get_spins(self):
        return self.run_obj.get_spins(0)

    def get_hidden(self):
        return self.run_obj.get_spins(1)

    def run(self, nsteps, T, *, seed=0, step_offset=0):
        self.run_obj.steps(self.rule, nsteps, T, seed=seed, step_offset=step_offset)
        st = self.run_obj.last_stats()
        self.launches += st["launches"]
        return st

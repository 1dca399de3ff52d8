"""One process per GPU: sharded direct J/K with one all-reduce per Fock build (SURVEY.md section 8e).

J and K are linear in the integrals, so any partition of the unique-quartet list gives partial J/K that sum.
Every rank holds the whole pair table and density; rank r evaluates the chunks c with c % nranks == r of every job's work list
(`shard_chunks`; mirrored on the device by k_shell4_one / k_shell4_multi with one CTA work unit of 2-16 work items per group per chunk and by
k_jk_direct with 1024 AO quartets per chunk, csrc/tuna_b200.cu), and the partial (J, K) stack — 2 * nD * nbf^2
doubles — is summed with ONE NCCL all-reduce on the compute stream.  torch is plumbing here: device buffers,
the stream, and torch.distributed.
"""
import numpy as np

CHUNK = 128    # items per scheduling chunk of the host-side model of the sharding (tests/test_distributed_cpu.py)


def shard_chunks(n_quartets: int, rank: int, nranks: int, chunk: int = CHUNK):
    """Chunk indices owned by `rank`: round-robin over the class-sorted quartet list (cost-balanced because
    neighbouring chunks have neighbouring angular classes)."""
    nchunks = (n_quartets + chunk - 1) // chunk
    return range(rank, nchunks, nranks)


class FockBuilder:
    """Direct-mode J/K for a fixed geometry on this rank's GPU; `build` is the call a user makes per SCF iteration.

    P (host, float64, (nD, nbf, nbf) or (nbf, nbf)) -> J, K (host).  Every step copies P host->device from pinned
    memory, runs the sharded kernels, all-reduces the partial J/K over ranks (if any) and reads J/K back.
    """

    def __init__(self, ctx, nD=1, tau=1e-16, group=None):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.ctx, self.nD, self.tau, self.group = ctx, nD, tau, group
        self.world = dist.get_world_size(group) if dist.is_available() and dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if self.world > 1 else 0
        self.device = torch.device("cuda", ctx.device)
        n = ctx.nbf
        self.n = n
        self.stream = torch.cuda.Stream(device=self.device)
        ctx.set_stream(self.stream.cuda_stream)
        ctx.set_shard(self.rank, self.world)
        self.dP = torch.empty((nD, n, n), dtype=torch.float64, device=self.device)
        self.dJK = torch.empty((2, nD, n, n), dtype=torch.float64, device=self.device)
        self.hP = torch.empty((nD, n, n), dtype=torch.float64).pin_memory()
        self.hJK = torch.empty((2, nD, n, n), dtype=torch.float64).pin_memory()
        self.h2d_bytes = self.hP.numel() * 8
        self.d2h_bytes = self.hJK.numel() * 8

    def build_device(self):
        """Kernels + collective only: inputs already in HBM (self.dP), result left in self.dJK.  Enqueues on self.stream."""
        self.ctx.set_stream(self.stream.cuda_stream)      # several builders (e.g. nD = 1 and nD = 2) may share one context
        self.ctx.jk_direct_dev(self.nD, self.dP.data_ptr(), self.dJK[0].data_ptr(), self.dJK[1].data_ptr(), self.tau)
        if self.world > 1:
            with self.torch.cuda.stream(self.stream):
                self.dist.all_reduce(self.dJK, group=self.group)

    def build(self, P):
        P = np.asarray(P, dtype=np.float64)
        single = P.ndim == 2
        Ps = P.reshape(self.nD, self.n, self.n)
        # build_device (tuna_jk_direct_dev) takes every density as symmetric.  A guess density can be asymmetric at the 1e-8 level;
        # such a P goes through tuna_jk_direct_general_dev, which splits it into symmetric and antisymmetric parts on the device (same
        # 1e-15 relative test, bitwise the J and K of tuna_jk_direct) and honours the shard, so its partial J/K are all-reduced alike.
        general = np.abs(Ps - Ps.transpose(0, 2, 1)).max() > 1e-15 * np.abs(Ps).max()
        self.hP.numpy()[...] = Ps
        with self.torch.cuda.stream(self.stream):
            self.dP.copy_(self.hP, non_blocking=True)
            if general:
                self.ctx.set_stream(self.stream.cuda_stream)
                self.ctx.jk_direct_general_dev(self.nD, self.dP.data_ptr(), self.dJK[0].data_ptr(), self.dJK[1].data_ptr(), self.tau)
                if self.world > 1:
                    self.dist.all_reduce(self.dJK, group=self.group)
            else:
                self.build_device()
            self.hJK.copy_(self.dJK, non_blocking=True)
        self.stream.synchronize()
        J, K = self.hJK.numpy()[0].copy(), self.hJK.numpy()[1].copy()
        return (J[0], K[0]) if single else (J, K)

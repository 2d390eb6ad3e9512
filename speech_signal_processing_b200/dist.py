"""One process per GPU: sharding helpers and the NCCL hooks of the hot path (SURVEY 8(e)).

* front-end / scoring / enrolment shard whole utterances (or speakers) across ranks: no data-path
  collective; rank 0 gathers the small (N, S) score matrix or just the argmax;
* UBM EM shards frames; each iteration all-reduces ONE flat float64 tensor
  ``[N (K), F (K*D), S (K*D), loglik, n_frames]`` (324 KB at K=512, D=39) over NCCL/NVLink and
  every rank runs the replicated M-step kernel.
"""
from __future__ import annotations

import os

import numpy as np


def shard_range(n: int, rank: int, world: int):
    """Contiguous block [lo, hi) of n items for this rank (sizes differ by at most one)."""
    base, rem = divmod(n, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def shard_by_load(lengths, world: int):
    """Assign items to ranks balancing the sum of ``lengths`` (longest-first greedy).  Returns a list
    of index arrays, each sorted ascending so that per-rank order stays the input order."""
    lengths = np.asarray(lengths, dtype=np.int64)
    order = np.argsort(-lengths, kind="stable")
    load = np.zeros(world, dtype=np.int64)
    out = [[] for _ in range(world)]
    for i in order:
        r = int(np.argmin(load))
        out[r].append(int(i))
        load[r] += lengths[i]
    return [np.array(sorted(ix), dtype=np.int64) for ix in out]


class Comm:
    """Thin wrapper over ``torch.distributed`` (NCCL on GPUs, gloo in the CPU tests)."""

    def __init__(self, backend: str | None = None):
        import torch
        import torch.distributed as dist

        self.dist = dist
        if not dist.is_initialized():
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            os.environ.setdefault("MASTER_PORT", "29511")
            backend = backend or ("nccl" if torch.cuda.is_available() else "gloo")
            if backend == "nccl":
                torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
            dist.init_process_group(backend=backend, rank=int(os.environ.get("RANK", "0")),
                                    world_size=int(os.environ.get("WORLD_SIZE", "1")))
        self.rank, self.world_size = dist.get_rank(), dist.get_world_size()

    def allreduce_sum(self, t):
        if self.world_size > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return t

    def allreduce_max(self, t):
        if self.world_size > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return t

    def broadcast(self, t, src: int = 0):
        if self.world_size > 1:
            self.dist.broadcast(t, src=src)
        return t

    def barrier(self):
        if self.world_size > 1:
            self.dist.barrier()

    def gather_rows(self, local, counts):
        """Concatenate per-rank row blocks (rank r holds counts[r] rows) on every rank."""
        import torch

        if self.world_size == 1:
            return local
        m = int(max(counts))
        pad = torch.zeros((m,) + tuple(local.shape[1:]), dtype=local.dtype, device=local.device)
        pad[: local.shape[0]] = local
        bufs = [torch.empty_like(pad) for _ in range(self.world_size)]
        self.dist.all_gather(bufs, pad)
        return torch.cat([b[: int(c)] for b, c in zip(bufs, counts)], dim=0)


def fit_ubm_sharded(comm: Comm, local_frames, n_components: int, **kw):
    """UBM EM with frames sharded across ranks; statistics all-reduced every iteration."""
    from .mixture import GaussianMixture

    gm = GaussianMixture(n_components=n_components, covariance_type="diag", comm=comm, **kw)
    return gm.fit(local_frames)


def map_enrol_sharded(comm: Comm, ubm, speaker_frames, relevance: float = 16.0):
    """Mean-only MAP enrolment with SPEAKERS sharded across ranks (each speaker's frames stay on one rank); the adapted
    means (S x K x D float64, 160 MB at S = 1000, K = 1024, D = 39) are all-gathered so that every rank ends up with
    the same replicated :class:`SharedModelSet` (UBM means appended as model S).  No collective on the frame data."""
    import torch

    from .mixture import SharedModelSet
    from .ubm import map_adapt

    n_spk = len(speaker_frames)
    lo, hi = shard_range(n_spk, comm.rank, comm.world_size)
    uw, umu, uvar = ubm._model_set()._params
    k, d = umu.shape[1], umu.shape[2]
    if hi > lo:
        _, mu, _ = map_adapt(ubm, speaker_frames[lo:hi], relevance=relevance, adapt=("means",))
    else:
        mu = torch.empty((0, k, d), dtype=torch.float64, device=umu.device)
    counts = [shard_range(n_spk, r, comm.world_size) for r in range(comm.world_size)]
    means = comm.gather_rows(mu, [b - a for a, b in counts])
    return SharedModelSet.with_ubm(uw[0], uvar[0], means, umu, device=umu.device)


def identify_sharded(comm: Comm, utts, speakers, ubm=None, precision="auto"):
    """Each rank scores its contiguous block of utterances against ALL (replicated) speaker models;
    every rank returns the full (N, S) LLR matrix and decisions."""
    import torch

    from .ubm import identify

    lo, hi = shard_range(len(utts), comm.rank, comm.world_size)
    pred, _ = identify(utts[lo:hi], speakers, ubm, precision=precision)
    counts = [shard_range(len(utts), r, comm.world_size) for r in range(comm.world_size)]
    counts = [b - a for a, b in counts]
    full = comm.gather_rows(torch.as_tensor(pred, device="cuda"), counts).cpu().numpy()
    return full, full.argmax(axis=1)

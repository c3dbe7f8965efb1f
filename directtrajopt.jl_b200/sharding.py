"""Multi-GPU partitioning of the evaluator (SURVEY.md section 8e), one process per GPU.

  partitioning A (independent problems, BASELINE config c5): ``split_batch`` gives each rank a contiguous
      block of problems; no communication on the data path at all.
  partitioning B (one long trajectory, config c4): ``ShardedEvaluator`` gives rank r the contiguous knot
      range ``knot_ranges(N, world)[r]``.  Every interval needs knots k and k+1, so a rank needs ONE halo
      knot (z doubles) of its right neighbour.  Linked shards (``peer_halo``) move it over NVLink P2P inside the
      evaluation stream: after uploading an iterate a rank pushes its first knot into the left neighbour's exchange
      window (CUDA-IPC mapped HBM) and flags it; the neighbour's kernels wait for the flag on the device
      (csrc/shard_link.cu).  Protocol: every rank calls ``upload`` (or ``upload_dev``) once per iterate.
      Time-dependent bilinear integrators with ``spline_order = 1`` read u_{k+1} on interval k, so interval k0 - 1
      of the left neighbour adds to the Hessian of this rank's first knot: every Hessian evaluation, the left neighbour
      pushes its last interval's compact second derivatives into this rank's window, and this rank assembles its
      first knot after they arrive (bit-identical to the unsharded Hessian).  Every rank then evaluates every Hessian
      (evaluation s of a rank reads evaluation s of its left neighbour); an unlinked such shard has no Hessian.
      The two scalars every rank needs -- objective (sum) and constraint violation (max) -- go through the same
      windows (``allreduce_scalars_dev``: one small kernel per rank, no collective library) or, as the
      fallback / in the CPU tests, through ``torch.distributed`` (NCCL on GPUs, gloo on CPU).

``torch.distributed`` is plumbing only: handle exchange, barrier and the fallback reduction.
"""
from __future__ import annotations

import numpy as np


def knot_ranges(N: int, world: int):
    """Contiguous 1-based inclusive knot ranges, balanced by the number of owned INTERVALS (knot k owns
    interval k -> k+1; knot N owns none)."""
    if world < 1 or world > N - 1:
        raise ValueError("need 1 <= world <= N-1 (every rank must own at least one interval)")
    n_int = N - 1
    base, extra = divmod(n_int, world)
    out, k = [], 1
    for r in range(world):
        cnt = base + (1 if r < extra else 0)
        k1 = k + cnt - 1
        if r == world - 1:
            k1 = N  # the last rank also owns the terminal knot
        out.append((k, k1))
        k = k1 + 1
    return out


def split_batch(batch: int, world: int):
    """Contiguous [begin, end) problem blocks per rank."""
    base, extra = divmod(batch, world)
    out, b = [], 0
    for r in range(world):
        cnt = base + (1 if r < extra else 0)
        out.append((b, b + cnt))
        b += cnt
    return out


class ShardedEvaluator:
    """One rank's share of a single long trajectory.

    ``evaluator_factory(prob, shard, device)`` builds the local evaluator (default: the CUDA
    ``Evaluator``); the CPU tests inject an oracle-backed stand-in to exercise the partition and the
    scalar reductions under gloo."""

    def __init__(self, prob, rank, world, device=None, dist=None, evaluator_factory=None, peer_halo=True, **kw):
        self.rank, self.world, self.dist = rank, world, dist
        self.ranges = knot_ranges(prob.trajectory.N, world)
        self.k0, self.k1 = self.ranges[rank]
        if evaluator_factory is None:
            from .evaluator import Evaluator

            evaluator_factory = lambda p, shard, device: Evaluator(p, shard=shard, device=device if device is not None else -1, **kw)
        self.local = evaluator_factory(prob, (self.k0, self.k1), device)
        self.z = prob.trajectory.dim
        self.z_begin = (self.k0 - 1) * self.z
        self.z_end = self.k1 * self.z
        self.z_halo_end = min(self.k1 + 1, prob.trajectory.N) * self.z
        self.peer_halo = False
        if peer_halo and world > 1 and dist is not None and hasattr(self.local, "shard_export"):
            # every rank publishes the IPC handle of its exchange window and maps everybody else's
            handles = [None] * world
            dist.all_gather_object(handles, self.local.shard_export())
            self.local.shard_link(rank, world, handles)
            # linking clears this rank's window: no peer may publish into it before every rank has linked
            dist.barrier()
            self.peer_halo = True

    def local_slice(self, Z):
        """This rank's input slice of the global primal vector (owned knots + the one-knot right halo)."""
        return np.ascontiguousarray(Z[self.z_begin:self.z_halo_end])

    def upload(self, Z):
        """Make this rank's slice of the global ``Z`` the resident iterate (and push the first knot to the left
        neighbour when the shards are linked).  Every rank calls this once per iterate."""
        Zloc = self.local_slice(Z)
        self.local.upload(Zloc)
        return Zloc

    def reduce_scalars(self, J_local: float, viol_local: float, device=None):
        """All-reduce (objective: sum, violation: max) -- the only collective of the sharded path."""
        if self.dist is None or self.world == 1:
            return J_local, viol_local
        import torch

        t = torch.tensor([J_local], dtype=torch.float64, device=device)
        v = torch.tensor([viol_local], dtype=torch.float64, device=device)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        self.dist.all_reduce(v, op=self.dist.ReduceOp.MAX)
        return float(t.item()), float(v.item())

    def barrier(self):
        if self.dist is not None and self.world > 1:
            self.dist.barrier()

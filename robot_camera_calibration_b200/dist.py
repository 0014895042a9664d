"""Multi-GPU plumbing: one process per GPU, observations sharded by the owner of
their eliminated block; per LM iteration the library sums the reduced system over
the ranks (band by band, behind its Schur kernel) and factors it with its block
columns distributed over the ranks (SURVEY.md 8e).  `torch.distributed` is used only to bootstrap the NCCL
communicator that librcc_ba.so owns (broadcast of the 128-byte unique id) and
to gather the eliminated-block parameters from their owners at the end.
"""
from __future__ import annotations

import copy

import numpy as np


def eliminated_is_view(scene, eliminate="auto"):
    if eliminate == "views":
        return True
    if eliminate == "markers":
        return False
    return len(scene.views) >= len(scene.markers)


def owner_ranges(counts, world):
    """Split eliminated blocks 0..n-1 into `world` contiguous ranges with
    (nearly) equal numbers of observation blocks.  Returns [(lo, hi)] per rank."""
    counts = np.asarray(counts, dtype=np.int64)
    n = len(counts)
    cum = np.concatenate([[0], np.cumsum(counts)])
    total = cum[-1]
    bounds = [0]
    for r in range(1, world):
        target = total * r / world
        b = int(np.searchsorted(cum, target, side="left"))
        bounds.append(min(max(b, bounds[-1]), n))
    bounds.append(n)
    return [(bounds[r], bounds[r + 1]) for r in range(world)]


def shard_scene(scene, rank, world, eliminate="auto"):
    """The observations whose eliminated block this rank owns.  Parameter arrays
    keep their global size and indexing (kept blocks and shared parameters are
    replicated; eliminated blocks this rank does not own simply have no
    observations here and stay untouched).  A corner layout (Scene.corners) is replicated and its slots go with their
    blocks.  Returns (sub_scene, (lo, hi))."""
    ev = eliminated_is_view(scene, eliminate)
    e_idx = scene.view_idx if ev else scene.marker_idx
    n_e = len(scene.views) if ev else len(scene.markers)
    counts = np.bincount(e_idx, minlength=n_e)
    lo, hi = owner_ranges(counts, world)[rank]
    keep = (e_idx >= lo) & (e_idx < hi)
    s = copy.copy(scene)
    s.view_idx, s.marker_idx = scene.view_idx[keep], scene.marker_idx[keep]
    s.cam_idx, s.pixels = scene.cam_idx[keep], scene.pixels[keep]
    if getattr(scene, "corner_slot", None) is not None:
        s.corner_slot = scene.corner_slot[keep]
    return s, (lo, hi)


def shard_priors(priors, elim_view, rank, owned):
    """The priors rank `rank`, owner of the eliminated blocks owned = (lo, hi), adds (rcc_ba_comm_init): priors on
    kept blocks and on the shared intr / dist / ext blocks go to rank 0, priors on an eliminated block to the rank
    that owns it.  priors: {kind: (index, mean, sqrt_information)}, kind "view" | "marker" | "intr" | "dist" | "ext";
    returns the same for this rank."""
    out = {}
    for kind, (index, mean, A) in priors.items():
        index = np.asarray(index, dtype=np.int64).reshape(-1)
        if kind in ("view", "marker") and (kind == "view") == elim_view:
            lo, hi = owned
            keep = (index >= lo) & (index < hi)
        else:
            keep = np.full(len(index), rank == 0)
        out[kind] = (index[keep], np.asarray(mean)[keep], np.asarray(A)[keep])
    return out


class DistributedBA:
    """One rank of a multi-GPU bundle adjustment.  Usage (under torchrun):

        dba = DistributedBA(scene, device=local_rank)      # scene = the FULL problem on every rank
        # priors={kind: (index, mean, sqrt_information)} (BAProblem.set_priors), the same full set on every rank:
        # each prior is added on exactly one rank (shard_priors)
        summary = dba.solve(max_iterations=30)
        views, markers, intr, dist = dba.gather_parameters()
    """

    def __init__(self, scene, device=0, eliminate="auto", rank=None, world=None, process_group=None, priors=None):
        import torch.distributed as dist
        from .problem import BAProblem
        self.dist = dist
        self.pg = process_group
        self.rank = dist.get_rank(process_group) if rank is None else rank
        self.world = dist.get_world_size(process_group) if world is None else world
        self.scene = scene
        self.elim_view = eliminated_is_view(scene, eliminate)
        self.local, self.range = shard_scene(scene, self.rank, self.world, eliminate)
        self.problem = BAProblem.from_scene(self.local, device=device,
                                            eliminate="views" if self.elim_view else "markers")
        if priors:
            for kind, (index, mean, A) in shard_priors(priors, self.elim_view, self.rank, self.range).items():
                self.problem.set_priors(kind, index, mean, A)
        if self.world > 1:
            ids = [BAProblem.comm_unique_id() if self.rank == 0 else None]
            dist.broadcast_object_list(ids, src=0, group=process_group)
            self.problem.comm_init(ids[0], self.rank, self.world)

    def solve(self, **kw):
        return self.problem.solve(**kw)

    def gather_parameters(self):
        """All ranks get the full refined parameter set (eliminated blocks from
        their owners, everything else is already identical on every rank)."""
        p = self.problem
        views, markers = p.get_view_poses(), p.get_marker_poses()
        intr, dist_c = p.get_intrinsics()
        if self.world > 1:
            mine = (views if self.elim_view else markers)[self.range[0]:self.range[1]]
            parts = [None] * self.world
            self.dist.all_gather_object(parts, (self.range, mine), group=self.pg)
            tgt = views if self.elim_view else markers
            for (lo, hi), arr in parts:
                tgt[lo:hi] = arr
        return views, markers, intr, dist_c

    def close(self):
        self.problem.close()

"""Needed-row frontier of a TRAIN_CF step: exact pruning of the per-batch full-graph propagation.

The reference re-runs the whole 3-layer propagation for every CF mini-batch (model.py:188) and then
gathers only the <= 3B batch rows of the result (model.py:189-191).  A row of layer ``l`` therefore
matters only if it is a batch row or reaches one through layers ``l+1 .. L``:

    F_L = {user, positive, negative ids},      F_{l-1} = F_l  U  cols(A[F_l, :])        (aggregator.py:54)

Rows outside ``F_l`` are never read and carry an exactly-zero gradient, so computing layer ``l`` --
forward and backward -- for ``F_l`` only gives the same loss and the same gradients as the reference.
At the Amazon-book shape a 256-sample batch needs ~730 rows of the last layer, ~3 k of the second and
~73 % of the first (58 % of its edges).

A level is a node bitmap (tested per task / per edge by the masked SpMM, csrc/spmm.cu) plus the
ascending list of its rows with a device-side count (enumerated by the bi-interaction kernels); the
tables stay indexed by node id, rows outside the frontier simply keep stale bytes.  Everything is
stream-ordered device work (csrc/frontier.cu), so the step still replays as one CUDA graph.
"""

from __future__ import annotations

import torch

from . import ops
from .graph import AttentiveGraph


class Frontier:
    def __init__(self, graph: AttentiveGraph, n_layers: int, max_ids: int):
        dev = graph.col_idx.device
        self.graph = graph
        self.n = graph.n
        self.n_layers = int(n_layers)
        words = (self.n + 31) // 32
        self.words = (words + 3) // 4 * 4  # keep every level's bitmap 16-byte aligned
        self.bitmaps = torch.zeros(self.n_layers, self.words, dtype=torch.int32, device=dev)
        # membership scratch of the level being built: one byte per node, written with plain stores by the mark / expand
        # kernels, folded into the level's bitmap (and cleared) by the listing pass
        self.flags = torch.zeros(self.words * 32, dtype=torch.uint8, device=dev)
        self.caps = [self.n] * (self.n_layers - 1) + [min(self.n, int(max_ids))]
        self.row_lists = [torch.zeros(c, dtype=torch.int32, device=dev) for c in self.caps]
        self.counts = torch.zeros(self.n_layers, dtype=torch.int32, device=dev)
        self.scratch = torch.zeros(ops.frontier_scratch_ints(self.n), dtype=torch.int32, device=dev)
        self.bad_ids = torch.zeros(1, dtype=torch.int32, device=dev)  # ids outside [0, n) seen so far (skipped)
        # backward of the upper (sparse) layers: True = scatter the edges of the few source rows (fp32 vector reductions, summed
        # in arrival order) instead of gathering over every destination row; False = the masked gather everywhere, whose fixed
        # summation order keeps training bit-identical from run to run
        self.scatter_backward = False
        self.serial = 0  # bumped by every user that (re)builds it, so a late backward can tell its levels were overwritten

    # level l in 1 .. L
    def mask(self, level: int) -> torch.Tensor:
        return self.bitmaps[level - 1]

    def rows(self, level: int) -> torch.Tensor:
        return self.row_lists[level - 1]

    def count(self, level: int) -> torch.Tensor:
        return self.counts[level - 1 : level]

    def cap(self, level: int) -> int:
        return self.caps[level - 1]

    def build(self, id_tensors) -> "Frontier":
        """(Re)build every level from the batch ids (int64 device tensors).  Stream-ordered, no host sync."""
        g = self.graph
        top = self.n_layers
        for ids in id_tensors:
            ops.frontier_mark_ids(ids, self.n, self.flags, self.bad_ids)
        ops.frontier_list(self.flags, self.mask(top), self.n, self.scratch, self.rows(top), self.count(top))
        for level in range(top - 1, 0, -1):
            ops.frontier_expand(g.plan, g.col_idx, self.rows(level + 1), self.count(level + 1), self.cap(level + 1), self.mask(level + 1), self.flags)
            ops.frontier_list(self.flags, self.mask(level), self.n, self.scratch, self.rows(level), self.count(level))
        return self

    def check_ids(self) -> None:
        """Host check (one small device read): raises like the reference's embedding lookup would have."""
        bad = int(self.bad_ids.item())
        if bad:
            self.bad_ids.zero_()
            raise IndexError(f"{bad} user / item ids outside [0, {self.n}) were passed to TRAIN_CF")

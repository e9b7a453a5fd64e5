"""Device-resident graph containers for the attentive matrix and for the attention refresh.

Layout in HBM (SURVEY.md section 7, step 2):

* ``AttentiveGraph``: the attentive matrix A as CSR (``row_ptr`` int32[N+1], ``col_idx`` int32[nnz],
  ``vals`` fp32[nnz]; canonical = (row, col)-sorted, duplicate (h, t) merged, exactly what
  ``A.coalesce()`` gives in the reference) plus the CSR of A^T (``t_ptr``, ``t_idx``, and the
  permutation ``t_perm`` that maps a transposed slot to its CSR slot, so a refresh only re-gathers
  ``t_vals = vals[t_perm]``).  The backward pass of ``A @ E`` is a *gather* over A^T -- no atomics.
* ``SpmmPlan``: the SpMM work list.  Rows longer than ``chunk`` non-zeros are split into chunks
  (heavy-tailed item / hub-entity rows) whose partial sums are reduced in a fixed order.
* ``EdgeIndex``: everything about an edge list ``(heads, relations, tails)`` the refresh needs and
  that never changes between refreshes: the slot of every edge in the coalesced structure, the
  per-relation degrees (reference ``model.py:309-312``) folded into one weight per edge, and the
  unique ``(tail, relation)`` pairs the edge score actually depends on.
"""

from __future__ import annotations

from dataclasses import dataclass

import os

import numpy as np
import torch

from . import ops

DEFAULT_CHUNK = 256


@dataclass
class SpmmPlan:
    tasks: torch.Tensor  # int32 [n_tasks, 4] = row, begin, end, partial_slot(-1 = direct)
    heavy: torch.Tensor  # int32 [n_heavy, 4] = row, first_slot, n_chunks, 0
    n_tasks: int
    n_heavy: int
    n_partials: int  # = number of heavy-chunk tasks; they come first in `tasks`
    n_rows: int  # rows of the matrix: an output (and an addend) needs at least this many
    light_rank: torch.Tensor | None = None  # int32 [n_rows]: a light row's task is n_partials + light_rank[row]; -1 = heavy row


def spmm_plan_host(row_ptr: np.ndarray, chunk: int = DEFAULT_CHUNK, sort_light: bool = False):
    """Host logic of the SpMM plan (pure numpy, unit-tested on CPU).

    Heavy chunks come first (they are the longest tasks), then every light row: in row order, or (``sort_light``, what
    ``make_plan`` uses) longest first, so that the warps of a CTA and the CTAs of a wave carry similar loads.
    Every row gets at least one task, so empty rows are still written (as zero / addend)."""
    row_ptr = np.asarray(row_ptr, dtype=np.int64)
    n = row_ptr.shape[0] - 1
    lens = np.diff(row_ptr)
    heavy_rows = np.nonzero(lens > chunk)[0]
    light_rows = np.nonzero(lens <= chunk)[0]
    n_chunks = (lens[heavy_rows] + chunk - 1) // chunk
    first_slot = np.concatenate([[0], np.cumsum(n_chunks)])[:-1] if heavy_rows.size else np.zeros(0, np.int64)
    n_partials = int(n_chunks.sum()) if heavy_rows.size else 0
    if heavy_rows.size:
        rep_rows = np.repeat(heavy_rows, n_chunks)
        k = np.arange(n_partials) - np.repeat(first_slot, n_chunks)
        begin = row_ptr[rep_rows] + k * chunk
        end = np.minimum(begin + chunk, row_ptr[rep_rows + 1])
        heavy_tasks = np.stack([rep_rows, begin, end, np.arange(n_partials)], axis=1)
        heavy = np.stack([heavy_rows, first_slot, n_chunks, np.zeros_like(heavy_rows)], axis=1)
    else:
        heavy_tasks = np.zeros((0, 4), np.int64)
        heavy = np.zeros((0, 4), np.int64)
    if sort_light:  # longest first (stable): neighbouring tasks -- the two halves of a warp, the warps of a CTA -- get equal lengths
        light_rows = light_rows[np.argsort(-lens[light_rows], kind="stable")]
    light_tasks = np.stack([light_rows, row_ptr[light_rows], row_ptr[light_rows + 1], np.full(light_rows.size, -1)], axis=1)
    tasks = np.concatenate([heavy_tasks, light_tasks]).astype(np.int32)
    assert tasks.shape[0] == n - heavy_rows.size + n_partials
    return tasks, heavy.astype(np.int32), n_partials


def make_plan(row_ptr: torch.Tensor, chunk: int = DEFAULT_CHUNK) -> SpmmPlan:
    rp = row_ptr.cpu().numpy()
    sort_light = os.environ.get("KGAT_PLAN_SORT", "1") == "1"  # measured at the Amazon-book shape: CF step 662 -> 648 us
    tasks, heavy, n_partials = spmm_plan_host(rp, chunk, sort_light=sort_light)
    dev = row_ptr.device
    # light rows follow the heavy chunks (spmm_plan_host): light_rank[row] = index of the row's task among them
    light_rank = np.full(rp.shape[0] - 1, -1, dtype=np.int32)
    light_rank[tasks[n_partials:, 0]] = np.arange(tasks.shape[0] - n_partials, dtype=np.int32)
    return SpmmPlan(
        tasks=torch.from_numpy(tasks).to(dev).contiguous(),
        heavy=torch.from_numpy(heavy).to(dev).contiguous(),
        n_tasks=int(tasks.shape[0]),
        n_heavy=int(heavy.shape[0]),
        n_partials=n_partials,
        n_rows=int(rp.shape[0] - 1),
        light_rank=torch.from_numpy(light_rank).to(dev).contiguous(),
    )


class AttentiveGraph:
    """CSR of A and of A^T on the device, with SpMM plans for both directions."""

    def __init__(self, n: int, row_ptr, col_idx, vals, chunk: int = DEFAULT_CHUNK):
        self.n = int(n)
        self.row_ptr, self.col_idx, self.vals = row_ptr, col_idx, vals
        self.nnz = int(col_idx.numel())
        self.chunk = chunk
        dev = col_idx.device
        # transposed structure: group the slots by (col, row)
        row_of_slot = torch.repeat_interleave(
            torch.arange(self.n, device=dev, dtype=torch.int64), (row_ptr[1:] - row_ptr[:-1]).to(torch.int64)
        )
        keys_t = col_idx.to(torch.int64) * self.n + row_of_slot
        order, _, _, uniq = ops.group_by_key(keys_t, key_bits=max(1, (self.n * self.n - 1).bit_length()))
        if uniq.numel() != self.nnz:
            raise ValueError("CSR structure holds duplicate (row, col) entries")
        self.t_perm = order  # transposed slot -> CSR slot
        self.t_ptr, self.t_idx = ops.decode_sorted_keys(uniq, self.n, self.n)
        self.t_vals = torch.empty_like(vals)
        self.plan = make_plan(row_ptr, chunk)
        self.t_plan = make_plan(self.t_ptr, chunk)
        self._partials = None
        self._indices64 = None
        self.refresh_transposed_values()

    # -- construction -------------------------------------------------------------------------
    @classmethod
    def from_coo(cls, rows: torch.Tensor, cols: torch.Tensor, vals: torch.Tensor, n: int, chunk: int = DEFAULT_CHUNK):
        """Coalesce an arbitrary-order COO (duplicates summed in input order) into CSR.
        Bit-exact structure w.r.t. ``torch.sparse_coo_tensor(...).coalesce()``."""
        rows = rows.to(torch.int64)
        cols = cols.to(torch.int64)
        if rows.numel() and (int(rows.min()) < 0 or int(rows.max()) >= n or int(cols.min()) < 0 or int(cols.max()) >= n):
            raise IndexError("attentive matrix index out of range")
        keys = (rows * n + cols).contiguous()
        order, _, group_ptr, uniq = ops.group_by_key(keys, key_bits=max(1, (n * n - 1).bit_length()))
        row_ptr, col_idx = ops.decode_sorted_keys(uniq, n, n)
        merged = ops.segment_sum(vals.to(torch.float32).contiguous(), order, group_ptr)
        return cls(n, row_ptr, col_idx, merged, chunk)

    @classmethod
    def from_sparse_coo(cls, att: torch.Tensor, chunk: int = DEFAULT_CHUNK):
        idx = att._indices()
        return cls.from_coo(idx[0], idx[1], att._values(), att.shape[0], chunk)

    # -- values -------------------------------------------------------------------------------
    def refresh_transposed_values(self):
        ops.gather_f32(self.vals, self.t_perm, out=self.t_vals)

    def set_values(self, vals: torch.Tensor):
        self.vals = vals
        self.refresh_transposed_values()

    # -- scratch ------------------------------------------------------------------------------
    def partials(self, d: int) -> torch.Tensor | None:
        need = max(self.plan.n_partials, self.t_plan.n_partials) * d
        if need == 0:
            return None
        if self._partials is None or self._partials.numel() < need:
            self._partials = torch.empty(need, dtype=torch.float32, device=self.col_idx.device)
        return self._partials

    # -- ops ----------------------------------------------------------------------------------
    def matmul(self, x: torch.Tensor, out: torch.Tensor | None = None, addend: torch.Tensor | None = None, row_mask=None, edge_mask=None,
               rows=None, n_rows_dev=None, tag: str = ""):
        """out = A @ x (+ addend)   -- reference aggregator.py:54.  ``row_mask`` / ``edge_mask`` / ``rows``: a frontier level's
        bitmap(s) and row list (ops.spmm)."""
        if out is None:
            out = torch.empty(self.n, x.shape[1], dtype=torch.float32, device=x.device)
        return ops.spmm(self.plan, self.col_idx, self.vals, x, out, addend, self.partials(x.shape[1]), row_mask=row_mask, edge_mask=edge_mask,
                        rows=rows, n_rows_dev=n_rows_dev, tag=tag)

    def matmul_t(self, x: torch.Tensor, out: torch.Tensor | None = None, addend: torch.Tensor | None = None, row_mask=None, edge_mask=None,
                 rows=None, n_rows_dev=None, tag: str = ""):
        """out = A^T @ x (+ addend)   -- autograd backward of aggregator.py:54"""
        if out is None:
            out = torch.empty(self.n, x.shape[1], dtype=torch.float32, device=x.device)
        return ops.spmm(self.t_plan, self.t_idx, self.t_vals, x, out, addend, self.partials(x.shape[1]), row_mask=row_mask, edge_mask=edge_mask,
                        rows=rows, n_rows_dev=n_rows_dev, tag=tag)

    # -- the reference-facing view --------------------------------------------------------------
    def indices64(self) -> torch.Tensor:
        if self._indices64 is None:
            dev = self.col_idx.device
            rows = torch.repeat_interleave(
                torch.arange(self.n, device=dev, dtype=torch.int64), (self.row_ptr[1:] - self.row_ptr[:-1]).to(torch.int64)
            )
            self._indices64 = torch.stack([rows, self.col_idx.to(torch.int64)])
        return self._indices64

    def coo_tensor(self) -> torch.Tensor:
        """Coalesced sparse COO view sharing ``vals`` (what ``model.attentive_matrix`` exposes)."""
        return torch.sparse_coo_tensor(self.indices64(), self.vals, size=(self.n, self.n), is_coalesced=True)


class EdgeIndex:
    """Static structure of an edge list for the attention refresh (reference model.py:318-366)."""

    def __init__(self, heads, rels, tails, relation_indices, n: int, chunk: int = DEFAULT_CHUNK):
        dev = heads.device
        heads = heads.to(torch.int64)
        tails = tails.to(torch.int64)
        rels = rels.to(torch.int64)
        relation_indices = relation_indices.to(torch.int64).to(dev)
        if heads.numel() and (int(heads.min()) < 0 or int(heads.max()) >= n or int(tails.min()) < 0 or int(tails.max()) >= n):
            raise IndexError("edge endpoint out of range")
        n_rel_ids = int(max(int(rels.max()) if rels.numel() else 0, int(relation_indices.max()) if relation_indices.numel() else 0)) + 1
        # edges whose relation is listed k times appear k times in the reference's COO -> weight k
        mult_table = torch.bincount(relation_indices, minlength=n_rel_ids).to(torch.float32)
        mult = mult_table[rels]
        keep = mult > 0
        self.input_edges = torch.nonzero(keep).flatten()  # kept edges, input order
        if not bool(keep.all()):
            heads, tails, rels, mult = heads[keep], tails[keep], rels[keep], mult[keep]
        self.n = n
        self.n_edges = int(heads.numel())
        nbits = max(1, (n * n - 1).bit_length())
        # slots: coalesced (h, t) structure
        order, slot_of_edge, slot_ptr, uniq = ops.group_by_key((heads * n + tails).contiguous(), key_bits=nbits)
        self.order = order  # sorted position -> kept-edge index
        self.slot_ptr = slot_ptr
        row_ptr, col_idx = ops.decode_sorted_keys(uniq, n, n)
        # per-relation degrees (bincount inside the relation batch, model.py:310-311)
        rbits = max(1, (n_rel_ids * n - 1).bit_length())
        _, g_h, p_h, uniq_rh = ops.group_by_key((rels * n + heads).contiguous(), key_bits=rbits)
        deg_h = (p_h[1:] - p_h[:-1])[g_h.long()].to(torch.int32)
        _, g_t, p_t, uniq_rt = ops.group_by_key((rels * n + tails).contiguous(), key_bits=rbits)
        deg_t = (p_t[1:] - p_t[:-1])[g_t.long()].to(torch.int32)
        o = order.long()
        need_mult = bool((mult != 1).any())
        self.edge_weight = ops.att_edge_weights(deg_h[o].contiguous(), deg_t[o].contiguous(), mult[o].contiguous() if need_mult else None)
        # unique (relation, tail) pairs, relation-major
        self.pair_rel = (uniq_rt // n).to(torch.int32).contiguous()
        self.pair_tail = (uniq_rt % n).to(torch.int32).contiguous()
        self.pair_of_edge = g_t[o].contiguous()  # slot-sorted edge position -> pair id
        self.n_pairs = int(uniq_rt.numel())
        # the same for the heads, and the relation of every edge (canonical-KGAT score mode needs x_h = e_h W_r and e_r too)
        self.head_pair_rel = (uniq_rh // n).to(torch.int32).contiguous()
        self.head_pair_node = (uniq_rh % n).to(torch.int32).contiguous()
        self.head_pair_of_edge = g_h[o].contiguous()
        self.edge_rel = rels[o].to(torch.int32).contiguous()
        self.edge_mult = mult[o].contiguous() if need_mult else None
        # the refreshed attentive matrix lives in this structure
        vals = torch.zeros(col_idx.numel(), dtype=torch.float32, device=dev)
        self.graph = AttentiveGraph(n, row_ptr, col_idx, vals, chunk)

    def sorted_from_input(self, per_edge_input: torch.Tensor) -> torch.Tensor:
        """Re-order a per-input-edge tensor into slot-sorted edge order."""
        return per_edge_input[self.input_edges][self.order.long()].contiguous()

"""KGAT model API -- drop-in for ``src.model.KGAT.model.{KGAT, KGATArgs, KGATMode}``
(reference src/model/KGAT/model.py:13-431), backed by hand-written sm_100a kernels.

Same constructor, same ``forward(*tensors, mode=KGATMode.X)`` dispatch, same optimiser hooks, same
parameter names / ``state_dict`` keys, same public sparse-COO ``attentive_matrix`` -- so the
reference's ``train`` / ``predict`` / ``recommend`` drivers (main.py:234-636) run unchanged with

    from kgat_b200.model import KGAT, KGATArgs, KGATMode

What changes is underneath: each mode is one short chain of fused CUDA kernels (see
``include/kgat_b200.h``), the attention refresh never leaves the device, and evaluation reuses the
propagated tables across the 256-user PREDICT batches.  There is no PyTorch / CPU fallback: using
the model without a CUDA device raises.

Reference quirks that are reproduced on purpose (SURVEY.md section 0): the attention score is the
value-path MLP + LayerNorm + tanh-sum scaled by per-relation degrees (Q1); attention dropout is live
when the refresh runs in ``train()`` mode (Q2); duplicate (h, t) entries are summed before the row
softmax and the result is (row, col)-sorted (Q3); item ids index the propagated table without a
``user_num`` offset (Q4).
"""

from __future__ import annotations

from dataclasses import dataclass, field
from enum import IntEnum
from typing import Any

import torch
from torch import nn

from . import ops
from ._lib import KgatLibraryError
from .aggregator import Aggregator, AggregatorArgs
from .frontier import Frontier
from .functions import (CFLossFunction, DropoutSpec, GraphedStep, KGLossFunction, PropagateFunction, last_table_grad,
                        propagate_backward, propagate_forward)
from .graph import AttentiveGraph, EdgeIndex
from .multi_head_attention import MultiHeadAttention
from .optim import DeferredRows, FusedAdam


@dataclass
class KGATArgs:
    user_num: int
    entity_num: int
    relation_num: int
    cf_embedding_dim: int = 64
    kg_embedding_dim: int = 64
    attentive_matrix: torch.Tensor | None = None
    message_dropout: list[float] = field(default_factory=lambda: [0.1, 0.1, 0.1])
    layer_size: list[int] = field(default_factory=lambda: [64, 32, 16])
    regularization_params: list[float] = field(default_factory=lambda: [1e-5, 1e-5])


@dataclass
class PathExplanation:
    """Result of ``KGAT.explain`` for P (user, item) pairs, k paths each, up to H hops (see ``ops.explain_paths``).
    A slot indexes ``attentive_matrix.indices()`` / ``.values()``; missing paths and positions after the last hop hold -1
    (``hops`` 0, ``weight`` 0)."""

    nodes: torch.Tensor  # int64 [P, k, H+1]: user node, intermediate nodes, item node
    slots: torch.Tensor  # int64 [P, k, H]
    hops: torch.Tensor  # int32 [P, k]
    weight: torch.Tensor  # fp32 [P, k]: product of the hop values
    count: torch.Tensor  # int64 [P, H]: number of paths of each length
    mass: torch.Tensor  # fp32 [P, H]: summed weight of those paths


@dataclass
class Recommendation:
    """Result of ``KGAT.recommend`` for U users: each user's top-k eligible problems, best first.  Positions from ``count`` on
    hold item -1 and score -inf."""

    items: torch.Tensor  # int64 [U, k]: problem ids
    scores: torch.Tensor  # fp32 [U, k]: the PREDICT scores of those problems
    count: torch.Tensor  # int32 [U]: min(k, number of eligible problems)


@dataclass
class TargetRanks:
    """Result of ``KGAT.rank`` for U users and M targets in all: row ``b`` is ``ptr[b] .. ptr[b+1]``, the targets of ``user_ids[b]``
    in ascending id."""

    ptr: torch.Tensor  # int64 [U+1]
    items: torch.Tensor  # int64 [M]: problem ids
    scores: torch.Tensor  # fp32 [M]: the PREDICT scores of those problems
    rank: torch.Tensor  # int64 [M]: eligible problems ranked before the target (0 = first), -1 when the target is not eligible
    eligible: torch.Tensor  # int64 [U]: number of eligible problems of the user


@dataclass
class Completion:
    """Result of ``KGAT.complete`` for Q queries ``(h, r, ?)``: each query's top-k eligible tails, lowest TransR energy first.
    Positions from ``count`` on hold tail -1 and energy +inf."""

    tails: torch.Tensor  # int64 [Q, k]: CKG node ids
    energy: torch.Tensor  # fp32 [Q, k]: ||e_h W_r + e_r - e_t W_r||^2, bit-identical to the TransR loss's term
    count: torch.Tensor  # int32 [Q]: min(k, number of eligible candidates)


@dataclass
class TailRanks:
    """Result of ``KGAT.kg_rank`` for Q triples ``(h, r, t)``."""

    energy: torch.Tensor  # fp32 [Q]: the TransR energy of the triple
    rank: torch.Tensor  # int64 [Q]: eligible candidates ranked before t (0 = first), -1 when t is not a candidate
    eligible: torch.Tensor  # int64 [Q]: number of eligible candidates, t included


class KGATMode(IntEnum):
    TRAIN_CF = 0
    TRAIN_KG = 1
    UPDATE_ATTENTION = 2
    PREDICT = 3


class _EntityEmbedding(nn.Embedding):
    """``nn.Embedding`` whose ``weight`` attribute first settles any deferred optimiser work on it (optim.DeferredRows): inside
    a run of TRAIN_KG steps the table's rows lag a bounded number of zero-gradient Adam updates behind; whoever looks at the
    parameter -- other modes, checkpoints, user code -- triggers the catch-up and sees exactly the reference's values.  The
    KG step itself reads ``_parameters["weight"]``.  Same state_dict keys, same repr, same init RNG consumption."""

    def __getattr__(self, name: str):
        if name == "weight":
            hook = self.__dict__.get("_kgat_settle")
            if hook is not None:
                hook()
        return super().__getattr__(name)

    def _get_name(self) -> str:
        return "Embedding"


class KGAT(nn.Module):
    def __init__(self, args: KGATArgs) -> None:
        super().__init__()
        # ---- same attributes, same construction order as the reference (model.py:34-97) ----
        self._user_num = args.user_num
        self._entity_num = args.entity_num
        self._relation_num = args.relation_num
        self._message_dropout = args.message_dropout
        self._layer_dims = args.layer_size
        self._layer_num = len(self._layer_dims)
        self._regularization_params = args.regularization_params
        self._cf_embedding_dim = args.cf_embedding_dim
        self._kg_embedding_dim = args.kg_embedding_dim
        n = self._user_num + self._entity_num

        self._user_entity_embedding = _EntityEmbedding(num_embeddings=n, embedding_dim=self._cf_embedding_dim)
        self._relation_embedding = nn.Embedding(num_embeddings=self._relation_num, embedding_dim=self._kg_embedding_dim)
        self._trans_matrix = nn.Parameter(data=torch.Tensor(self._relation_num, self._cf_embedding_dim, self._kg_embedding_dim))
        nn.init.xavier_uniform_(tensor=self._user_entity_embedding.weight)
        nn.init.xavier_uniform_(tensor=self._relation_embedding.weight)
        nn.init.xavier_uniform_(tensor=self._trans_matrix)

        self._aggregator_layers = nn.ModuleList()
        dims = [self._cf_embedding_dim, *self._layer_dims]
        for l in range(self._layer_num):
            self._aggregator_layers.append(
                Aggregator(AggregatorArgs(input_dim=dims[l], output_dim=dims[l + 1], dropout=self._message_dropout[l]))
            )

        # public for visualisation (model.py:83-92): a sparse-COO parameter without gradient
        self.attentive_matrix = nn.Parameter(
            data=torch.sparse_coo_tensor(
                indices=torch.empty(size=(2, 0), dtype=torch.long),
                values=torch.empty(size=(0,), dtype=torch.float32),
                size=torch.Size([n, n]),
            )
        )
        if args.attentive_matrix is not None:
            self.attentive_matrix.data = args.attentive_matrix
        self.attentive_matrix.requires_grad = False

        self._multi_head_attention = MultiHeadAttention(
            cf_embedding_dim=self._cf_embedding_dim, kg_embedding_dim=self._kg_embedding_dim
        )

        # ---- device-side caches (not part of the state_dict) ----
        self._graph_cache: AttentiveGraph | None = None
        self._graph_key: tuple | None = None
        self._graph_version = 0
        self._edge_cache: EdgeIndex | None = None
        self._edge_key: tuple | None = None
        self._table_cache: list | None = None
        self._table_key: tuple | None = None
        # test hooks: inject dropout decisions instead of drawing them (parity with the reference RNG)
        self._injected_message_keep_bits: list | None = None  # per layer int32 [N, ceil(d_out/32)]
        self._injected_head_bits: torch.Tensor | None = None  # uint8 [n_edges], input edge order
        self.spmm_chunk = 256
        # CUDA-graph fast path behind model(...) / loss.backward() for the two training modes (functions.GraphedStep)
        self.api_graphs = True
        self._api_steps: dict = {}
        self._last_step: dict = {}
        self._kg_fast = None  # closure re-submitting the last TRAIN_KG step after re-checking everything that can change between calls
        # TRAIN_CF computes every layer only for the rows the batch can reach (frontier.py): exact, ~2x less work at the
        # Amazon-book shape.  False = the reference's literal full-graph propagation per batch.
        self.cf_pruning = True
        self._frontiers: dict = {}
        # Edge score of the attention refresh: "reference" = what the reference computes (value path of its multi-head attention +
        # LayerNorm + tanh-sum, degree-weighted: SURVEY.md Q1, the parity target); "kgat" = the KGAT paper's
        # pi(h, r, t) = (W_r e_t)^T tanh(W_r e_h + e_r) that north_star names, followed by the same duplicate merge + row softmax.
        self.score_mode = "reference"
        # KG phase through this API: update the batch's rows and a rotating 1 / kg_window slice of the entity table per step
        # instead of sweeping all N rows (bit-identical once settled; see optim.DeferredRows).  False = per-step sweep.
        self.kg_deferred_adam = True
        self.kg_window = 16
        self._user_entity_embedding.__dict__["_kgat_settle"] = self._settle

    # ------------------------------------------------------------------------------------------
    # plumbing
    # ------------------------------------------------------------------------------------------
    @property
    def node_num(self) -> int:
        return self._user_num + self._entity_num

    def _settle(self) -> None:
        """Bring every row of the entity table up to the KG optimiser's step count (no-op unless a deferred phase is open)."""
        opt = self.__dict__.get("_kg_optimizer")
        if opt is not None and opt.deferred is not None and opt.deferred.active:
            opt.deferred.flush()

    def _emb_raw(self) -> torch.nn.Parameter:
        """The entity table without settling deferred rows (the KG step's own accesses)."""
        return self._user_entity_embedding._parameters["weight"]

    def state_dict(self, *a, **k):
        self._settle()
        return super().state_dict(*a, **k)

    def train(self, mode: bool = True):
        self._settle()
        return super().train(mode)

    def named_parameters(self, *a, **k):
        self._settle()
        return super().named_parameters(*a, **k)

    def _device(self) -> torch.device:
        dev = self._emb_raw().device
        if dev.type != "cuda":
            raise KgatLibraryError(
                "kgat_b200.KGAT runs on a CUDA device only (call .to('cuda')); there is no CPU / PyTorch fallback"
            )
        return dev

    def _ids(self, t: Any) -> torch.Tensor:
        if isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == torch.int64 and t.is_contiguous():
            return t
        t = torch.as_tensor(t)
        return t.to(device=self._device(), dtype=torch.int64, non_blocking=True).contiguous()

    def _layers(self):
        return [agg.kernel_params() for agg in self._aggregator_layers]

    def _apply(self, fn, *a, **k):
        self._settle()
        out = super()._apply(fn, *a, **k)
        self._invalidate()
        return out

    def load_state_dict(self, *a, **k):
        self._settle()
        out = super().load_state_dict(*a, **k)
        self._invalidate()
        return out

    def _invalidate(self) -> None:
        self._graph_cache = self._graph_key = None
        self._table_cache = self._table_key = None
        self._api_steps = {}
        self._last_step = {}
        self._kg_fast = None
        self._frontiers = {}

    def _frontier(self, graph: AttentiveGraph, n_ids: int, fresh: bool = False) -> Frontier | None:
        """Needed-row frontier buffers for TRAIN_CF batches of ``n_ids`` ids on ``graph`` (None when pruning is off)."""
        if not self.cf_pruning:
            return None
        if fresh:
            return Frontier(graph, self._layer_num, n_ids)
        key = (id(graph), n_ids)
        f = self._frontiers.get(key)
        if f is None:
            if len(self._frontiers) > 4:
                self._frontiers.clear()
            f = self._frontiers[key] = Frontier(graph, self._layer_num, n_ids)
        return f

    def _graph(self) -> AttentiveGraph:
        """CSR / CSC containers of the current ``attentive_matrix`` (rebuilt when it is replaced)."""
        att = self.attentive_matrix.data
        key = (att._values().data_ptr(), att._indices().data_ptr(), att._nnz(), att.device)
        if self._graph_cache is None or key != self._graph_key:
            dev = self._device()
            if att.device != dev:
                att = att.to(dev)
            self._graph_cache = AttentiveGraph.from_sparse_coo(att, chunk=self.spmm_chunk)
            self._graph_key = key
            self._graph_version += 1
        return self._graph_cache

    def _drop_spec(self) -> DropoutSpec:
        if not self.training:
            return DropoutSpec(ps=[0.0] * self._layer_num)
        ps = [float(agg.message_dropout.p) for agg in self._aggregator_layers]
        if self._injected_message_keep_bits is not None:
            return DropoutSpec(ps=ps, keep_bits=self._injected_message_keep_bits)
        seed = int(torch.randint(0, 2**62, (1,)).item()) if any(p > 0 for p in ps) else 0
        return DropoutSpec(ps=ps, seed=seed)

    # ------------------------------------------------------------------------------------------
    # A3: propagation
    # ------------------------------------------------------------------------------------------
    def _tables(self) -> list[torch.Tensor]:
        """[E0, E1, ..., EL].  With autograd disabled and no live dropout the result is cached
        until a parameter or the attentive matrix changes (the reference re-propagates for every
        256-user PREDICT batch, model.py:388)."""
        graph = self._graph()
        e0 = self._user_entity_embedding.weight
        drop = self._drop_spec()
        flat = [t for grp in self._layers() for t in grp]
        needs_grad = torch.is_grad_enabled() and any(t.requires_grad for t in [e0, *flat])
        if needs_grad:
            outs = PropagateFunction.apply(graph, drop, e0, *flat)
            return [e0, *outs]
        deterministic = all(p == 0.0 for p in drop.ps)
        key = (self._graph_version, graph.vals.data_ptr(), graph.vals._version, e0.data_ptr(), e0._version, *[t._version for t in flat])
        if deterministic and self._table_cache is not None and key == self._table_key:
            return self._table_cache
        layers = [tuple(t.detach() for t in grp) for grp in self._layers()]
        st = propagate_forward(graph, e0.detach(), layers, drop, save=False)
        if deterministic:
            self._table_cache, self._table_key = st.tables, key
        return st.tables

    def _build_cf_embeddings(self) -> torch.Tensor:
        """(user_num + entity_num, concatenated_dim) -- model.py:124-140."""
        return torch.cat(self._tables(), dim=1)

    # ------------------------------------------------------------------------------------------
    # A5 / A6: losses
    # ------------------------------------------------------------------------------------------
    def _use_api_graphs(self, params) -> bool:
        if not (self.api_graphs and self._injected_message_keep_bits is None and torch.is_grad_enabled()):
            return False
        for p in params:
            if not p.requires_grad:
                return False
        return not torch._C._cuda_isCurrentStreamCapturing()

    def _api_step(self, kind: str, batch: int, params, extra_key, n_ids, make_bodies) -> GraphedStep:
        key = (kind, batch, self.training, tuple(p.data_ptr() for p in params), extra_key)
        step = self._api_steps.get(key)
        if step is None:
            if len(self._api_steps) > 8:
                self._api_steps.clear()
            bodies = make_bodies()
            step = self._api_steps[key] = GraphedStep(params, batch, n_ids, bodies[0], bodies[1])
            step.pre_submit = bodies[2] if len(bodies) > 2 else None
        self._last_step[kind] = step
        return step

    def _ids_fast(self, tensors):
        """Index tensors for the graphed API path: int64 tensors already on the device, or views of pinned host memory
        (copied by the step's own launch call), pass through untouched; anything else goes through ``_ids``."""
        out = []
        for t in tensors:
            # host tensors need not be pinned: the step's copy (cudaMemcpyAsync in kgat_step_submit / Tensor.copy_) stages pageable
            # memory before it returns; is_pinned() alone costs ~1 us per tensor
            if type(t) is torch.Tensor and t.dtype is torch.int64 and t.is_contiguous():
                out.append(t)
            else:
                out.append(self._ids(t))
        return out

    def _calc_cf_loss(self, user_ids, positive_item_ids, negative_item_ids) -> torch.Tensor:
        graph = self._graph()
        flat = [t for grp in self._layers() for t in grp]
        params = [self._user_entity_embedding.weight, *flat]
        if self._use_api_graphs(params):
            ids = self._ids_fast((user_ids, positive_item_ids, negative_item_ids))

            def make_bodies():
                reg = float(self._regularization_params[0])
                layers = [tuple(t.detach() for t in grp) for grp in self._layers()]
                ps = [float(a.message_dropout.p) if self.training else 0.0 for a in self._aggregator_layers]
                seed = int(torch.randint(0, 2**62, (1,)).item()) if any(p > 0 for p in ps) else 0
                frontier = self._frontier(graph, 3 * ids[0].numel(), fresh=True)  # owned by this step's captured graphs

                def body_fwd(st):
                    st.counter.add_(1)
                    st.frontier = frontier  # (introspection: tests / tools read the step's frontier levels)
                    drop = DropoutSpec(ps=ps, seed=seed, seed_dev=st.counter)
                    if frontier is not None:
                        frontier.build([st.ids.view(-1)])
                    st.prop = propagate_forward(graph, params[0].detach(), layers, drop, save=True, frontier=frontier)
                    ops.bpr_forward(st.prop.tables, st.ids[0], st.ids[1], st.ids[2], reg, st.loss, st.scratch, publish=st.publish)
                    st.published = True

                def body_bwd(st):
                    n_tab = len(st.prop.tables)

                    def inject(l, buf):
                        grads = [None] * n_tab
                        grads[l] = buf
                        ops.bpr_backward(st.prop.tables, grads, st.ids[0], st.ids[1], st.ids[2], reg, st.scratch, st.g_loss)

                    g_last = last_table_grad(st.prop, frontier)
                    inject(n_tab - 1, g_last)
                    g_e0, pgrads = propagate_backward(graph, st.prop, layers, g_last, inject, frontier=frontier)
                    return [g_e0] + [t for grp in pgrads for t in grp]
                return body_fwd, body_bwd

            step = self._api_step("cf", ids[0].numel(), params,
                                  (id(graph), graph.vals.data_ptr(), graph.t_vals.data_ptr(), self.cf_pruning), 3, make_bodies)
            return step.submit(ids)
        u, p, n = self._ids(user_ids), self._ids(positive_item_ids), self._ids(negative_item_ids)
        return CFLossFunction.apply(
            graph, u, p, n, float(self._regularization_params[0]), self._drop_spec(),
            self._frontier(graph, u.numel() + p.numel() + n.numel()), self._user_entity_embedding.weight, *flat,
        )

    def _make_kg_fast(self, step: GraphedStep, params, opt, deferred):
        """The steady state of a KG phase: the same step object is re-submitted ~12 k times per epoch and the host is the
        bottleneck (a KG step is ~40 us of GPU work), so everything ``_calc_kg_loss`` decides is decided once and this closure only
        re-checks, with identity / integer comparisons, what can change between two calls.  Returns None to fall back."""
        emb, rel, w = params
        emb_mod, rel_mod, own = self._user_entity_embedding._parameters, self._relation_embedding._parameters, self._parameters
        ptrs = (emb.data_ptr(), rel.data_ptr(), w.data_ptr())
        training, want_deferred, window, batch = self.training, self.kg_deferred_adam, self.kg_window, step._batch
        state_version = opt.state_version if opt is not None else 0
        int64, Tensor, capturing, grad_enabled = torch.int64, torch.Tensor, torch._C._cuda_isCurrentStreamCapturing, torch.is_grad_enabled
        last_step = self._last_step

        def fast(h, r, pt, nt):
            if not (self.api_graphs and self.training is training and self.kg_deferred_adam is want_deferred and self.kg_window == window
                    and self._injected_message_keep_bits is None and grad_enabled()):
                return None
            if emb_mod["weight"] is not emb or rel_mod["weight"] is not rel or own["_trans_matrix"] is not w:
                return None
            if (emb.data_ptr(), rel.data_ptr(), w.data_ptr()) != ptrs or not (emb.requires_grad and rel.requires_grad and w.requires_grad):
                return None
            if self.__dict__.get("_kg_optimizer") is not opt or (opt is not None and (opt.deferred is not deferred or opt.state_version != state_version)):
                return None
            for t in (h, r, pt, nt):
                if type(t) is not Tensor or t.dtype is not int64 or not t.is_contiguous() or t.numel() != batch:
                    return None
            if capturing():
                return None
            if deferred is not None:
                deferred.ensure_phase()
            last_step["kg"] = step
            return step.submit((h, r, pt, nt))

        return fast

    def _calc_kg_loss(self, heads, relations, positive_tails, negative_tails) -> torch.Tensor:
        fast = self._kg_fast
        if fast is not None:
            loss = fast(heads, relations, positive_tails, negative_tails)
            if loss is not None:
                return loss
            self._kg_fast = None
        self._device()
        params = [self._emb_raw(), self._relation_embedding.weight, self._trans_matrix]
        if self._use_api_graphs(params):
            ids = self._ids_fast((heads, relations, positive_tails, negative_tails))
            opt = self.__dict__.get("_kg_optimizer")
            deferred = None
            if self.kg_deferred_adam and opt is not None and params[0].shape[1] % 64 == 0:
                deferred = opt.deferred
                if deferred is None or deferred.param is not params[0] or deferred.window != self.kg_window:
                    if deferred is not None:
                        deferred.flush()
                    deferred = opt.deferred = DeferredRows(opt, params[0], window=self.kg_window)
                if not deferred.active and not (deferred.usable() and len({int(opt.state[p]["step"]) if opt.state[p] else 0 for p in params}) == 1):
                    deferred = None  # no optimiser state yet (first step): the per-step sweep creates it
            if deferred is None:
                self._settle()

            def make_bodies():
                reg = float(self._regularization_params[1])
                emb, rel, w = (p.detach() for p in params)
                b = ids[0].numel()
                # One pass computes loss and gradients (csrc/losses.cu: kgat_transr_step): the embedding gradient lands in <= 3B
                # compact rows (row_slot: node -> row), which the fused Adam replay reads directly.  The dense N x d
                # ``embedding.weight.grad`` autograd would hand out (model.py:204-261) is kept valid as well -- zero outside the
                # batch's rows, which are copied in after the pass and cleared again before the next one -- so anything that
                # inspects ``.grad`` or steps another optimiser sees the reference's gradient.
                g_dense = torch.zeros_like(emb)
                g_rel, g_w = torch.zeros_like(rel), torch.zeros_like(w)
                row_slot = torch.full((emb.shape[0],), -1, dtype=torch.int32, device=emb.device)
                g_rows = torch.zeros(3 * b, emb.shape[1], dtype=torch.float32, device=emb.device)
                prev_ids = torch.zeros(4, b, dtype=torch.int64, device=emb.device)
                d = deferred
                if d is not None:
                    exp_avg, exp_avg_sq = d.state_tensors()

                keep = (prev_ids[0], prev_ids[2], prev_ids[3])  # whose rows the dense view holds (row 1, the relations, stays unused)

                def body_fwd(st):
                    if d is None:
                        ops.transr_release_rows(g_dense, prev_ids.view(-1), row_slot)  # the previous batch's rows and slot claims
                        ops.transr_step(emb, rel, w, st.ids[0], st.ids[1], st.ids[2], st.ids[3], reg, st.loss, None, st.scratch, row_slot,
                                        g_rows, g_rel, g_w, publish=st.publish)
                    else:
                        # rows this batch reads first take the zero-gradient updates they were spared (csrc/adam.cu, rolling window); the
                        # same launch claims the compact gradient rows, zeroes the gradient buffers and clears the previous batch's rows
                        # of the dense view.  (The previous batch's slot claims were consumed by the rolling update; ``pre_submit``
                        # below covers the steps where it did not run.)
                        ops.adam_rolling_prepare(st.ids[0], st.ids[2], st.ids[3], row_slot, g_rows, g_rel, g_w, emb, exp_avg, exp_avg_sq,
                                                 d.row_step, d.step_dev, d.s0, d.table, d.hyper, prev_ids=keep, dense=g_dense)
                        ops.transr_step_claimed(emb, rel, w, st.ids[0], st.ids[1], st.ids[2], st.ids[3], reg, st.loss, None, st.scratch,
                                                row_slot, g_rows, g_rel, g_w, publish=st.publish)
                    st.published = True

                def body_bwd(st):
                    if d is None:
                        ops.transr_rows_to_dense(g_rows, row_slot, st.ids[0], st.ids[2], st.ids[3], g_dense)
                        prev_ids.copy_(st.ids)
                    else:
                        ops.transr_rows_to_dense(g_rows, row_slot, st.ids[0], st.ids[2], st.ids[3], g_dense, keep_ids=keep)
                        st.adam_rolling = dict(deferred=d, ids=(st.ids[0], st.ids[2], st.ids[3]), row_slot=row_slot)
                    st.adam_grads, st.adam_row_slot0 = [g_rows, g_rel, g_w], row_slot
                    return [g_dense, g_rel, g_w]

                def pre_submit(st):
                    # slot claims left behind by a step the rolling update never consumed (first launch after the capture warm-up,
                    # backward without update, update through the generic optimiser path): release them outside the graph
                    if st.updated != st.serial or st.serial == 0:
                        ops.transr_release_rows(g_dense, prev_ids.view(-1), row_slot)

                return (body_fwd, body_bwd, pre_submit) if d is not None else (body_fwd, body_bwd)

            key = None if deferred is None else (id(deferred), deferred.state_tensors()[0].data_ptr())
            if deferred is not None:
                deferred.ensure_phase()
            step = self._api_step("kg", ids[0].numel(), params, key, 4, make_bodies)
            if deferred is not None or not self.kg_deferred_adam or opt is None:  # (otherwise the next call may be able to defer: re-decide)
                self._kg_fast = self._make_kg_fast(step, params, opt, deferred)
            return step.submit(ids)
        self._settle()
        return KGLossFunction.apply(
            self._ids(heads), self._ids(relations), self._ids(positive_tails), self._ids(negative_tails),
            float(self._regularization_params[1]), self._user_entity_embedding.weight, self._relation_embedding.weight,
            self._trans_matrix,
        )

    # ------------------------------------------------------------------------------------------
    # A7 / A8: attention refresh
    # ------------------------------------------------------------------------------------------
    def _edge_index(self, heads, relations, tails, relation_indices) -> EdgeIndex:
        dev = self._device()
        heads, relations, tails = (torch.as_tensor(t).to(dev) for t in (heads, relations, tails))
        relation_indices = torch.as_tensor(relation_indices).to(dev)
        h64, r64, t64 = heads.to(torch.int64), relations.to(torch.int64), tails.to(torch.int64)
        # content key: two independent wrapping checksums (one host sync per refresh)
        c1 = int((h64 * 1000003 + t64 * 7919 + r64 * 104729).sum().item())
        c2 = int(((h64 ^ (t64 << 20)) * (r64 + 3)).sum().item())
        key = (heads.numel(), c1, c2, tuple(relation_indices.tolist()), dev)
        if self._edge_cache is None or key != self._edge_key:
            self._edge_cache = EdgeIndex(h64, r64, t64, relation_indices, self.node_num, chunk=self.spmm_chunk)
            self._edge_key = key
        return self._edge_cache

    @torch.no_grad()
    def _update_attention(self, heads, relations, tails, relation_indices) -> None:
        """model.py:318-366, entirely on the device: per-pair value path -> per-edge score ->
        duplicate merge + row softmax over CSR slots -> published as a coalesced COO view."""
        idx = self._edge_index(heads, relations, tails, relation_indices)
        mha = self._multi_head_attention
        params = mha.kernel_params()
        emb = self._user_entity_embedding.weight.detach()
        w = self._trans_matrix.detach()
        graph = idx.graph
        vals = graph.vals  # refreshed in place: pointers captured by CUDA graphs / the COO view stay valid
        p = mha.dropout_p if self.training else 0.0
        if self.score_mode == "kgat":
            rel = self._relation_embedding.weight.detach()
            x_t = ops.att_pair_project(emb, w, idx.pair_tail, idx.pair_rel)
            x_h = ops.att_pair_project(emb, w, idx.head_pair_node, idx.head_pair_rel)
            edge_score = ops.att_edge_scores_kgat(x_h, idx.head_pair_of_edge, x_t, idx.pair_of_edge, rel, idx.edge_rel)
            ones = getattr(idx, "_unit_weight", None)
            if ones is None:
                ones = idx._unit_weight = torch.ones_like(idx.edge_weight) if idx.edge_mult is None else idx.edge_mult.to(torch.float32)
            ops.att_row_softmax(graph.row_ptr, idx.slot_ptr, ones, vals, edge_score=edge_score)
        elif self.score_mode != "reference":
            raise ValueError(f"unknown score_mode {self.score_mode!r} (\"reference\" or \"kgat\")")
        elif p == 0.0:
            _, score = ops.att_pair_scores(emb, w, idx.pair_tail, idx.pair_rel, params, mha.head_num, mha.ln_eps)
            ops.att_row_softmax(graph.row_ptr, idx.slot_ptr, idx.edge_weight, vals, pair_score=score, pair_of_edge=idx.pair_of_edge)
        else:
            pair_v, _ = ops.att_pair_scores(emb, w, idx.pair_tail, idx.pair_rel, params, mha.head_num, mha.ln_eps, want_v=True, want_score=False)
            head_bits = None
            seed = 0
            if self._injected_head_bits is not None:
                head_bits = idx.sorted_from_input(self._injected_head_bits.to(emb.device))
            else:
                seed = int(torch.randint(0, 2**62, (1,)).item())
            edge_score = ops.att_edge_scores_dropout(pair_v, idx.pair_of_edge, params, p, head_bits, seed, 0, mha.head_num, mha.ln_eps)
            ops.att_row_softmax(graph.row_ptr, idx.slot_ptr, idx.edge_weight, vals, edge_score=edge_score)
        graph.refresh_transposed_values()
        coo = graph.coo_tensor()
        self.attentive_matrix.data = coo
        self._graph_cache = graph
        self._graph_key = (coo._values().data_ptr(), coo._indices().data_ptr(), coo._nnz(), coo.device)
        self._graph_version += 1

    # ------------------------------------------------------------------------------------------
    # A9: scoring (+ the fused ranking extension, SURVEY.md section 8f rank 1)
    # ------------------------------------------------------------------------------------------
    def _calc_score(self, user_ids, item_ids) -> torch.Tensor:
        tables = self._tables()
        users, items = self._ids(user_ids), self._ids(item_ids)
        if any(t.requires_grad for t in tables):  # autograd requested: differentiable (rare) path
            table = torch.cat(tables, dim=1)
            return torch.matmul(table[users], table[items].transpose(0, 1))
        return ops.sgemm_nt(ops.gather_concat(tables, users), ops.gather_concat(tables, items))

    @torch.no_grad()
    def recommend_topk(self, user_ids, item_ids, k: int, mask_ptr=None, mask_items=None, want_values: bool = False):
        """Scores ``user_ids x item_ids`` -> optional masking of known positives to -inf
        (metrics_calculator.py:118, main.py:592-600; CSR-like ``mask_ptr`` / ``mask_items`` int32 on the
        device, column positions) -> descending top-k with lowest-index-first ties
        (metrics_calculator.py:121 ``torch.sort`` order).  Returns int32 (n_users, k) column indices."""
        scores = self._calc_score(user_ids, item_ids)
        if mask_ptr is not None:
            ops.mask_scores_(scores, mask_ptr, mask_items)
        return ops.topk_rows(scores, k, want_values)

    @torch.no_grad()
    def recommend(self, user_ids, items, k: int = 20, exclude=None, require=None) -> "Recommendation":
        """Each user's top-``k`` problems among ``items``, in one call for any number of users, without a score matrix.

        ``user_ids``: 1-D int32 / int64, CPU or CUDA, in ``[0, user_num)``, repeats allowed.  ``items``: an int ``n`` (= ``arange(n)``)
        or a 1-D tensor of unique problem ids in ``[0, entity_num)``; its order breaks score ties.  ``exclude``: ``None`` or a
        ``metrics.InteractionCSR`` over the same ``user_num`` (e.g. training positives and solved problems); problem ``p`` is not
        recommended to ``u`` when it is in ``u``'s list.  ``require``: ``None`` or a list of non-empty groups of entity ids; ``p``
        passes a group when the current ``attentive_matrix`` stores an entry at ``(user_num + p, user_num + e)`` for some ``e`` of
        the group (whatever its value), and must pass every group -- e.g. ``[[rating_1600, ..., rating_1900], [tag_dp]]``.

        A score is exactly the fp32 value ``model(u, p, mode=PREDICT)`` and ``recommend_topk`` give; the order is score
        descending (NaN first, -0 after +0), then earlier position in ``items``.  ``1 <= k <= 128``; users with fewer than ``k``
        eligible problems get ``count < k`` and -1 / -inf padding.

        Like PREDICT the scores use row ``p`` of the propagated table (quirk Q4, reproduced on purpose, SURVEY.md), while the
        filter reads the problem's own CKG node ``user_num + p``, as ``explain`` does.  Uses the cached propagation after settling
        deferred KG rows, and honours train / eval mode as PREDICT does: call it in ``eval()``."""
        k = int(k)
        if not 1 <= k <= 128:
            raise ValueError(f"k must be in [1, 128], got {k}")
        dev = self._device()
        users, cand = self._users_and_items(user_ids, items, exclude)
        if require is not None:
            require = ops.require_groups(require, self._entity_num)
        # ranges and duplicates in one read-back: the only host synchronisation of the call
        dup = ops.duplicate_count(cand)
        users32, cand32 = ops.range_check([("user ids", users, self._user_num), ("item ids", cand, self._entity_num)], dev,
                                          flags=[("items holds duplicate ids", dup)])
        tables = self._tables()
        n_cand = None
        if require is not None:
            _, cand32, n_cand = ops.launch_recommend_filter(self._graph(), cand32, require, self._user_num)
        ex_ptr, ex_items = (exclude.ptr_dev.to(dev), exclude.items.to(dev)) if exclude is not None else (None, None)
        out_items, scores, count = ops.launch_recommend_topk(tables, users32, cand32, k, ex_ptr, ex_items, n_cand=n_cand)
        return Recommendation(items=out_items, scores=scores, count=count)

    @torch.no_grad()
    def recommend_capped(self, user_ids, items, k, caps, exclude=None, require=None) -> "Recommendation":
        """Each user's top-``k`` problems with at most ``cap`` problems of each capped group: a varied practice set, e.g.
        ``caps=[([t], 3) for t in tags] + [([r], 4) for r in ratings] + [([geometry], 0)]``.

        ``user_ids``, ``items``, ``k``, ``exclude`` and ``require`` mean what they mean for ``recommend``.  ``caps``: a list of at
        most 128 ``(group, cap)`` pairs, a group a non-empty list of entity ids and a cap an int >= 0.  Problem ``p`` is a member
        of a group when the current ``attentive_matrix`` stores an entry at ``(user_num + p, user_num + e)`` for some ``e`` of the
        group -- ``require``'s membership rule.  For every row, the eligible problems (``items``, then ``require``, minus
        ``exclude[u]``) are walked in ``recommend``'s order, score descending then earlier position in ``items``; ``p`` is
        accepted when every capped group it is a member of holds fewer than ``cap`` accepted problems so far, and the walk
        stops at ``k`` acceptances.  A problem in no capped group is always accepted; cap 0 keeps a group out entirely.

        Returns the accepted problems in acceptance order with their fp32 ``PREDICT`` scores, bit-identical to ``recommend``'s,
        and ``count``; positions from ``count`` on hold -1 / -inf.  With every cap >= ``k`` the result equals ``recommend``'s.
        The exact answer can lie arbitrarily deep in the ranking, so the GPU works in rounds (at most one per group plus one)
        and the host reads the number of unfinished rows after each.  ValueError for every argument ``recommend`` rejects and
        for malformed ``caps``.  Uses the cached propagation after settling deferred KG rows, draws no random numbers, and
        honours train / eval mode as PREDICT does: call it in ``eval()``."""
        k = int(k)
        if not 1 <= k <= 128:
            raise ValueError(f"k must be in [1, 128], got {k}")
        dev = self._device()
        users, cand = self._users_and_items(user_ids, items, exclude)
        groups, cap_values = ops.cap_groups(caps, self._entity_num)
        if require is not None:
            require = ops.require_groups(require, self._entity_num)
        dup = ops.duplicate_count(cand)
        users32, cand32 = ops.range_check([("user ids", users, self._user_num), ("item ids", cand, self._entity_num)], dev,
                                          flags=[("items holds duplicate ids", dup)])
        tables = self._tables()
        graph = self._graph()
        n_cand = None
        if require is not None:
            _, cand32, n_cand = ops.launch_recommend_filter(graph, cand32, require, self._user_num)
        ex_ptr, ex_items = (exclude.ptr_dev.to(dev), exclude.items.to(dev)) if exclude is not None else (None, None)
        out_items, scores, count, _ = ops.launch_recommend_capped(tables, graph, users32, cand32, k, groups, cap_values, self._user_num, ex_ptr,
                                                                  ex_items, n_cand=n_cand)
        return Recommendation(items=out_items, scores=scores, count=count)

    def _users_and_items(self, user_ids, items, exclude):
        """``user_ids`` / ``items`` of ``recommend`` and ``rank`` as int64 on the device (ranges are checked by the caller's
        read-back); ValueError for a malformed argument or an ``exclude`` over another number of users."""
        dev = self._device()
        users = torch.as_tensor(user_ids)
        if users.dim() != 1 or users.dtype not in (torch.int32, torch.int64):
            raise ValueError(f"user_ids must be a 1-D int32 / int64 tensor, got {users.dtype} of shape {tuple(users.shape)}")
        users = users.to(device=dev, dtype=torch.int64)
        if isinstance(items, int):
            if not 0 <= items <= self._entity_num:
                raise ValueError(f"items = {items} must lie in [0, {self._entity_num}]")
            cand = torch.arange(items, device=dev)
        else:
            cand = torch.as_tensor(items)
            if cand.dim() != 1 or cand.dtype not in (torch.int32, torch.int64):
                raise ValueError(f"items must be an int or a 1-D int32 / int64 tensor, got {cand.dtype} of shape {tuple(cand.shape)}")
            cand = cand.to(device=dev, dtype=torch.int64)
        if exclude is not None and exclude.user_num != self._user_num:
            raise ValueError(f"exclude covers {exclude.user_num} users, the model has {self._user_num}")
        return users, cand

    @torch.no_grad()
    def rank(self, user_ids, items, targets, exclude=None) -> "TargetRanks":
        """The exact rank of every held-out problem of every listed user among ``items``, in one call, without a score matrix.

        ``user_ids``, ``items`` and ``exclude`` are those of ``recommend`` (ints / tensors, repeats of users allowed, ``items``'
        order breaks score ties).  ``targets``: a ``metrics.InteractionCSR`` over the same ``user_num`` of the problems to rank,
        e.g. the test split; row ``b`` of the result holds ``targets[user_ids[b]]`` in ascending id.

        Score ``s(u, c)``: the fp32 ``model(u, c, mode=PREDICT)`` value (the sequential ``fmaf`` chain over ``E0|...|EL``,
        zero-padded to 16 columns; quirk Q4: row ``c``).  Key ``K(u, c) = (float_key(s) << 32) | (0xFFFFFFFF - pos(c))``, ``pos``
        the position in ``items``: ``recommend``'s order.  A problem is eligible for ``u`` when it is in ``items`` and not in
        ``exclude[u]``.  For an eligible target ``p``::

            rank(u, p) = #{c eligible for u : K(u, c) > K(u, p)}

        so ``rank < k <= 128`` means ``recommend(u, items, k, exclude).items[b, rank] == p``.  A target that is not eligible gets
        rank -1 (its score is still given).  ``eligible[b]`` counts the eligible problems of ``u``.  Only integers are counted, so
        the result does not depend on how the GPU splits the work.

        ValueError for every argument ``recommend`` rejects, for ``targets`` over another number of users, and for ``targets``
        whose item range exceeds ``entity_num``.  Uses the cached propagation after settling deferred KG rows, and honours train /
        eval mode as PREDICT does: call it in ``eval()``.  One host synchronisation (the range-check read-back)."""
        dev = self._device()
        users, cand = self._users_and_items(user_ids, items, exclude)
        if targets.user_num != self._user_num:
            raise ValueError(f"targets cover {targets.user_num} users, the model has {self._user_num}")
        if targets.item_num > self._entity_num:
            raise ValueError(f"targets hold problem ids up to {targets.item_num - 1}, the model has {self._entity_num} entities")
        t_ptr, t_items = targets.ptr_dev.to(dev), targets.items.to(dev)
        out_ptr = ops.target_rows(t_ptr, users)
        users32, cand32, n_targets = ops.range_check([("user ids", users, self._user_num), ("item ids", cand, self._entity_num)], dev,
                                                     flags=[("items holds duplicate ids", ops.duplicate_count(cand))], values=[out_ptr[-1]])
        tables = self._tables()
        ex_ptr, ex_items = (exclude.ptr_dev.to(dev), exclude.items.to(dev)) if exclude is not None else (None, None)
        ptr, t, scores, rank, eligible = ops.launch_rank(tables, users32, cand32, t_ptr, t_items, out_ptr, n_targets, ex_ptr, ex_items,
                                                         arange=isinstance(items, int), n_pos=self._entity_num)
        return TargetRanks(ptr=ptr, items=t, scores=scores, rank=rank, eligible=eligible)

    def _transr_params(self):
        """The trained TransR half (entity table after settling deferred KG rows, relation embeddings, projections), read without
        invalidating any cache or captured step."""
        self._settle()
        return self._emb_raw().detach(), self._relation_embedding._parameters["weight"].detach(), self._trans_matrix.detach()

    @staticmethod
    def _exclude_keys(exclude, node_num: int, relation_num: int):
        if exclude is None:
            return None
        if exclude.node_num != node_num or exclude.relation_num != relation_num:
            raise ValueError(f"exclude is a TripleSet over {exclude.node_num} nodes and {exclude.relation_num} relations, the model has "
                             f"{node_num} and {relation_num}")
        return exclude.keys

    @torch.no_grad()
    def complete(self, heads, relations, candidates, k: int = 10, exclude=None) -> "Completion":
        """Knowledge-graph completion with the trained TransR half: for every query ``(heads[q], relations[q], ?)`` the ``k`` most
        plausible tails among ``candidates``, in one call, without an energy matrix.

        ``heads`` / ``relations``: 1-D int32 / int64 CKG node ids in ``[0, node_num)`` and relation ids in ``[0, relation_num)``
        -- the ids of ``CKG.heads / relations / tails``, the triples TransR trains on.  The edge list holds each relation's
        inverse, so "which rating has problem p" is the query ``(user_num + p, r)`` with ``r`` the inverse of the rating
        relation.  ``candidates``: an int ``n`` (= ``arange(n)``) or a 1-D tensor of unique node ids; its order breaks ties.
        ``exclude``: ``None`` or a ``metrics.TripleSet`` of known triples; ``c`` is not returned for ``(h, r)`` when ``(h, r, c)``
        is in it (the filtered protocol).

        Energy ``E(h, r, t) = ||e_h W_r + e_r - e_t W_r||^2`` in fp32, bit-identical to the per-sample term of the TransR loss.
        Order: energy ascending (the key ``float_key(-E)`` of ``recommend``'s order; a NaN energy first), then earlier position
        in ``candidates``.  ``1 <= k <= 128``; queries with fewer than ``k`` eligible candidates get ``count < k`` and -1 / +inf
        padding.

        Settles deferred KG rows and reads the parameters only: no cache or captured step is invalidated and no RNG is drawn,
        so calling it between training steps leaves training unchanged.  ValueError for every malformed argument.  One host
        synchronisation (the range-check read-back)."""
        self._device()
        emb, rel, w = self._transr_params()
        ex = self._exclude_keys(exclude, self.node_num, self._relation_num)
        tails, energy, count = ops.complete_topk(emb, rel, w, self._query_ids(heads, "heads"), self._query_ids(relations, "relations"),
                                                 self._candidates(candidates), k, ex)
        return Completion(tails=tails, energy=energy, count=count)

    @torch.no_grad()
    def kg_rank(self, heads, relations, tails, candidates, exclude=None) -> "TailRanks":
        """The filtered rank of each triple's tail among ``candidates``: link prediction for the trained TransR half.

        Arguments as for ``complete``; ``tails``: 1-D node ids of the same length.  A candidate ``c`` is eligible for
        ``(h, r, t)`` when ``(h, r, c)`` is not in ``exclude`` or ``c == t`` (the target itself stays eligible).  With ``complete``'s
        key ``K``::

            rank(q) = #{c eligible, c != t : K(q, c) > K(q, t)}

        so ``rank < k`` means ``complete(..., k, exclude minus (h, r, t)).tails[q, rank] == t``.  -1 when ``t`` is not in
        ``candidates``.  ``energy`` is ``E(h, r, t)`` in any case, and ``energy(h, r, n) - energy(h, r, p)`` is the TransR loss's
        margin bit for bit.  Only integers are counted, so the result does not depend on how the GPU splits the work.  Reads
        parameters only, as ``complete``; one host synchronisation."""
        self._device()
        emb, rel, w = self._transr_params()
        ex = self._exclude_keys(exclude, self.node_num, self._relation_num)
        energy, rank, eligible = ops.kg_rank(emb, rel, w, self._query_ids(heads, "heads"), self._query_ids(relations, "relations"),
                                             self._query_ids(tails, "tails"), self._candidates(candidates), ex)
        return TailRanks(energy=energy, rank=rank, eligible=eligible)

    def _query_ids(self, ids, name: str) -> torch.Tensor:
        t = torch.as_tensor(ids)
        if t.dim() != 1 or t.dtype not in (torch.int32, torch.int64):
            raise ValueError(f"{name} must be a 1-D int32 / int64 tensor, got {t.dtype} of shape {tuple(t.shape)}")
        return t.to(device=self._device(), dtype=torch.int64)

    def _candidates(self, candidates):
        if isinstance(candidates, bool) or not isinstance(candidates, (int, torch.Tensor)):
            raise ValueError("candidates must be an int or a 1-D int32 / int64 tensor of node ids")
        return candidates if isinstance(candidates, int) else self._query_ids(candidates, "candidates")

    @torch.no_grad()
    def explain(self, user_ids, item_ids, k: int = 10, max_hops: int | None = None) -> "PathExplanation":
        """Why item ``item_ids[j]`` reaches user ``user_ids[j]``: the top-``k`` simple paths of 1 .. ``max_hops`` hops from the
        user's CKG node to the item's CKG node ``user_num + item`` through the current ``attentive_matrix`` A, ranked by the
        product of their attention values (weight descending, then fewer hops, then lower (v1, v2)), with the number and
        summed weight of all such paths per length.  A hop (v, w) is a stored entry A[v, w]: the direction in which
        propagation carries w's embedding into v.

        ``max_hops`` defaults to ``min(3, number of layers)``.  Ids: int32 / int64, CPU or CUDA; users in
        ``[0, user_num)``, items in ``[0, entity_num)``.

        Unlike PREDICT, which scores problem ``p`` from row ``p`` of the propagated table (quirk Q4, reproduced on purpose,
        SURVEY.md), the paths end at the problem's own CKG node ``user_num + p``, the node the graph links to its solvers,
        contest, tags and rating.

        Reads only the attentive matrix: it does not settle deferred KG rows, invalidate caches or captured steps, or draw
        from torch's RNG, so calling it between training steps leaves training unchanged."""
        max_hops = min(3, self._layer_num) if max_hops is None else int(max_hops)
        users, items = self._ids(user_ids).flatten(), self._ids(item_ids).flatten()
        if users.numel() != items.numel():
            raise ValueError(f"user_ids and item_ids differ in length ({users.numel()} != {items.numel()})")
        if users.numel():
            lo_u, hi_u, lo_i, hi_i = torch.stack([users.min(), users.max(), items.min(), items.max()]).tolist()
            if lo_u < 0 or hi_u >= self._user_num:
                raise ValueError(f"user ids must lie in [0, {self._user_num})")
            if lo_i < 0 or hi_i >= self._entity_num:
                raise ValueError(f"item ids must lie in [0, {self._entity_num})")
        nodes, slots, hops, weight, count, mass = ops.explain_paths(self._graph(), users, items + self._user_num, k, max_hops)
        return PathExplanation(nodes=nodes, slots=slots, hops=hops, weight=weight, count=count, mass=mass)

    # ------------------------------------------------------------------------------------------
    # A10: optimisers
    # ------------------------------------------------------------------------------------------
    def build_optimizer(self, cf_lr: float, kg_lr: float) -> None:
        """Two independent Adam optimisers over all parameters (model.py:393-405)."""
        self._cf_optimizer = FusedAdam(params=self.parameters(), lr=cf_lr)
        self._kg_optimizer = FusedAdam(params=self.parameters(), lr=kg_lr)

    def update_cf_weights(self) -> None:
        step = self._last_step.get("cf")
        if step is None or not step.try_fused_update(self._cf_optimizer):
            self._cf_optimizer.step_and_zero()

    def update_kg_weights(self) -> None:
        step = self._last_step.get("kg")
        if step is None or not step.try_fused_update(self._kg_optimizer):
            self._kg_optimizer.step_and_zero()

    # ------------------------------------------------------------------------------------------
    # A2: dispatch
    # ------------------------------------------------------------------------------------------
    def forward(self, *args: Any, mode: KGATMode) -> torch.Tensor | None:  # noqa: ANN401
        match mode:
            case KGATMode.TRAIN_CF:
                self._settle()
                return self._calc_cf_loss(*args)
            case KGATMode.TRAIN_KG:
                return self._calc_kg_loss(*args)
            case KGATMode.UPDATE_ATTENTION:
                self._settle()
                self._update_attention(*args)
                return None
            case KGATMode.PREDICT:
                self._settle()
                return self._calc_score(*args)
        raise ValueError(f"unknown mode {mode!r}")

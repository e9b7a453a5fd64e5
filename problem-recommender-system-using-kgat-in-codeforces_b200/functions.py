"""Autograd glue: the hand-written forward/backward kernels wrapped as ``torch.autograd.Function``s
so that the reference's driver code (``loss.backward()``, ``main.py:312, 341``) keeps working.

* ``CFLossFunction``      TRAIN_CF: 3-layer attentive propagation + BPR loss (model.py:165-202)
* ``KGLossFunction``      TRAIN_KG: TransR loss (model.py:204-261)
* ``PropagateFunction``   propagation alone, differentiable w.r.t. dense output gradients
                          (used by PREDICT when autograd is enabled and by ``Aggregator.forward``)

No dense N x 176 concat is materialised: layer outputs stay in their own row-major buffers and the
BPR kernels gather from the four tables directly (K3 of SURVEY.md section 2b).
"""

from __future__ import annotations

import contextlib
import gc
from dataclasses import dataclass, field

import torch

from . import ops
from .graph import AttentiveGraph

f32 = torch.float32


@dataclass
class DropoutSpec:
    """Message-dropout configuration of one forward pass (aggregator.py:62)."""

    ps: list[float]  # per layer; 0 disables (eval mode)
    seed: int = 0
    keep_bits: list | None = None  # optional injected masks, one int32 [N, ceil(d_out/32)] per layer
    seed_dev: torch.Tensor | None = None  # optional device u64/i64 mixed into the seed (graph replay)


@dataclass
class PropState:
    tables: list  # [E0, E1, ..., EL]
    side: list = field(default_factory=list)  # S_l = A @ E_{l-1}
    inv_norm: list = field(default_factory=list)
    flags: list = field(default_factory=list)
    ps: list = field(default_factory=list)


import os as _os

_L1_GRID = _os.environ.get("KGAT_L1_GRID") == "1"  # A/B switch: first layer through the grid-per-task kernel (early exit on dead rows)

# Test hook: fill every freshly allocated propagation buffer with NaN (0xFF for flag bytes), so that a pruned step that
# read a row outside its frontier would poison the loss / gradients (tests/test_gpu_pruning.py).
POISON_STALE_ROWS = False


def _buf(*shape, dtype=f32, device=None) -> torch.Tensor:
    if not POISON_STALE_ROWS:
        return torch.empty(*shape, dtype=dtype, device=device)
    return torch.full(shape, 255 if dtype == torch.uint8 else float("nan"), dtype=dtype, device=device)


def _row_args(frontier, level: int) -> dict:
    if frontier is None:
        return {}
    return {"rows": frontier.rows(level), "n_rows_dev": frontier.count(level), "max_rows": frontier.cap(level), "tag": f"_L{level}"}


def propagate_forward(graph: AttentiveGraph, e0: torch.Tensor, layers, drop: DropoutSpec, save: bool = True, frontier=None) -> PropState:
    """E_{l} = Agg_l(E_{l-1}, A) for all layers (model.py:124-140, aggregator.py:37-65).

    With a ``frontier`` (frontier.Frontier, already built for this batch) layer ``l`` is computed for the rows of level
    ``l`` only; the other rows of the returned tables hold stale bytes that nothing downstream reads."""
    n = e0.shape[0]
    dev = e0.device
    st = PropState(tables=[e0])
    for l, (w1, b1, w2, b2) in enumerate(layers):
        x = st.tables[-1]
        d_out = w1.shape[0]
        if frontier is None:
            side = graph.matmul(x, out=_buf(n, x.shape[1], device=dev))
        elif l == 0 and _L1_GRID:
            side = graph.matmul(x, out=_buf(n, x.shape[1], device=dev), row_mask=frontier.mask(1), tag="_L1")
        else:
            side = graph.matmul(x, out=_buf(n, x.shape[1], device=dev), row_mask=frontier.mask(l + 1), rows=frontier.rows(l + 1),
                                n_rows_dev=frontier.count(l + 1), tag=f"_L{l + 1}")
        out = _buf(n, d_out, device=dev)
        inv = _buf(n, device=dev) if save else None
        flags = _buf(n, d_out, dtype=torch.uint8, device=dev) if save else None
        p = float(drop.ps[l])
        ops.biagg_forward(
            x, side, w1, b1, w2, b2, out, inv, flags, dropout_p=p, seed=drop.seed, offset=(l + 1) << 40,
            keep_bits=None if drop.keep_bits is None else drop.keep_bits[l], seed_dev=drop.seed_dev, **_row_args(frontier, l + 1),
        )
        st.tables.append(out)
        if save:
            st.side.append(side)
            st.inv_norm.append(inv)
            st.flags.append(flags)
            st.ps.append(p)
    return st


def last_table_grad(st: PropState, frontier=None) -> torch.Tensor:
    """Zeroed gradient buffer of the last table (only the frontier's batch rows are zeroed / valid under pruning)."""
    if frontier is None:
        return torch.zeros_like(st.tables[-1])
    g = _buf(*st.tables[-1].shape, device=st.tables[-1].device)
    top = frontier.n_layers
    ops.frontier_zero_rows(g, frontier.rows(top), frontier.count(top), frontier.cap(top))
    return g


def propagate_backward(graph: AttentiveGraph, st: PropState, layers, g_last: torch.Tensor, inject, frontier=None):
    """Backward through all layers.  ``g_last`` is the dense gradient w.r.t. the last table;
    ``inject(l, G)`` adds the loss's direct gradient for table ``l`` into the dense buffer ``G``
    (called for l = L-1 .. 0, after the propagated part of G has been written).
    Returns (g_E0, [(gW1, gb1, gW2, gb2) per layer]).

    With a ``frontier`` the backward of layer ``l`` runs over level ``l``'s rows: ``A^T g_S`` gathers only the edges whose
    source row is in level ``l`` and produces the rows of level ``l-1`` (all rows for the embedding table, whose
    gradient the dense Adam sweep reads in full)."""
    n = st.tables[0].shape[0]
    dev = g_last.device
    g = g_last
    param_grads = [None] * len(layers)
    for l in range(len(layers), 0, -1):
        w1, b1, w2, b2 = layers[l - 1]
        x = st.tables[l - 1]
        d_in, d_out = x.shape[1], w1.shape[0]
        n_ctas = ops.biagg_backward_ctas(n if frontier is None else frontier.cap(l), d_in, d_out, rows=frontier is not None)
        partials = torch.empty(n_ctas * (2 * d_in * d_out + 2 * d_out), dtype=f32, device=dev)
        g_s = _buf(n, d_in, device=dev)
        g_e = _buf(n, d_in, device=dev)
        ops.biagg_backward(g, st.tables[l], st.inv_norm[l - 1], st.flags[l - 1], x, st.side[l - 1], w1, w2, st.ps[l - 1],
                           g_s, g_e, partials, n_ctas, **_row_args(frontier, l))
        gw1, gb1, gw2, gb2 = torch.empty_like(w1), torch.empty_like(b1), torch.empty_like(w2), torch.empty_like(b2)
        ops.biagg_reduce_param_grads(partials, n_ctas, d_in, d_out, gw1, gb1, gw2, gb2)
        param_grads[l - 1] = (gw1, gb1, gw2, gb2)
        if frontier is None:
            g_prev = graph.matmul_t(g_s, addend=g_e)  # dL/dE_{l-1} = g_E(direct) + A^T g_S
        elif l > 1 and frontier.scatter_backward:
            # few gradient sources (level l) feeding the rows of level l-1: scatter their edges instead of streaming every
            # edge of every destination row past the source bitmap
            g_prev = _buf(n, d_in, device=dev)
            ops.frontier_zero_rows(g_prev, frontier.rows(l - 1), frontier.count(l - 1), frontier.cap(l - 1))
            ops.spmm_scatter_rows(graph.plan, graph.col_idx, graph.vals, g_s, g_prev, frontier.rows(l), frontier.count(l), frontier.cap(l),
                                  frontier.mask(l), addend=g_e, tag=f"_L{l}")
        else:
            below = {"row_mask": frontier.mask(l - 1), "rows": frontier.rows(l - 1), "n_rows_dev": frontier.count(l - 1)} if l > 1 else {}
            g_prev = graph.matmul_t(g_s, out=_buf(n, d_in, device=dev), addend=g_e, edge_mask=frontier.mask(l), tag=f"_L{l}", **below)
        inject(l - 1, g_prev)
        g = g_prev
    return g, param_grads


def _bump(frontier) -> int:
    frontier.serial = getattr(frontier, "serial", 0) + 1
    return frontier.serial


def _flat_layers(flat):
    return [tuple(flat[i : i + 4]) for i in range(0, len(flat), 4)]


class CFLossFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, graph, users, pos, neg, reg, drop, frontier, e0, *flat):
        layers = _flat_layers([t.detach() for t in flat])
        e0d = e0.detach()
        if frontier is not None:
            frontier.build([users, pos, neg])
        st = propagate_forward(graph, e0d, layers, drop, save=True, frontier=frontier)
        b = users.numel()
        loss = torch.empty(1, dtype=f32, device=e0.device)
        scratch = torch.empty(2 * b, dtype=f32, device=e0.device)
        ops.bpr_forward(st.tables, users, pos, neg, reg, loss, scratch)
        ctx.graph, ctx.st, ctx.layers = graph, st, layers
        ctx.ids = (users, pos, neg)
        ctx.reg, ctx.scratch = reg, scratch
        ctx.frontier = frontier
        ctx.frontier_serial = None if frontier is None else _bump(frontier)
        return loss.reshape(())

    @staticmethod
    def backward(ctx, g_loss):
        st, layers, graph = ctx.st, ctx.layers, ctx.graph
        users, pos, neg = ctx.ids
        frontier = ctx.frontier
        if frontier is not None and frontier.serial != ctx.frontier_serial:
            frontier.build([users, pos, neg])  # another forward re-used the frontier buffers in between: rebuild for this batch
            ctx.frontier_serial = _bump(frontier)
        g_loss = g_loss.reshape(1).to(f32).contiguous()
        n_tab = len(st.tables)

        def inject(l, buf):
            grads = [None] * n_tab
            grads[l] = buf
            ops.bpr_backward(st.tables, grads, users, pos, neg, ctx.reg, ctx.scratch, g_loss)

        g_last = last_table_grad(st, frontier)
        inject(n_tab - 1, g_last)
        g_e0, pgrads = propagate_backward(graph, st, layers, g_last, inject, frontier=frontier)
        flat = [t for grp in pgrads for t in grp]
        return (None, None, None, None, None, None, None, g_e0, *flat)


class PropagateFunction(torch.autograd.Function):
    """(E1, ..., EL) = propagate(E0); backward takes dense output gradients."""

    @staticmethod
    def forward(ctx, graph, drop, e0, *flat):
        layers = _flat_layers([t.detach() for t in flat])
        st = propagate_forward(graph, e0.detach(), layers, drop, save=True)
        ctx.graph, ctx.st, ctx.layers = graph, st, layers
        return tuple(st.tables[1:])

    @staticmethod
    def backward(ctx, *g_tables):
        st, layers, graph = ctx.st, ctx.layers, ctx.graph
        g_last = g_tables[-1]
        g_last = torch.zeros_like(st.tables[-1]) if g_last is None else g_last.contiguous()

        def inject(l, buf):
            if l >= 1 and g_tables[l - 1] is not None:
                buf.add_(g_tables[l - 1])

        g_e0, pgrads = propagate_backward(graph, st, layers, g_last, inject)
        flat = [t for grp in pgrads for t in grp]
        return (None, None, g_e0, *flat)


class KGLossFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, heads, rels, pos_t, neg_t, reg, emb, rel_emb, w):
        embd, reld, wd = emb.detach(), rel_emb.detach(), w.detach()
        b = heads.numel()
        loss = torch.empty(1, dtype=f32, device=emb.device)
        scratch = torch.empty(2 * b, dtype=f32, device=emb.device)
        ops.transr_forward(embd, reld, wd, heads, rels, pos_t, neg_t, reg, loss, scratch)
        ctx.saved = (embd, reld, wd, heads, rels, pos_t, neg_t, scratch)
        ctx.reg = reg
        return loss.reshape(())

    @staticmethod
    def backward(ctx, g_loss):
        embd, reld, wd, heads, rels, pos_t, neg_t, scratch = ctx.saved
        g_loss = g_loss.reshape(1).to(f32).contiguous()
        g_emb, g_rel, g_w = torch.zeros_like(embd), torch.zeros_like(reld), torch.zeros_like(wd)
        ops.transr_backward(embd, reld, wd, heads, rels, pos_t, neg_t, ctx.reg, scratch, g_loss, g_emb, g_rel, g_w)
        return (None, None, None, None, None, g_emb, g_rel, g_w)


# ----------------------------------------------------------------------------------------------
# CUDA-graph fast path behind the reference-facing API (model(...), loss.backward(), update_*_weights(), loss.item())
# ----------------------------------------------------------------------------------------------
@contextlib.contextmanager
def capture_graph(graph: torch.cuda.CUDAGraph):
    """``torch.cuda.graph(graph)`` with Python's cyclic garbage collector paused during the capture.  Captured steps and
    optimiser plans sit in reference cycles, so an unreachable one is destroyed whenever a collection runs; a collection in the
    middle of a capture would destroy its CUDAGraph there, with CUDA calls that a capturing stream does not permit, and
    invalidate the capture.  ``torch.cuda.graph`` collects once before the capture begins."""
    enabled = gc.isenabled()
    gc.disable()
    try:
        with torch.cuda.graph(graph):
            yield
    finally:
        if enabled:
            gc.enable()


class GraphedStep:
    """One training mode's forward AND backward captured as ONE CUDA graph over static buffers.

    The reference driver always runs ``loss = model(...); loss.backward(); model.update_*_weights(); loss.item()``
    (main.py:306-314, 334-343); an epoch is ~15 k such steps and a KG step is ~60 us of GPU work, so the API path is
    bound by host time per call.  Here ``model(...)`` is one C call (``kgat_step_submit``: copy of the step's ids into
    the static buffer + launch of the graph) whose graph computes the loss, publishes it to a pinned host ring
    (``kgat_publish_loss``) and goes straight on to the gradients w.r.t. a unit upstream gradient; the returned
    ``LazyLoss`` makes ``loss.backward()`` a hand-over of the static gradient buffers (no autograd engine run) and
    ``loss.item()`` a host-side poll of the ring (no stream synchronisation: the backward / Adam kernels queued behind
    the loss keep running).  Anything else done with the loss falls back to a real autograd node (``GraphedLoss``).
    """

    RING = 1024  # published losses kept readable on the host

    def __init__(self, params, batch: int, n_ids: int, body_fwd, body_bwd):
        from . import _lib

        dev = params[0].device
        self.params = list(params)
        self.device = dev
        self.ids = torch.zeros(n_ids, batch, dtype=torch.int64, device=dev)
        self.loss = torch.zeros(1, dtype=f32, device=dev)
        self.loss_scalar = self.loss.reshape(())
        self.g_loss = torch.ones(1, dtype=f32, device=dev)  # the unit upstream gradient the captured backward uses
        self.scratch = torch.empty(ops.transr_scratch_numel(batch, params[0].shape[-1]), dtype=f32, device=dev)
        self.counter = torch.zeros(1, dtype=torch.int64, device=dev)  # forward calls so far (dropout stream)
        self.pub_serial = torch.zeros(1, dtype=torch.int64, device=dev)  # losses published so far (device side)
        self.ring = torch.zeros(self.RING, dtype=torch.int64).pin_memory()  # (serial << 32) | float bits, written by the GPU
        self._ring_words = self.ring.numpy()
        self._ring_f32 = self._ring_words.view("<f4")
        self.serial = 0  # forward launches so far (host side; equals pub_serial once the launches have run)
        self.adopted = 0  # serial whose gradients were handed to the parameters
        self.updated = 0  # serial whose gradients went through the fused optimiser step
        self.grads = None
        self.adam_grads = None  # optional: the gradient tensors the fused optimiser replay reads instead of `grads` ...
        self.adam_row_slot0 = None  # ... with compact rows for the first parameter (ops.adam_apply row_slot0)
        self.adam_rolling = None  # ... or the rolling-window update of optim.DeferredRows: dict(deferred, ids, row_slot)
        self.pre_submit = None  # optional host-side check run before every launch (set by the model)
        self._adam = {}
        self._lib = _lib.load()
        # the captured graph bakes in the addresses of every buffer the bodies' closures own (needed-row frontier, static
        # gradient tables, previous-batch ids ...): keep the closures -- and with them those buffers -- alive as long as the graph
        self._bodies = (body_fwd, body_bwd)

        # the loss kernel of the forward body publishes (serial, loss) itself when the body passes ``publish=st.publish`` on and
        # reports so (``st.published = True``); otherwise a one-thread launch does it
        self.publish = ops.publish_args(self.pub_serial, self.ring)
        self.published = False

        def whole(st):
            st.published = False
            body_fwd(st)
            if not st.published:
                ops.publish_loss(st.loss, st.pub_serial, st.ring)
            return body_bwd(st)

        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):  # eager warm-up (no parameter is modified by forward / backward)
            whole(self)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        self.pub_serial.zero_()
        self.ring.zero_()
        torch.cuda.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        with capture_graph(self.graph):
            self.grads = whole(self)
        self._exec = self.graph.raw_cuda_graph_exec()
        self._ids_ptr = self.ids.data_ptr()
        self._ids_bytes = self.ids.numel() * 8
        self._batch, self._row_bytes = batch, batch * 8
        self._dev_index = dev.index if dev.index is not None else torch.cuda.current_device()
        self._grad_key = tuple(g.data_ptr() for g in self.grads)
        self._param_ids = tuple(id(p) for p in self.params)

    # -- forward ---------------------------------------------------------------------------------
    def submit(self, ids) -> "LazyLoss":
        """Copy the ids into the static buffer and launch forward + backward.  ``ids``: int64 tensors on the device or in
        pinned host memory; consecutive rows of one [n_ids, B] block travel in the same call as the launch."""
        for p, g in zip(self.params, self.grads):
            pg = p.grad
            if pg is not None and (pg is g or pg.data_ptr() == g.data_ptr()):
                p.grad = pg.clone()  # an un-applied gradient still aliases our buffer (accumulation): keep its value
        # consecutive int64 rows of one [n_ids, B] block (device, or host: pinned or not, cudaMemcpyAsync stages pageable memory
        # before it returns) travel in the same C call as the launch
        if self.pre_submit is not None:
            self.pre_submit(self)
        first = ids[0]
        base = first.data_ptr()
        stride = self._row_bytes
        one_block = True
        for i, t in enumerate(ids):
            if t.data_ptr() != base + i * stride or t.numel() != self._batch:
                one_block = False
                break
        stream = torch._C._cuda_getCurrentRawStream(self._dev_index)
        if one_block:
            rc = self._lib.kgat_step_submit(self._ids_ptr, base, self._ids_bytes, self._exec, stream)
        else:
            for dst, src in zip(self.ids, ids):
                dst.copy_(src, non_blocking=True)
            rc = self._lib.kgat_graph_launch(self._exec, stream)
        if rc != 0:
            from ._lib import check

            check(rc, "api step launch")
        self.serial += 1
        return LazyLoss.make(self)

    # -- backward --------------------------------------------------------------------------------
    def adopt_grads(self, serial: int) -> None:
        """``loss.backward()``: hand the static gradient buffers (computed at forward time) to the parameters."""
        if serial != self.serial:
            raise RuntimeError(
                "kgat_b200: backward() of a loss whose forward buffers were reused by a later model(...) call. "
                "The API fast path assumes forward -> backward -> update per step (as the reference driver does); "
                "set model.api_graphs = False for free-form autograd use."
            )
        if self.adopted == serial:
            raise RuntimeError("Trying to backward through the graph a second time (kgat_b200 API fast path keeps no graph to retain)")
        self.adopted = serial
        for p, g in zip(self.params, self.grads):
            if p.grad is None:
                p.grad = g
            else:
                p.grad = p.grad + g  # accumulation: never in place into a buffer we may not own

    # -- optimiser -------------------------------------------------------------------------------
    def try_fused_update(self, opt) -> bool:
        """``update_*_weights()`` right after ``backward()``: replay the captured Adam step over (params, static grads) and
        drop the gradients.  Returns False (nothing done) whenever the situation is anything but exactly that."""
        if self.adopted != self.serial or self.updated == self.serial:
            return False
        for p, g in zip(self.params, self.grads):
            if p.grad is not g:
                return False
        plan = opt.fast_plan(self.params, self.adam_grads if self.adam_grads is not None else self.grads, self._grad_key,
                             row_slot0=self.adam_row_slot0, rolling=self.adam_rolling)
        if plan is None:
            return False
        opt.fast_replay(plan, self.params)
        self.updated = self.serial
        return True

    # -- loss value ------------------------------------------------------------------------------
    def read_loss(self, serial: int) -> float:
        """Host value of the loss published by forward number ``serial`` (polls the pinned ring; no stream sync)."""
        import time

        if self.serial - serial >= self.RING:
            raise RuntimeError("kgat_b200: this loss value is no longer available (more than 1024 later steps were issued)")
        slot = serial % self.RING
        words = self._ring_words
        want = serial & 0xFFFFFFFF
        spins = 0
        deadline = None
        while True:
            w = int(words[slot])
            if ((w >> 32) & 0xFFFFFFFF) == want:
                return float(self._ring_f32[2 * slot])
            spins += 1
            if spins & 1023 == 0:
                now = time.perf_counter()
                if deadline is None:
                    deadline = now + 20.0
                elif now > deadline:
                    torch.cuda.synchronize()  # surfaces a CUDA error if the step faulted
                    if ((int(words[slot]) >> 32) & 0xFFFFFFFF) == want:
                        return float(self._ring_f32[2 * slot])
                    raise RuntimeError("kgat_b200: the loss of this step was never published")

    def loss_tensor(self, serial: int) -> torch.Tensor:
        """A plain 0-dim device tensor holding the loss of forward ``serial`` (no autograd)."""
        if serial == self.serial:
            return self.loss_scalar.clone()
        return torch.tensor(self.read_loss(serial), dtype=f32, device=self.device)


class LazyLoss(torch.Tensor):
    """The 0-dim loss returned by the API fast path.  ``backward()`` / ``item()`` / ``float()`` / ``detach()`` are served
    directly by the step's static buffers; any other use materialises a real autograd-tracked tensor first."""

    @staticmethod
    def make(step: GraphedStep) -> "LazyLoss":
        t = torch.Tensor._make_subclass(LazyLoss, step.loss_scalar)
        t._step, t._serial, t._real = step, step.serial, None
        return t

    def _materialize(self) -> torch.Tensor:
        if self._real is None:
            step = self._step
            if self._serial == step.serial:
                self._real = GraphedLoss.apply(step, self._serial, *step.params)
            else:
                self._real = step.loss_tensor(self._serial)
        return self._real

    def backward(self, gradient=None, retain_graph=None, create_graph=False, inputs=None):
        if gradient is not None or create_graph or inputs is not None or self._real is not None:
            return self._materialize().backward(gradient, retain_graph, create_graph, inputs)
        self._step.adopt_grads(self._serial)

    def item(self) -> float:
        return self._step.read_loss(self._serial)

    def __float__(self) -> float:
        return self._step.read_loss(self._serial)

    def tolist(self) -> float:
        return self._step.read_loss(self._serial)

    def detach(self) -> torch.Tensor:
        return self._step.loss_tensor(self._serial)

    def __repr__(self) -> str:
        return f"tensor({self.item():.4f}, device='{self._step.device}', grad_fn=<KgatGraphedStep>)"

    @classmethod
    def __torch_function__(cls, func, types, args=(), kwargs=None):
        def real(a):
            if isinstance(a, LazyLoss):
                return a._materialize()
            if isinstance(a, (list, tuple)):
                return type(a)(real(x) for x in a)
            return a

        with torch._C.DisableTorchFunctionSubclass():
            return func(*[real(a) for a in args], **{k: real(v) for k, v in (kwargs or {}).items()})


class GraphedLoss(torch.autograd.Function):
    """Slow-path autograd node of a graphed step (composition with other tensors, non-unit upstream gradient, ...)."""

    @staticmethod
    def forward(ctx, step: GraphedStep, serial: int, *params):
        ctx.step, ctx.serial = step, serial
        return step.loss_scalar.clone()

    @staticmethod
    def backward(ctx, g_loss):
        step = ctx.step
        if ctx.serial != step.serial:
            raise RuntimeError(
                "kgat_b200: backward() of a loss whose forward buffers were reused by a later model(...) call. "
                "The API fast path assumes forward -> backward -> update per step (as the reference driver does); "
                "set model.api_graphs = False for free-form autograd use."
            )
        # the step's graph already produced the gradients for a unit upstream gradient; they are linear in it
        return (None, None, *[g * g_loss for g in step.grads])

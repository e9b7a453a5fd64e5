"""``torch.optim.Adam``-compatible optimiser backed by the multi-tensor Adam kernel (K11).

The reference builds two ``torch.optim.Adam(self.parameters(), lr)`` with default hyper-parameters
(model.py:404-405) and calls ``step()`` / ``zero_grad()`` (model.py:407-419).  ``FusedAdam`` keeps
those semantics -- parameters without a gradient are skipped, state is created lazily per
parameter, each parameter has its own step count -- but updates every tensor of a step in one
kernel launch instead of ~10 ``_foreach`` launches.
"""

from __future__ import annotations

import torch

from . import ops
from .functions import capture_graph


class DeferredRows:
    """Rolling-window (bounded-deferral) exact Adam for ONE row-sparse parameter of a FusedAdam -- the entity table in
    the KG phase -- behind the reference-facing API (csrc/adam.cu: adam_rolling_*; the epoch engine has its own copy of this
    protocol).  While a run of consecutive TRAIN_KG steps lasts, a step updates the batch's rows and a rotating 1 / window
    slice of the table instead of sweeping all N rows; every row is brought up to date (``flush``) before anything but the
    next TRAIN_KG step can look at the table.  Results are bit-identical to the per-step sweep."""

    def __init__(self, opt: "FusedAdam", param: torch.nn.Parameter, window: int = 16, capacity: int = 16384):
        dev = param.device
        self.opt, self.param, self.window, self.capacity = opt, param, int(window), int(capacity)
        self.row_step = torch.zeros(param.shape[0], dtype=torch.int32, device=dev)
        self.s0 = torch.zeros(1, dtype=torch.int64, device=dev)
        self.step_dev = torch.zeros(1, dtype=torch.int64, device=dev)
        self.hyper = torch.zeros(8, dtype=torch.float32, device=dev)
        self.table = torch.empty(2 * self.capacity, dtype=torch.float32, device=dev)
        self.active = False  # a phase is open: rows may lag behind step_dev
        self.phase_len = 0  # optimiser steps taken in the open phase
        self.host_step = -1  # optimiser step count (host) the device counter corresponds to
        self.hyper_key = None  # (lr, betas, eps) the open phase's bias-correction table was built for

    def state_tensors(self):
        st = self.opt.state[self.param]
        return st["exp_avg"], st["exp_avg_sq"]

    def usable(self) -> bool:
        st = self.opt.state.get(self.param)
        return bool(st) and int(st["step"]) >= 1

    def ensure_phase(self) -> None:
        """Open a phase at the optimiser's current step (no-op while one is open, in sync and has table entries left)."""
        group = self.opt.param_groups[0]
        hyper_key = (group["lr"], group["betas"], group["eps"])
        if self.active and self.phase_len < self.capacity - 2 and hyper_key == self.hyper_key:
            return  # (that the optimiser has not moved under the open phase is checked where it matters: FusedAdam.fast_plan)
        cur = int(self.opt.state[self.param]["step"])
        self.flush()  # (with the scalars the open phase was built for: a changed lr / betas / eps only applies from here on)
        self.hyper_key = hyper_key
        b1, b2 = group["betas"]
        self.step_dev.fill_(cur)
        self.s0.fill_(cur)
        self.row_step.zero_()
        ops.adam_hyper_table(self.s0, self.capacity, group["lr"], b1, b2, self.table)
        ops.adam_set_hyper(max(cur, 1), group["lr"], b1, b2, group["eps"], self.hyper)  # the constants the first replay reads
        self.active, self.phase_len, self.host_step = True, 0, cur

    def stepped(self) -> None:
        self.phase_len += 1
        self.host_step += 1

    def flush(self) -> None:
        """Bring every row up to the optimiser's step count; closes the phase."""
        if self.active and self.phase_len > 0:
            m, v = self.state_tensors()
            ops.adam_lazy_flush(self.param.data, m, v, self.row_step, self.step_dev, self.s0, self.table, self.hyper)
            torch.autograd.graph.increment_version(self.param)
        self.active, self.phase_len = False, 0


class FusedAdam(torch.optim.Optimizer):
    def __init__(self, params, lr: float = 1e-3, betas=(0.9, 0.999), eps: float = 1e-8, use_graphs: bool = True):
        super().__init__(params, dict(lr=lr, betas=betas, eps=eps))
        self.deferred: DeferredRows | None = None  # set by the model for its KG optimiser
        self.state_version = 0  # bumped whenever the state tensors may have been replaced (load_state_dict)
        self._hyper: dict[int, torch.Tensor] = {}
        # When the same (parameter, gradient-buffer) set shows up step after step -- the model's API fast path hands
        # autograd static gradient buffers -- the whole update (bias-correction scalars from a device step counter +
        # the multi-tensor kernel) is captured once as a CUDA graph and replayed.
        self.use_graphs = use_graphs
        self._plans: dict = {}
        self._seen: set = set()
        self._fast: dict = {}

    def _graphed_step(self, group, ps) -> bool:
        if not self.use_graphs or not ps or torch.cuda.is_current_stream_capturing():
            return False
        steps = {self.state[p]["step"] if self.state[p] else 0 for p in ps}
        if len(steps) != 1 or not all(p.is_cuda for p in ps):
            return False
        cur = steps.pop()
        beta1, beta2 = group["betas"]
        key = (tuple((p.data_ptr(), p.grad.data_ptr()) for p in ps), group["lr"], beta1, beta2, group["eps"])
        plan = self._plans.get(key)
        if plan is None:
            if key not in self._seen or cur == 0:  # first sighting: take the generic path (also warms the kernels up)
                if len(self._seen) > 64:
                    self._seen.clear()
                self._seen.add(key)
                return False
            if len(self._plans) > 8:
                self._plans.clear()
            dev = ps[0].device
            plan = {"step_dev": torch.full((1,), cur, dtype=torch.int64, device=dev), "hyper": torch.empty(8, dtype=torch.float32, device=dev),
                    "count": cur, "graph": torch.cuda.CUDAGraph()}
            params, grads = [p.data for p in ps], [p.grad for p in ps]
            ms, vs = [self.state[p]["exp_avg"] for p in ps], [self.state[p]["exp_avg_sq"] for p in ps]
            torch.cuda.synchronize()
            with capture_graph(plan["graph"]):
                ops.adam_advance(plan["step_dev"], group["lr"], beta1, beta2, group["eps"], plan["hyper"])
                ops.adam_apply(params, grads, ms, vs, plan["hyper"])
            self._plans[key] = plan
        if plan["count"] != cur:  # someone else advanced these parameters: resynchronise the device counter
            plan["step_dev"].fill_(cur)
            plan["count"] = cur
        plan["graph"].replay()
        plan["count"] += 1
        for p in ps:
            self.state[p]["step"] += 1
            torch.autograd.graph.increment_version(p)
        return True

    # -- the API fast path (functions.GraphedStep.try_fused_update) ---------------------------------
    def flush_deferred(self) -> None:
        if self.deferred is not None:
            self.deferred.flush()

    def state_dict(self):
        self.flush_deferred()
        return super().state_dict()

    def load_state_dict(self, state_dict):
        self.flush_deferred()
        self._fast.clear()
        self.state_version += 1
        return super().load_state_dict(state_dict)

    def fast_plan(self, ps, grads, grads_key=None, row_slot0=None, rolling=None):
        """Captured ``adam_advance + adam_apply`` over exactly ``(ps, grads)`` (static gradient buffers of a graphed step),
        or None when it cannot be used yet: first sighting (the generic path creates the state and warms the kernels up),
        parameters with different step counts, graphs disabled, or some other parameter of the group holds a gradient."""
        if not self.use_graphs or torch._C._cuda_isCurrentStreamCapturing():
            return None
        group = self.param_groups[0]
        n_with = 0
        for p in group["params"]:
            if p.grad is not None:
                n_with += 1
        if n_with != len(ps) or len(self.param_groups) != 1:  # (the caller has checked that every p in ps holds its gradient)
            return None
        beta1, beta2 = group["betas"]
        if grads_key is None:
            grads_key = tuple(g.data_ptr() for g in grads)
        key = (id(ps[0]), len(ps), grads_key, group["lr"], beta1, beta2, group["eps"], rolling is not None)
        plan = self._fast.get(key)
        if rolling is None and self.deferred is not None and self.deferred.active:
            self.deferred.flush()  # a per-step sweep is about to run: every row must be at the same step first
        if plan is None:
            steps = {int(self.state[p]["step"]) if self.state[p] else 0 for p in ps}
            if len(steps) != 1 or 0 in steps:
                if rolling is not None:
                    raise RuntimeError("kgat_b200: rolling KG update without optimiser state (internal error)")
                return None
            if len(self._fast) > 8:
                self._fast.clear()
            dev = ps[0].device
            cur = steps.pop()
            d = rolling["deferred"] if rolling is not None else None
            plan = {"step_dev": d.step_dev if d is not None else torch.full((1,), cur, dtype=torch.int64, device=dev),
                    "hyper": d.hyper if d is not None else torch.empty(8, dtype=torch.float32, device=dev),
                    "count": cur, "graph": torch.cuda.CUDAGraph(), "states": [self.state[p] for p in ps], "grads": list(grads),
                    "state_ptrs": [self.state[p]["exp_avg"].data_ptr() for p in ps], "deferred": d}
            params = [p.data for p in ps]
            ms, vs = [self.state[p]["exp_avg"] for p in ps], [self.state[p]["exp_avg_sq"] for p in ps]
            torch.cuda.synchronize()
            if d is not None:
                # the step's own advance + (claimed rows, small dense tensors, window slice) in one launch; the captured step_dev /
                # row_step contents are restored below (the capture itself does not run anything)
                h, pt, nt = rolling["ids"]
                with capture_graph(plan["graph"]):
                    ops.adam_advance(d.step_dev, group["lr"], beta1, beta2, group["eps"], d.hyper)
                    ops.adam_rolling_apply(h, pt, nt, rolling["row_slot"], grads[0], params[0], ms[0], vs[0], d.row_step, d.window,
                                           params[1:], list(grads)[1:], ms[1:], vs[1:], d.step_dev, d.s0, d.table, d.hyper)
            else:
                with capture_graph(plan["graph"]):
                    ops.adam_advance(plan["step_dev"], group["lr"], beta1, beta2, group["eps"], plan["hyper"])
                    ops.adam_apply(params, list(grads), ms, vs, plan["hyper"], row_slot0=row_slot0)
            plan["exec"] = plan["graph"].raw_cuda_graph_exec()
            from . import _lib

            plan["launch"] = _lib.load().kgat_graph_launch
            plan["dev_index"] = dev.index if dev.index is not None else torch.cuda.current_device()
            self._fast[key] = plan
        states = plan["states"]
        cur = states[0]["step"]
        for st, ptr in zip(states, plan["state_ptrs"]):
            if st["step"] != cur or st["exp_avg"].data_ptr() != ptr:  # load_state_dict / external steps changed the state under us
                self._fast.clear()
                return None
        if plan["deferred"] is not None:
            if plan["deferred"].host_step != cur or not plan["deferred"].active:
                plan["deferred"].flush()  # the optimiser moved under the open phase: close it, take the generic step
                return None
            plan["count"] = cur
        elif plan["count"] != cur:  # someone else advanced these parameters: resynchronise the device counter
            plan["step_dev"].fill_(cur)
            plan["count"] = cur
        return plan

    def fast_replay(self, plan, ps) -> None:
        rc = plan["launch"](plan["exec"], torch._C._cuda_getCurrentRawStream(plan["dev_index"]))
        if rc != 0:
            from ._lib import check

            check(rc, "adam graph launch")
        plan["count"] += 1
        for st in plan["states"]:
            st["step"] += 1
        d = plan["deferred"]
        if d is not None:
            d.phase_len += 1
            d.host_step += 1
        torch._C._increment_version(ps)  # the kernel wrote through raw pointers: tell autograd the data changed
        for p in ps:
            p.grad = None

    @torch.no_grad()
    def step(self, closure=None):
        loss = closure() if closure is not None else None
        self._step_impl()
        return loss

    def step_and_zero(self) -> None:
        """``step()`` followed by ``zero_grad()`` (set to None) -- what the reference's ``update_*_weights`` do
        (model.py:407-419) -- without torch.optim's per-call hook / profiler wrappers, which cost more host time than
        the 80 us of GPU work of a KG step.  Falls back to the wrapped methods as soon as any hook is registered."""
        from torch.optim import optimizer as _o

        if (getattr(self, "_optimizer_step_pre_hooks", None) or getattr(self, "_optimizer_step_post_hooks", None)
                or getattr(_o, "_global_optimizer_pre_hooks", None) or getattr(_o, "_global_optimizer_post_hooks", None)):
            self.step()
            self.zero_grad()
            return
        with torch.no_grad():
            self._step_impl()
        for group in self.param_groups:
            for p in group["params"]:
                p.grad = None

    def _step_impl(self) -> None:
        self.flush_deferred()  # the generic step sweeps every row: none may lag
        for group in self.param_groups:
            with_grad = [p for p in group["params"] if p.grad is not None]
            if all(not p.grad.is_sparse and p.grad.is_contiguous() for p in with_grad) and self._graphed_step(group, with_grad):
                continue
            by_step: dict[int, list] = {}
            for p in with_grad:
                if p.grad is None:
                    continue
                if p.grad.is_sparse:
                    raise RuntimeError("FusedAdam does not support sparse gradients")
                st = self.state[p]
                if not st:
                    st["step"] = 0
                    st["exp_avg"] = torch.zeros_like(p, memory_format=torch.preserve_format)
                    st["exp_avg_sq"] = torch.zeros_like(p, memory_format=torch.preserve_format)
                st["step"] += 1
                by_step.setdefault(st["step"], []).append(p)
            beta1, beta2 = group["betas"]
            for step, ps in by_step.items():
                dev = ps[0].device
                hyper = self._hyper.get((dev, step % 2))
                if hyper is None:
                    hyper = self._hyper[(dev, step % 2)] = torch.empty(8, dtype=torch.float32, device=dev)
                ops.adam_set_hyper(step, group["lr"], beta1, beta2, group["eps"], hyper)
                ops.adam_apply(
                    [p.data for p in ps],
                    [p.grad.contiguous() for p in ps],
                    [self.state[p]["exp_avg"] for p in ps],
                    [self.state[p]["exp_avg_sq"] for p in ps],
                    hyper,
                )
                for p in ps:  # the kernel wrote through raw pointers: tell autograd the data changed
                    torch.autograd.graph.increment_version(p)

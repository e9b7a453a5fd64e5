"""CUDA-graph training engine: the same kernels as the autograd path, issued as one captured graph
per training step (CF: 3-layer propagation fwd + BPR + hand-written backward + Adam; KG: TransR fwd +
backward + Adam), so an epoch of ~15 k short steps is replayed without per-kernel launch overhead.

The engine works on the *same* parameters and the *same* Adam state as ``model._cf_optimizer`` /
``model._kg_optimizer`` (FusedAdam), so API steps and engine steps can be mixed.  Step-dependent
scalars (Adam bias corrections, dropout stream, which pre-sampled batch to use) live in device
memory and are advanced by tiny kernels inside the graph; nothing is baked in at capture time.

Semantics are those of the reference epoch body (main.py:290-361); see ``trainer.run_epoch`` for the
un-captured equivalent through the public model API (the two are tested to agree).
"""

from __future__ import annotations

import os

import torch

from . import _lib, ops
from .functions import DropoutSpec, capture_graph, last_table_grad, propagate_backward, propagate_forward
from .model import KGAT, KGATMode
from .optim import FusedAdam
from .trainer import CF_BATCH, KG_BATCH, EpochData

f32 = torch.float32


class _AdamSlot:
    """Device-side view of one FusedAdam optimiser for a fixed parameter list."""

    def __init__(self, opt: FusedAdam, params):
        self.opt, self.params = opt, list(params)
        dev = self.params[0].device
        group = opt.param_groups[0]
        self.lr, (self.b1, self.b2), self.eps = group["lr"], group["betas"], group["eps"]
        steps = set()
        for p in self.params:
            st = opt.state[p]
            if not st:
                st["step"] = 0
                st["exp_avg"] = torch.zeros_like(p, memory_format=torch.preserve_format)
                st["exp_avg_sq"] = torch.zeros_like(p, memory_format=torch.preserve_format)
            steps.add(int(st["step"]))
        if len(steps) != 1:
            raise RuntimeError("TrainEngine needs all parameters of a phase to share one Adam step count")
        self._host_step = steps.pop()
        self.step_dev = torch.full((1,), self._host_step, dtype=torch.int64, device=dev)
        self.hyper = torch.empty(8, dtype=f32, device=dev)
        self.exp_avg = [opt.state[p]["exp_avg"] for p in self.params]
        self.exp_avg_sq = [opt.state[p]["exp_avg_sq"] for p in self.params]

    def apply(self, grads, row_slot0=None, advance: bool = True):
        if advance:  # (False: the step counter and scalars were advanced with the batch selection, ops.step_begin)
            ops.adam_advance(self.step_dev, self.lr, self.b1, self.b2, self.eps, self.hyper)
        ops.adam_apply([p.data for p in self.params], grads, self.exp_avg, self.exp_avg_sq, self.hyper, row_slot0=row_slot0)

    def resync(self) -> bool:
        """Pick up what happened to the optimiser between engine epochs (API steps advance the host-side step count; load_state_dict
        replaces the moment tensors).  Returns True when captured graphs that bake the moment pointers in must be dropped."""
        steps = {int(self.opt.state[p]["step"]) for p in self.params}
        if len(steps) != 1:
            raise RuntimeError("TrainEngine needs all parameters of a phase to share one Adam step count")
        step = steps.pop()
        if step != self._host_step:
            self.step_dev.fill_(step)
            self._host_step = step
        moved = any(self.opt.state[p]["exp_avg"].data_ptr() != m.data_ptr() or self.opt.state[p]["exp_avg_sq"].data_ptr() != v.data_ptr()
                    for p, m, v in zip(self.params, self.exp_avg, self.exp_avg_sq))
        group = self.opt.param_groups[0]
        if (group["lr"], tuple(group["betas"]), group["eps"]) != (self.lr, (self.b1, self.b2), self.eps):
            # a scheduler / the user changed the optimiser's scalars: the captured steps bake them in as kernel arguments
            self.lr, (self.b1, self.b2), self.eps = group["lr"], group["betas"], group["eps"]
            moved = True
        if moved:
            self.exp_avg = [self.opt.state[p]["exp_avg"] for p in self.params]
            self.exp_avg_sq = [self.opt.state[p]["exp_avg_sq"] for p in self.params]
        return moved

    def sync_host(self, n_steps: int):
        self._host_step += n_steps
        for p in self.params:
            self.opt.state[p]["step"] += n_steps
            torch.autograd.graph.increment_version(p)

    def snapshot(self):
        return ([p.detach().clone() for p in self.params], [t.clone() for t in self.exp_avg], [t.clone() for t in self.exp_avg_sq], self.step_dev.clone())

    def restore(self, snap):
        ps, ms, vs, step = snap
        for dst, src in zip([p.data for p in self.params] + self.exp_avg + self.exp_avg_sq, ps + ms + vs):
            dst.copy_(src)
        self.step_dev.copy_(step)


class TrainEngine:
    def __init__(self, model: KGAT, cf_batch: int = CF_BATCH, kg_batch: int = KG_BATCH, use_graphs: bool = True, lazy_kg_adam: bool = False,
                 kg_adam: str | None = None, kg_window: int = 16):
        if not hasattr(model, "_cf_optimizer"):
            raise RuntimeError("call model.build_optimizer(...) before creating a TrainEngine")
        self.model = model
        self.dev = model._device()
        self.use_graphs = use_graphs
        self.cf_batch, self.kg_batch = cf_batch, kg_batch
        emb = model._user_entity_embedding.weight
        self.cf_params = [emb] + [t for grp in model._layers() for t in grp]
        self.kg_params = [emb, model._relation_embedding.weight, model._trans_matrix]
        self.cf_adam = _AdamSlot(model._cf_optimizer, self.cf_params)
        self.kg_adam = _AdamSlot(model._kg_optimizer, self.kg_params)
        dev = self.dev
        self.cf_ids = torch.zeros(3, cf_batch, dtype=torch.int64, device=dev)
        self.kg_ids = torch.zeros(4, kg_batch, dtype=torch.int64, device=dev)
        self.cf_loss = torch.zeros(1, dtype=f32, device=dev)
        self.kg_loss = torch.zeros(1, dtype=f32, device=dev)
        self.cf_loss_sum = torch.zeros(1, dtype=f32, device=dev)
        self.kg_loss_sum = torch.zeros(1, dtype=f32, device=dev)
        self.one = torch.ones(1, dtype=f32, device=dev)
        self.cf_scratch = torch.empty(2 * cf_batch, dtype=f32, device=dev)
        self.kg_scratch = torch.empty(ops.transr_scratch_numel(kg_batch, self.kg_params[1].shape[1]), dtype=f32, device=dev)
        self.kg_grads = [torch.zeros_like(p) for p in self.kg_params]
        # KG phase: the embedding-table gradient of a TransR batch lives in <= 3B compact rows (one slot per distinct
        # node, csrc/losses.cu: transr_claim_rows) instead of a zero-filled N x d table that Adam would re-read
        self.kg_row_slot = torch.full((emb.shape[0],), -1, dtype=torch.int32, device=dev)
        self.kg_grad_rows = torch.zeros(3 * kg_batch, emb.shape[1], dtype=f32, device=dev)
        # KG-phase Adam over the embedding table (csrc/adam.cu; all three are bit-identical, tested):
        #   "rolling" (default)  bounded deferral: the batch rows and a rotating 1/kg_window slice of the table are brought up to date
        #                        per step, the zero-gradient updates replayed in registers (KG step 58 -> 36 us at the C3 shape)
        #   "dense"              the per-step 245 MB sweep over table + moments (what torch.optim.Adam does; 0.85-0.95 of HBM peak)
        #   "lazy"               unbounded deferral, a documented negative result (12.5 s vs 4.4 s per epoch when it was measured):
        #                        a row idle for g steps replays g dependent (sqrt, divide) updates inside the step that reads it
        if kg_adam is None:
            kg_adam = "lazy" if lazy_kg_adam else os.environ.get("KGAT_KG_ADAM", "rolling")
        if kg_adam not in ("rolling", "dense", "lazy"):
            raise ValueError(f"kg_adam must be 'rolling', 'dense' or 'lazy', got {kg_adam!r}")
        self.kg_adam_mode = kg_adam
        self.lazy_kg_adam = kg_adam == "lazy"
        self.kg_window = int(os.environ.get("KGAT_KG_WINDOW", kg_window))
        # slice replay on a second stream (a parallel branch of the captured step).  Off: measured 43.0 vs 37.0 us per KG step -- the two
        # cross-stream edges cost more than the overlap with the latency-bound TransR kernel buys
        self.kg_fork = os.environ.get("KGAT_KG_FORK", "0") == "1"
        self._kg_side = torch.cuda.Stream(device=self.dev) if self.kg_fork else None
        if self.kg_window < 1:
            raise ValueError("kg_window must be >= 1")
        self.kg_row_step = torch.zeros(emb.shape[0], dtype=torch.int32, device=dev)
        self.kg_s0 = torch.zeros(1, dtype=torch.int64, device=dev)
        self.kg_table = None
        self._resident: EpochData | None = None
        self.device_sampler = None  # sampler.DeviceSampler: draw every batch on the device inside the captured step
        self._graphs: dict = {}
        self._graph_token = None

    # ------------------------------------------------------------------------------------------
    # the two training steps, written out without autograd
    # ------------------------------------------------------------------------------------------
    def _cf_body(self, select: bool):
        m = self.model
        begun = False
        if select and self.device_sampler is not None:
            self.device_sampler.cf_batch(self.cf_adam.step_dev, self.cf_ids)
        elif select:  # batch selection + the optimiser's step counter / scalars in one launch
            ad = self.cf_adam
            ops.step_begin(self._resident.cf, ad.step_dev, self.cf_ids.view(-1), ad.lr, ad.b1, ad.b2, ad.eps, ad.hyper)
            begun = True
        u, p, n = self.cf_ids[0], self.cf_ids[1], self.cf_ids[2]
        graph = m._graph()
        layers = [tuple(t.detach() for t in grp) for grp in m._layers()]
        drop = m._drop_spec()
        if m.training and drop.keep_bits is None and any(q > 0 for q in drop.ps):
            drop = DropoutSpec(ps=drop.ps, seed=drop.seed, seed_dev=self.cf_adam.step_dev)
        frontier = m._frontier(graph, 3 * self.cf_batch)
        self.frontier = frontier
        if frontier is not None:
            frontier.build([self.cf_ids.view(-1)])
        st = propagate_forward(graph, m._user_entity_embedding.weight.detach(), layers, drop, save=True, frontier=frontier)
        reg = float(m._regularization_params[0])
        ops.bpr_forward(st.tables, u, p, n, reg, self.cf_loss, self.cf_scratch, loss_sum=self.cf_loss_sum)
        n_tab = len(st.tables)

        def inject(l, buf):
            grads = [None] * n_tab
            grads[l] = buf
            ops.bpr_backward(st.tables, grads, u, p, n, reg, self.cf_scratch, self.one)

        g_last = last_table_grad(st, frontier)
        inject(n_tab - 1, g_last)
        g_e0, pgrads = propagate_backward(graph, st, layers, g_last, inject, frontier=frontier)
        self.cf_adam.apply([g_e0] + [t for grp in pgrads for t in grp], advance=not begun)

    def _kg_body(self, select: bool):
        m = self.model
        begun = False  # rolling mode: the optimiser step counter was advanced together with the batch selection
        if select and self.device_sampler is not None:
            self.device_sampler.kg_batch(self.kg_adam.step_dev, self.kg_ids)
        elif select and self.kg_adam_mode == "rolling":
            ad = self.kg_adam
            ops.step_begin(self._resident.kg, ad.step_dev, self.kg_ids.view(-1), ad.lr, ad.b1, ad.b2, ad.eps, ad.hyper)
            begun = True
        elif select:
            ops.select_batch(self._resident.kg, self.kg_adam.step_dev, self.kg_ids.view(-1))
        h, r, pt, nt = self.kg_ids[0], self.kg_ids[1], self.kg_ids[2], self.kg_ids[3]
        emb, rel, w = (p.detach() for p in self.kg_params)
        reg = float(m._regularization_params[1])
        ad = self.kg_adam
        if self.lazy_kg_adam:
            tails = self.kg_ids[2:4].view(-1)  # positive + negative tails, contiguous
            # rows this batch reads must first receive the zero-gradient updates they skipped
            for ids in (h, tails):
                ops.adam_lazy_catchup(emb, ad.exp_avg[0], ad.exp_avg_sq[0], self.kg_row_step, ids, ad.step_dev, self.kg_s0, self.kg_table, ad.hyper)
            ops.transr_forward(emb, rel, w, h, r, pt, nt, reg, self.kg_loss, self.kg_scratch)
            for g in self.kg_grads[1:]:
                ops.fill_(g, 0.0)  # kg_grads[0] (embedding) stays zero outside the touched rows, re-zeroed by sparse_rows
            ops.transr_backward(emb, rel, w, h, r, pt, nt, reg, self.kg_scratch, self.one, *self.kg_grads)
            ops.adam_advance(ad.step_dev, ad.lr, ad.b1, ad.b2, ad.eps, ad.hyper)
            ops.adam_apply([p.data for p in ad.params[1:]], self.kg_grads[1:], ad.exp_avg[1:], ad.exp_avg_sq[1:], ad.hyper)
            for ids in (h, tails):
                ops.adam_sparse_rows(emb, self.kg_grads[0], ad.exp_avg[0], ad.exp_avg_sq[0], self.kg_row_step, ids, ad.step_dev, self.kg_s0, ad.hyper)
        elif self.kg_adam_mode == "rolling":
            # step counter and Adam scalars move first (with the batch selection when the epoch is resident), so nothing after the
            # prepare launch writes a scalar the slice replay reads: it runs on a second stream beside TransR and the row updates
            if not begun:
                ops.adam_advance(ad.step_dev, ad.lr, ad.b1, ad.b2, ad.eps, ad.hyper)
            ops.adam_rolling_prepare(h, pt, nt, self.kg_row_slot, self.kg_grad_rows, self.kg_grads[1], self.kg_grads[2], emb, ad.exp_avg[0],
                                     ad.exp_avg_sq[0], self.kg_row_step, ad.step_dev, self.kg_s0, self.kg_table, ad.hyper, advanced=True)
            dense = ([p.data for p in ad.params[1:]], self.kg_grads[1:], ad.exp_avg[1:], ad.exp_avg_sq[1:])

            def apply(parts):
                ops.adam_rolling_apply(h, pt, nt, self.kg_row_slot, self.kg_grad_rows, emb, ad.exp_avg[0], ad.exp_avg_sq[0], self.kg_row_step,
                                       self.kg_window, *dense, ad.step_dev, self.kg_s0, self.kg_table, ad.hyper, parts=parts)

            fork = self.kg_fork
            if fork:
                main = torch.cuda.current_stream()
                self._kg_side.wait_stream(main)
                with torch.cuda.stream(self._kg_side):
                    apply(2)
            ops.transr_step_claimed(emb, rel, w, h, r, pt, nt, reg, self.kg_loss, self.kg_loss_sum, self.kg_scratch, self.kg_row_slot,
                                    self.kg_grad_rows, self.kg_grads[1], self.kg_grads[2])
            apply(1 if fork else 3)
            if fork:
                main.wait_stream(self._kg_side)
            return
        else:
            ops.transr_step(emb, rel, w, h, r, pt, nt, reg, self.kg_loss, self.kg_loss_sum, self.kg_scratch, self.kg_row_slot,
                            self.kg_grad_rows, self.kg_grads[1], self.kg_grads[2])
            ad.apply([self.kg_grad_rows] + self.kg_grads[1:], row_slot0=self.kg_row_slot)
            return
        self.kg_loss_sum.add_(self.kg_loss)

    def _kg_phase_begin(self, n_kg: int):
        """Lazy / rolling Adam bookkeeping: phase origin = current optimiser step, per-step bias-correction table."""
        if self.kg_adam_mode == "dense" or n_kg == 0:
            return
        ad = self.kg_adam
        self.kg_s0.copy_(ad.step_dev)
        self.kg_row_step.zero_()
        if self.lazy_kg_adam:
            self.kg_grads[0].zero_()
        need = 2 * (n_kg + 2)  # +2: the capture warm-up may run one extra (undone) step
        if self.kg_table is None or self.kg_table.numel() < need:
            self.kg_table = torch.empty(max(need, 2 * 16384), dtype=f32, device=self.dev)
            self._graphs.pop(("kg", True), None)
            self._graphs.pop(("kg", False), None)
        ops.adam_hyper_table(self.kg_s0, self.kg_table.numel() // 2, ad.lr, ad.b1, ad.b2, self.kg_table)
        ops.adam_set_hyper(1, ad.lr, ad.b1, ad.b2, ad.eps, ad.hyper)  # constants (1-b1, b2, 1-b2, eps) for the first catch-up

    def _kg_phase_end(self, n_kg: int):
        if self.kg_adam_mode == "dense" or n_kg == 0:
            return
        ad = self.kg_adam
        emb = self.kg_params[0].detach()
        ops.adam_lazy_flush(emb, ad.exp_avg[0], ad.exp_avg_sq[0], self.kg_row_step, ad.step_dev, self.kg_s0, self.kg_table, ad.hyper)

    # ------------------------------------------------------------------------------------------
    # capture / replay
    # ------------------------------------------------------------------------------------------
    def _token(self):
        g = self.model._graph()
        return (id(g), g.vals.data_ptr(), g.t_vals.data_ptr(), self.model.training, id(self._resident), id(self.device_sampler),
                self.model.cf_pruning)

    def _get(self, kind: str, select: bool):
        """Returns a callable running one step (a captured graph replay when graphs are enabled)."""
        body = self._cf_body if kind == "cf" else self._kg_body
        if not self.use_graphs:
            return lambda: body(select)
        token = self._token()
        if token != self._graph_token:
            self._graphs.clear()
            self._graph_token = token
        key = (kind, select)
        if key not in self._graphs:
            adam = self.cf_adam if kind == "cf" else self.kg_adam
            snap = adam.snapshot()
            sums = (self.cf_loss_sum.clone(), self.kg_loss_sum.clone())
            row_step = self.kg_row_step.clone()
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                body(select)  # eager warm-up (lazy kernel attributes, allocator pools); undone below
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            adam.restore(snap)
            self.cf_loss_sum.copy_(sums[0])
            self.kg_loss_sum.copy_(sums[1])
            self.kg_row_step.copy_(row_step)
            if kind == "kg":
                self.kg_grads[0].zero_()
            g = torch.cuda.CUDAGraph()
            before = _lib.LaunchCounter.count
            with capture_graph(g):
                body(select)
            kernels = _lib.LaunchCounter.count - before  # our kernels recorded in this graph
            _lib.LaunchCounter.count = before

            def replay(g=g, kernels=kernels):
                _lib.LaunchCounter.count += kernels
                g.replay()

            self._graphs[key] = replay
        return self._graphs[key]

    # ------------------------------------------------------------------------------------------
    # public
    # ------------------------------------------------------------------------------------------
    def bind_resident(self, data: EpochData):
        """Keep an epoch of pre-sampled batches in HBM: cf [n_cf, 3, B], kg [n_kg, 4, B] int64."""
        cf = torch.stack([t.to(self.dev) for t in data.cf], dim=1).contiguous()
        kg = torch.stack([t.to(self.dev) for t in data.kg], dim=1).contiguous()
        holder = EpochData(cf=cf, kg=kg, edges=tuple(t.to(self.dev) for t in data.edges))
        self._resident = holder
        return holder

    def run_epoch(self, data: EpochData | None = None, read_loss_every_step: bool = False, n_cf: int | None = None, n_kg: int | None = None,
                  refresh: bool = True):
        """One reference epoch body.  ``data=None`` uses the batches bound with ``bind_resident``
        (selected on the device by the optimiser step counter: step s uses batch s mod n); a host
        ``EpochData`` (pinned tensors) is copied host->device step by step instead.
        Returns (mean CF loss, mean KG loss, bytes host->device, bytes device->host)."""
        m = self.model
        m.train()
        resident = data is None
        src = self._resident if resident else data
        if src is None:
            raise RuntimeError("no resident epoch bound and no data given")
        n_cf = int(src.cf.shape[0] if resident else src.n_cf) if n_cf is None else n_cf
        n_kg = int(src.kg.shape[0] if resident else src.n_kg) if n_kg is None else n_kg
        h2d = d2h = 0
        if self.cf_adam.resync() | self.kg_adam.resync():  # steps taken / state replaced through the model API since the last epoch
            self._graphs.clear()
        self.cf_loss_sum.zero_()
        self.kg_loss_sum.zero_()
        cf_host = kg_host = 0.0
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        step = self._get("cf", resident) if n_cf else None
        ev[0].record()
        for i in range(n_cf):
            if not resident:
                for j in range(3):
                    self.cf_ids[j].copy_(data.cf[j][i], non_blocking=True)
                h2d += 3 * self.cf_batch * 8
            step()
            if read_loss_every_step:
                cf_host += float(self.cf_loss.item())
                d2h += 4
        self.cf_adam.sync_host(n_cf)
        ev[1].record()
        self._kg_phase_begin(n_kg)
        step = self._get("kg", resident) if n_kg else None
        for i in range(n_kg):
            if not resident:
                for j in range(4):
                    self.kg_ids[j].copy_(data.kg[j][i], non_blocking=True)
                h2d += 4 * self.kg_batch * 8
            step()
            if read_loss_every_step:
                kg_host += float(self.kg_loss.item())
                d2h += 4
        self._kg_phase_end(n_kg)
        self.kg_adam.sync_host(n_kg)
        ev[2].record()
        if refresh:
            eh, er, et, ri = src.edges
            if not eh.is_cuda:
                h2d += eh.numel() * eh.element_size() + er.numel() * 8 + et.numel() * et.element_size() + ri.numel() * 8
            m(eh, er, et, ri, mode=KGATMode.UPDATE_ATTENTION)
        ev[3].record()
        if not read_loss_every_step:
            cf_host, kg_host = float(self.cf_loss_sum.item()), float(self.kg_loss_sum.item())
            d2h += 8
        ev[3].synchronize()
        self.last_phase_ms = {"cf": ev[0].elapsed_time(ev[1]), "kg": ev[1].elapsed_time(ev[2]), "refresh": ev[2].elapsed_time(ev[3]),
                              "n_cf": n_cf, "n_kg": n_kg}
        return cf_host / max(n_cf, 1), kg_host / max(n_kg, 1), h2d, d2h

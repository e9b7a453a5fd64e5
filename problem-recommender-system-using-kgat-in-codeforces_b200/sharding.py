"""Row-sharded multi-GPU propagation (SURVEY.md section 8e): one process per GPU, the CKG rows are
partitioned across the ranks and every propagation layer exchanges the freshly computed rows with an
NCCL all-gather over NVLink; the backward pass all-gathers the side-gradient and gathers over the
local rows of A^T (no atomics, no reduce-scatter); dense-parameter gradients are all-reduced.

Partition: *cyclic* -- rank r owns the rows {i : i mod P == r}.  The survey suggested contiguous
nnz-balanced ranges; on a CKG the node types sit in contiguous id blocks (users, items, entities)
with a 10-15x spread in row length, so contiguous ranges are either nnz- or row-balanced, never
both, and the bi-interaction GEMMs cost per *row*.  The cyclic split balances both statistically,
gives equal shard sizes (all-gather without padding waste) and needs only ``i % P, i // P``.

Tables live in the *padded cyclic layout*: global row i sits at ``(i % P) * max_rows + i // P`` so a
rank's rows are one contiguous slice, which is exactly what ``all_gather_into_tensor`` wants.

The orchestration is written against a small ``LocalOps`` interface so the same code runs with the
CUDA kernels (``KernelOps``) on GPUs and -- in the CPU tests, world_size 2 over gloo -- with plain
torch ops injected by the test.

Phases of the reference epoch (main.py:290-361):
  CF steps   row-sharded as above (this is where the propagation cost is),
  KG steps   replicated (a TransR batch touches <= 1536 rows; sharding it would add a 40 MB
             all-gather per step for a 50 us kernel),
  refresh    replicated and deterministic (10 ms once per epoch).
"""

from __future__ import annotations

from dataclasses import dataclass

import numpy as np
import torch
import torch.distributed as dist


# ----------------------------------------------------------------------------------------------
# partition (pure index math, CPU-tested)
# ----------------------------------------------------------------------------------------------
@dataclass(frozen=True)
class CyclicPartition:
    n: int
    world: int
    rank: int

    @property
    def max_rows(self) -> int:
        return (self.n + self.world - 1) // self.world

    @property
    def padded(self) -> int:
        return self.max_rows * self.world

    def count(self, rank: int | None = None) -> int:
        r = self.rank if rank is None else rank
        return len(range(r, self.n, self.world))

    def local_rows(self, rank: int | None = None) -> np.ndarray:
        r = self.rank if rank is None else rank
        return np.arange(r, self.n, self.world, dtype=np.int64)

    def to_padded(self, ids):
        """global row id -> row in the padded cyclic layout (numpy array or torch tensor)."""
        return (ids % self.world) * self.max_rows + ids // self.world

    def slice(self, rank: int | None = None) -> slice:
        r = self.rank if rank is None else rank
        return slice(r * self.max_rows, r * self.max_rows + self.count(r))

    def full_slice(self, rank: int | None = None) -> slice:
        r = self.rank if rank is None else rank
        return slice(r * self.max_rows, (r + 1) * self.max_rows)

    def scatter_rows(self, table: torch.Tensor) -> torch.Tensor:
        """[n, d] in global order -> [padded, d] in the padded cyclic layout (pad rows zero)."""
        out = table.new_zeros((self.padded, table.shape[1]))
        idx = torch.arange(self.n, device=table.device)
        out[self.to_padded(idx)] = table
        return out

    def gather_rows(self, padded_table: torch.Tensor) -> torch.Tensor:
        idx = torch.arange(self.n, device=padded_table.device)
        return padded_table[self.to_padded(idx)]


def shard_csr(row_ptr: np.ndarray, col_idx: np.ndarray, part: CyclicPartition, local_range: tuple[int, int] | None = None):
    """Local CSR of the rows owned by ``part.rank`` (or of the sub-range ``local_range`` of them): (row_ptr_local,
    col_idx in padded layout, slot_ids = positions of the local non-zeros in the global value array)."""
    rows = part.local_rows()
    if local_range is not None:
        rows = rows[local_range[0] : local_range[1]]
    lens = (row_ptr[rows + 1] - row_ptr[rows]).astype(np.int64)
    lp = np.concatenate([[0], np.cumsum(lens)])
    starts = np.repeat(row_ptr[rows].astype(np.int64), lens)
    within = np.arange(int(lp[-1]), dtype=np.int64) - np.repeat(lp[:-1], lens)
    slot_ids = starts + within
    cols = part.to_padded(col_idx[slot_ids].astype(np.int64))
    return lp.astype(np.int32), cols.astype(np.int32), slot_ids.astype(np.int32)


# ----------------------------------------------------------------------------------------------
# local compute interface
# ----------------------------------------------------------------------------------------------
class KernelOps:
    """LocalOps backed by the sm_100a kernels."""

    def __init__(self):
        from . import ops
        from .graph import make_plan

        self.ops, self.make_plan = ops, make_plan
        self._partials = None

    def make_local_graph(self, row_ptr, col_idx, slot_ids, device, chunk=256):
        rp = torch.from_numpy(row_ptr).to(device)
        return {"row_ptr": rp, "col_idx": torch.from_numpy(col_idx).to(device), "slot_ids": torch.from_numpy(slot_ids).to(device),
                "plan": self.make_plan(rp, chunk), "vals": torch.empty(col_idx.shape[0], dtype=torch.float32, device=device)}

    def refresh_values(self, lg, global_vals):
        self.ops.gather_f32(global_vals, lg["slot_ids"], out=lg["vals"])

    def spmm(self, lg, x_full, out, addend=None):
        plan = lg["plan"]
        need = plan.n_partials * x_full.shape[1]
        if need and (self._partials is None or self._partials.numel() < need):
            self._partials = torch.empty(need, dtype=torch.float32, device=x_full.device)
        return self.ops.spmm(plan, lg["col_idx"], lg["vals"], x_full, out, addend, self._partials)

    def biagg_forward(self, e, s, layer, out, p, seed, offset, seed_dev=None, peer_out=None):
        n, d_out = e.shape[0], layer[0].shape[0]
        inv = torch.empty(n, dtype=torch.float32, device=e.device)
        flags = torch.empty(n, d_out, dtype=torch.uint8, device=e.device)
        self.ops.biagg_forward(e, s, *layer, out, inv, flags, dropout_p=p, seed=seed, offset=offset, seed_dev=seed_dev, peer_out=peer_out)
        return inv, flags

    def biagg_backward(self, g_out, out, inv, flags, e, s, layer, p, g_s, g_e, peer_out=None, accumulate_into=None):
        w1, b1, w2, b2 = layer
        n, d_in, d_out = e.shape[0], e.shape[1], w1.shape[0]
        n_ctas = self.ops.biagg_backward_ctas(n, d_in, d_out)
        partials = torch.empty(n_ctas * (2 * d_in * d_out + 2 * d_out), dtype=torch.float32, device=e.device)
        self.ops.biagg_backward(g_out, out, inv, flags, e, s, w1, w2, p, g_s, g_e, partials, n_ctas, peer_out=peer_out)
        grads = accumulate_into if accumulate_into is not None else [torch.empty_like(t) for t in (w1, b1, w2, b2)]
        self.ops.biagg_reduce_param_grads(partials, n_ctas, d_in, d_out, *grads, accumulate=accumulate_into is not None)
        return grads

    def bpr_forward(self, tables, u, p, n, reg, loss, scratch):
        self.ops.bpr_forward(tables, u, p, n, reg, loss, scratch)

    def bpr_backward(self, tables, grads, u, p, n, reg, scratch, g_loss):
        self.ops.bpr_backward(tables, grads, u, p, n, reg, scratch, g_loss)


def all_gather_rows(full: torch.Tensor, part: CyclicPartition):
    """In-place all-gather of a [padded, d] table whose own slice has just been written."""
    if part.world == 1:
        return
    mine = full[part.full_slice()]
    dist.all_gather_into_tensor(full, mine)


class CollectiveExchange:
    """Row exchange through ``torch.distributed`` collectives (NCCL all-gather on GPUs, gloo in the CPU tests).
    Channels: ("t", l) = layer table l, ("g", l) = side gradient of layer l."""

    fused = False

    def __init__(self, part: CyclicPartition, dims, device):
        pad = part.padded
        self.part = part
        self.tables = [torch.zeros(pad, d, dtype=torch.float32, device=device) for d in dims]
        self.gs_full = [torch.zeros(pad, d, dtype=torch.float32, device=device) for d in dims[:-1]]

    def _buf(self, kind, l):
        return self.tables[l] if kind == "t" else self.gs_full[l]

    can_push = False

    def peer_out(self, kind, l, row0=0):
        return None

    def gather(self, kind, l, pushed=False):
        all_gather_rows(self._buf(kind, l), self.part)

    def all_reduce_flat(self, flat):
        dist.all_reduce(flat)
        return flat

    def barrier(self):
        pass

    def check(self):
        pass

    def close(self):
        pass


class PeerExchange:
    """Row exchange over NVLink peer memory (peer.py / csrc/peer.cu): the tables live in an IPC arena mapped by
    every rank; producers store their rows into every peer's table (from the bi-interaction kernels' own epilogue
    when ``fused``, else with one push kernel) and a flag handshake replaces the collective.  The parameter-gradient
    all-reduce is the same pattern: every rank deposits its partial in slot ``rank`` of every peer and all ranks
    add the slots in rank order (bit-identical results on every rank)."""

    def __init__(self, part: CyclicPartition, dims, device, n_flat: int, fused=()):
        """``fused``: which producers store into the peers' tables from their own epilogue -- "t" the bi-interaction
        forward (layer tables), "g" its backward (side gradients), "e" Adam (embedding rows) -- instead of a push
        kernel after them.  Measured at the C3 shape, the fused stores only pay where they leave the SM as wide,
        coalesced bursts from a kernel that is not memory-bound: the mma.sync forward (tile staged in shared memory,
        512-byte warp stores) hid half of them at 2 GPUs (126 us fused vs 103 + 47 us kernel + push); the backward's
        8-byte fragment stores, the HBM-bound Adam sweep (4 GPUs: 319 vs 127 + 100 us, 69 vs 20 + 40 us) and the
        thread-per-row 16-byte stores of the tcgen05 forward epilogue (8 GPUs: 502 vs 60 us + push) do not.  Default:
        nothing fused, every table goes out with the push kernel at NVLink rate."""
        from .peer import PeerArena

        self.part, self.fused_kinds = part, tuple(fused)
        self.fused = "e" in self.fused_kinds
        pad = part.padded
        spec = {f"t{l}": (pad, d) for l, d in enumerate(dims)}
        spec.update({f"g{l}": (pad, d) for l, d in enumerate(dims[:-1])})
        self.n_flat = (n_flat + 3) // 4 * 4
        spec["flat"] = (part.world, self.n_flat)
        self._chan = {name: i for i, name in enumerate(spec)}
        self._chan["barrier"] = len(spec)
        self.arena = PeerArena(part.rank, part.world, device, spec, n_channels=len(spec) + 1)
        self.tables = [self.arena.table(f"t{l}") for l in range(len(dims))]
        self.gs_full = [self.arena.table(f"g{l}") for l in range(len(dims) - 1)]
        self._row0 = part.rank * part.max_rows

    can_push = True

    def peer_out(self, kind, l, row0=0):
        """Device pointer array: row ``row0`` of this rank's slice of the table in every peer's arena (for fused
        epilogue stores); None when this producer is not fused."""
        k = "e" if (kind, l) == ("t", 0) else kind
        return self.arena.peer_ptrs(f"{kind}{l}", self._row0 + row0) if k in self.fused_kinds and self.part.world > 1 else None

    def push_rows(self, kind, l, row0, n_rows, max_ctas=0):
        """Rows [row0, row0 + n_rows) of this rank's slice -> every peer's table, on the current stream: push kernel, or
        (max_ctas < 0) the copy engines."""
        if max_ctas < 0:
            self.arena.copy(f"{kind}{l}", self._row0 + row0, n_rows)
        else:
            self.arena.push(f"{kind}{l}", self._row0 + row0, n_rows, max_ctas)

    def gather(self, kind, l, pushed=False):
        name = f"{kind}{l}"
        if not pushed:
            self.arena.push(name, self._row0, self.part.max_rows)
        self.arena.signal_wait(self._chan[name])

    def all_reduce_flat(self, flat):
        slots = self.arena.table("flat")
        slots[self.part.rank, : flat.numel()].copy_(flat)
        self.arena.push("flat", self.part.rank, 1)
        self.arena.signal_wait(self._chan["flat"])
        torch.sum(slots[:, : flat.numel()], dim=0, out=flat)
        return flat

    def barrier(self):
        self.arena.signal_wait(self._chan["barrier"])

    def check(self):
        self.arena.check()

    def close(self):
        self.arena.close()


# ----------------------------------------------------------------------------------------------
# sharded CF step
# ----------------------------------------------------------------------------------------------
class ShardedPropagation:
    """Forward / backward of the 3-layer propagation + BPR loss on row shards.

    ``layers``: list of (W1, b1, W2, b2) replicated on every rank.  ``e0_full``: [padded, d0] table
    in padded layout whose own slice holds the current local embedding rows."""

    def __init__(self, part: CyclicPartition, local_a, local_at, ops: "KernelOps", dims, device, exchange=None, chunk_bounds=None):
        """``local_a``: the local rows of A as one graph, or a list of graphs over consecutive sub-ranges
        ``chunk_bounds`` = [(start, stop), ...] of the local rows.  With several chunks (and a peer exchange) the rows a
        chunk has produced travel to the peers on a side stream while the next chunk is being computed."""
        self.part, self.at, self.ops = part, local_at, ops
        self.a = list(local_a) if isinstance(local_a, (list, tuple)) else [local_a]
        self.bounds = list(chunk_bounds) if chunk_bounds is not None else [(0, part.count())]
        assert len(self.a) == len(self.bounds)
        self.dims = list(dims)  # [d0, d1, ..., dL]
        pad = part.padded
        self.ex = exchange if exchange is not None else CollectiveExchange(part, self.dims, device)
        self.tables = self.ex.tables
        self.gs_full = self.ex.gs_full
        self.g_tables = [torch.zeros(pad, d, dtype=torch.float32, device=device) for d in self.dims]
        self.device = device
        self.saved = None
        self.side = None
        if self.ex.can_push and len(self.bounds) > 1:
            self.side = torch.cuda.Stream(device=device, priority=-1)
        self._side_busy = False
        import os

        # side-stream transfers: -1 = copy engines (no SM taken from the compute kernels), > 0 = push kernel with that many CTAs
        self.push_ctas = int(os.environ.get("KGAT_PUSH_CTAS", "-1"))

    # rows [r0, r1) of this rank's slice of table (kind, l) have just been produced on the current stream
    def _send(self, kind, l, r0, r1, fused):
        if fused or not self.ex.can_push:
            return
        if self.side is None:
            self.ex.push_rows(kind, l, r0, r1 - r0)
            return
        ev = torch.cuda.Event()
        ev.record()
        self.side.wait_event(ev)
        with torch.cuda.stream(self.side):
            self.ex.push_rows(kind, l, r0, r1 - r0, self.push_ctas)
        self._side_busy = True

    def _complete(self, kind, l):
        if self._side_busy:
            torch.cuda.current_stream().wait_stream(self.side)
            self._side_busy = False
        self.ex.gather(kind, l, pushed=self.ex.can_push)

    def forward(self, layers, ps, seed, u, p, n, reg, loss, scratch, seed_dev=None):
        part = self.part
        sl = part.slice()
        # the embedding rows: mirrored into the peers' tables by the Adam kernel of the previous step when that is
        # fused (the tables start out complete: scatter_from_model), so only the handshake is left
        self.ex.gather("t", 0, pushed=self.ex.fused)
        saved = []
        for l, layer in enumerate(layers):
            x_full = self.tables[l]
            x_loc = x_full[sl]
            s_loc = torch.empty(part.count(), self.dims[l], dtype=torch.float32, device=self.device)
            out_loc = self.tables[l + 1][sl]
            invs, flagss = [], []
            for a_c, (r0, r1) in zip(self.a, self.bounds):
                self.ops.spmm(a_c, x_full, s_loc[r0:r1])
                # each rank draws its rows' dropout decisions from its own Philox stream (seed + rank); the counter
                # advances by at most 32 per row, so chunk c starts at 32 * r0
                peer_out = self.ex.peer_out("t", l + 1, r0)
                inv, flags = self.ops.biagg_forward(x_loc[r0:r1], s_loc[r0:r1], layer, out_loc[r0:r1], ps[l], seed + 7919 * part.rank,
                                                    ((l + 1) << 40) + 32 * r0, seed_dev, **({"peer_out": peer_out} if peer_out is not None else {}))
                self._send("t", l + 1, r0, r1, peer_out is not None)
                invs.append(inv)
                flagss.append(flags)
            self._complete("t", l + 1)
            saved.append((s_loc, invs, flagss))
        self.ops.bpr_forward(self.tables, u, p, n, reg, loss, scratch)
        self.saved = (saved, (u, p, n), reg, scratch, ps)
        return loss

    def backward(self, layers, g_loss):
        """Returns (g_e0_local [count, d0], [param grads per layer] summed over ranks)."""
        part = self.part
        sl = part.slice()
        saved, (u, p, n), reg, scratch, ps = self.saved
        L = len(layers)
        n_tab = L + 1

        def inject(l):
            grads = [None] * n_tab
            grads[l] = self.g_tables[l]
            self.ops.bpr_backward(self.tables, grads, u, p, n, reg, scratch, g_loss)

        self.g_tables[L].zero_()
        inject(L)
        pgrads = [None] * L
        for l in range(L, 0, -1):
            s_loc, invs, flagss = saved[l - 1]
            x_loc = self.tables[l - 1][sl]
            g_s_loc = self.gs_full[l - 1][sl]
            g_e_loc = torch.empty(part.count(), self.dims[l - 1], dtype=torch.float32, device=self.device)
            g_out_loc, out_loc = self.g_tables[l][sl], self.tables[l][sl]
            for c, (r0, r1) in enumerate(self.bounds):
                peer_out = self.ex.peer_out("g", l - 1, r0)
                kw = {"peer_out": peer_out} if peer_out is not None else {}
                if c > 0:
                    kw["accumulate_into"] = pgrads[l - 1]
                pgrads[l - 1] = self.ops.biagg_backward(g_out_loc[r0:r1], out_loc[r0:r1], invs[c], flagss[c], x_loc[r0:r1], s_loc[r0:r1],
                                                        layers[l - 1], ps[l - 1], g_s_loc[r0:r1], g_e_loc[r0:r1], **kw)
                self._send("g", l - 1, r0, r1, peer_out is not None)
            self._complete("g", l - 1)
            self.ops.spmm(self.at, self.gs_full[l - 1], self.g_tables[l - 1][sl], addend=g_e_loc)
            inject(l - 1)
        if part.world > 1:
            flat = self.ex.all_reduce_flat(torch.cat([t.reshape(-1) for grp in pgrads for t in grp]))
            off = 0
            for grp in pgrads:
                for t in grp:
                    t.copy_(flat[off : off + t.numel()].view_as(t))
                    off += t.numel()
        return self.g_tables[0][sl], pgrads


# ----------------------------------------------------------------------------------------------
# engine + bench entry for N > 1
# ----------------------------------------------------------------------------------------------
class ShardedEngine:
    """Epoch driver for P ranks: sharded CF phase, replicated KG phase and refresh."""

    def __init__(self, model, part: CyclicPartition, use_graphs: bool = True, exchange: str | None = None):
        """``exchange``: "peer" (default; NVLink peer memory: every produced table is pushed into the peers' copies by a
        store kernel, flag handshake instead of a collective), "peer-fwd" / "peer-all" (the bi-interaction forward /
        every producer stores into the peers' tables from its own epilogue) or "nccl" (all-gather / all-reduce
        collectives, the baseline the peer path is measured against).  Environment override: KGAT_EXCHANGE."""
        import os

        from . import ops
        from .engine import TrainEngine

        self.model, self.part, self.kops, self.ops = model, part, KernelOps(), ops
        self.use_graphs = use_graphs
        self.exchange_kind = exchange or os.environ.get("KGAT_EXCHANGE", "peer")
        if self.exchange_kind == "peer-push":
            self.exchange_kind = "peer"
        if self.exchange_kind not in ("peer", "peer-fwd", "peer-all", "nccl"):
            raise ValueError(f"unknown exchange {self.exchange_kind!r}")
        self.exchange = None
        self._cf_kernels = 0
        # Row chunks per layer: chunk c's rows travel to the peers (side stream, copy engines) while chunk c + 1 is
        # computed.  Off by default: at the C3 shape the per-rank kernels are already 10-60 us, and splitting them costs
        # more (ramp-up, per-CTA weight staging) than the hidden transfer saves -- 4 GPUs: 795 us per CF step
        # unchunked, 1,095 us with 2 chunks, 1,215 us with 4 (tools/prof_sharded.py).  For tables that do not fit one
        # GPU (C5) the kernels are 100x longer and the trade flips.
        self.n_chunks = max(1, int(os.environ.get("KGAT_SHARD_CHUNKS", "1")))
        self._cf_graph = None
        self._cf_graph_key = None
        self._cf_padded = None
        self._cf_src = None
        self.cf_ids = None
        self.dev = model._device()
        self.single = TrainEngine(model, use_graphs=True)  # KG phase (replicated) reuses the 1-GPU engine
        self.layers = [tuple(t.detach() for t in grp) for grp in model._layers()]
        dims = [model._cf_embedding_dim, *model._layer_dims]
        if part.world > 1 and self.exchange_kind != "nccl":
            n_flat = sum(t.numel() for grp in self.layers for t in grp)
            fused = {"peer": (), "peer-fwd": ("t",), "peer-all": ("t", "g", "e")}[self.exchange_kind]
            self.exchange = PeerExchange(part, dims, self.dev, n_flat, fused=fused)
        self._build_graph(dims)
        n_loc = part.count()
        d0 = dims[0]
        self.e0_m = torch.zeros(n_loc, d0, device=self.dev)
        self.e0_v = torch.zeros(n_loc, d0, device=self.dev)
        self.layer_m = [[torch.zeros_like(t) for t in grp] for grp in self.layers]
        self.layer_v = [[torch.zeros_like(t) for t in grp] for grp in self.layers]
        self.step_dev = torch.zeros(1, dtype=torch.int64, device=self.dev)
        self.hyper = torch.empty(8, device=self.dev)
        self.loss = torch.zeros(1, device=self.dev)
        self.loss_sum = torch.zeros(1, device=self.dev)
        self.scratch = torch.empty(2 * 256, device=self.dev)
        self.one = torch.ones(1, device=self.dev)
        self.scatter_from_model()

    def _build_graph(self, dims):
        g = self.model._graph()
        self._graph_id = (id(g), g.vals.data_ptr())
        rp, ci = g.row_ptr.cpu().numpy(), g.col_idx.cpu().numpy()
        tp, ti = g.t_ptr.cpu().numpy(), g.t_idx.cpu().numpy()
        n_loc = self.part.count()
        n_chunks = self.n_chunks if self.exchange is not None else 1
        cuts = [n_loc * c // n_chunks for c in range(n_chunks + 1)]
        self.bounds = [(cuts[c], cuts[c + 1]) for c in range(n_chunks) if cuts[c + 1] > cuts[c]]
        self.a = [self.kops.make_local_graph(*shard_csr(rp, ci, self.part, b), self.dev) for b in self.bounds]
        self.at = self.kops.make_local_graph(*shard_csr(tp, ti, self.part), self.dev)
        self.prop = ShardedPropagation(self.part, self.a, self.at, self.kops, dims, self.dev, exchange=self.exchange,
                                       chunk_bounds=self.bounds)
        self.refresh_values()

    def refresh_values(self):
        g = self.model._graph()
        for a_c in self.a:
            self.kops.refresh_values(a_c, g.vals)
        self.kops.refresh_values(self.at, g.t_vals)

    def scatter_from_model(self):
        w = self.model._user_entity_embedding.weight.detach()
        self.prop.tables[0].copy_(self.part.scatter_rows(w))
        self.prop.ex.barrier()  # nobody stores rows into a table its owner is still overwriting

    def gather_to_model(self):
        self.prop.ex.gather("t", 0)
        self.model._user_entity_embedding.weight.data.copy_(self.part.gather_rows(self.prop.tables[0]))
        torch.autograd.graph.increment_version(self.model._user_entity_embedding.weight)

    def cf_step(self, u, p, n):
        """One sharded CF step; ``u, p, n`` are already rows of the padded cyclic layout."""
        m, part = self.model, self.part
        ps = [float(a.message_dropout.p) if m.training else 0.0 for a in m._aggregator_layers]
        reg = float(m._regularization_params[0])
        self.prop.forward(self.layers, ps, 12345, u, p, n, reg, self.loss, self.scratch, seed_dev=self.step_dev)
        g_e0, pgrads = self.prop.backward(self.layers, self.one)
        opt = m._cf_optimizer.param_groups[0]
        self.ops.adam_advance(self.step_dev, opt["lr"], opt["betas"][0], opt["betas"][1], opt["eps"], self.hyper)
        e0_loc = self.prop.tables[0][part.slice()]
        params = [e0_loc] + [t for grp in self.layers for t in grp]
        grads = [g_e0.contiguous()] + [t for grp in pgrads for t in grp]
        ms = [self.e0_m] + [t for grp in self.layer_m for t in grp]
        vs = [self.e0_v] + [t for grp in self.layer_v for t in grp]
        peer_e0 = self.prop.ex.peer_out("t", 0)
        self.ops.adam_apply(params, grads, ms, vs, self.hyper, **({"peer_param0": peer_e0} if peer_e0 is not None else {}))
        self.loss_sum.add_(self.loss)

    def _cf_graphed_step(self):
        """select the current batch (device step counter) + one sharded CF step; captured as ONE CUDA graph
        including the NCCL all-gathers / all-reduce (all ranks capture the same sequence)."""
        self.ops.select_batch(self._cf_padded, self.step_dev, self.cf_ids.view(-1))
        self.cf_step(self.cf_ids[0], self.cf_ids[1], self.cf_ids[2])

    def _cf_runner(self):
        if not self.use_graphs:
            return self._cf_graphed_step
        key = (self._graph_id, id(self._cf_padded), self.model.training)
        if self._cf_graph is None or key != self._cf_graph_key:
            # warm-up step (communicators, lazy kernel attributes), undone afterwards
            e0_loc = self.prop.tables[0][self.part.slice()]
            snap = [t.clone() for t in [e0_loc, self.e0_m, self.e0_v, self.step_dev, self.loss_sum] + [t for grp in self.layers for t in grp]
                    + [t for grp in self.layer_m for t in grp] + [t for grp in self.layer_v for t in grp]]
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                self._cf_graphed_step()
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            live = [e0_loc, self.e0_m, self.e0_v, self.step_dev, self.loss_sum] + [t for grp in self.layers for t in grp] \
                + [t for grp in self.layer_m for t in grp] + [t for grp in self.layer_v for t in grp]
            for dst, src in zip(live, snap):
                dst.copy_(src)
            self.prop.ex.gather("t", 0)  # the peers' mirrors of my embedding rows go back to the restored values too
            if self.part.world > 1:
                dist.barrier()
            from . import _lib
            from .functions import capture_graph

            g = torch.cuda.CUDAGraph()
            before = _lib.LaunchCounter.count
            with capture_graph(g):
                self._cf_graphed_step()
            self._cf_kernels = _lib.LaunchCounter.count - before
            _lib.LaunchCounter.count = before
            self._cf_graph, self._cf_graph_key = g, key

        def replay(g=self._cf_graph, kernels=self._cf_kernels):
            from . import _lib

            _lib.LaunchCounter.count += kernels
            g.replay()

        return replay

    def run_epoch(self, data, n_cf=None, n_kg=None, refresh=True):
        """``data``: EpochData on the device (cf [n,3,B], kg [n,4,B] stacked, as TrainEngine.bind_resident)."""
        m = self.model
        m.train()
        g = m._graph()
        if (id(g), g.vals.data_ptr()) != self._graph_id:
            self._build_graph([m._cf_embedding_dim, *m._layer_dims])
            self.scatter_from_model()
        n_cf = data.cf.shape[0] if n_cf is None else n_cf
        n_kg = data.kg.shape[0] if n_kg is None else n_kg
        self.loss_sum.zero_()
        if self._cf_src is not data.cf:  # batch ids -> rows of the padded cyclic layout, once per bound epoch array
            self._cf_padded = self.part.to_padded(data.cf).contiguous()
            self._cf_src = data.cf
            self.cf_ids = torch.zeros(3, data.cf.shape[2], dtype=torch.int64, device=self.dev)
            self.scratch = torch.empty(2 * data.cf.shape[2], device=self.dev)
        step = self._cf_runner() if n_cf else None
        for i in range(n_cf):
            step()
        cf_loss = float(self.loss_sum.item()) / max(n_cf, 1)
        if self.exchange is not None:
            self.exchange.check()
        self.gather_to_model()
        for grp in m._layers():  # aggregator weights were updated in place (they are the model's tensors)
            for t in grp:
                torch.autograd.graph.increment_version(t)
        kg_loss = 0.0
        if n_kg:
            self.single._resident = data
            kg_loss = self.single.run_epoch(None, n_cf=0, n_kg=n_kg, refresh=False)[1]
        if refresh:
            eh, er, et, ri = data.edges
            from .model import KGATMode

            m(eh, er, et, ri, mode=KGATMode.UPDATE_ATTENTION)
            g = m._graph()
            if (id(g), g.vals.data_ptr()) != self._graph_id:
                self._build_graph([m._cf_embedding_dim, *m._layer_dims])
            else:
                self.refresh_values()
        if self.part.world > 1:  # replicas of the replicated parameters: rank 0 wins (ulp-level atomics drift)
            for t in (m._relation_embedding.weight, m._trans_matrix, m._user_entity_embedding.weight):
                dist.broadcast(t.data, src=0)
        self.scatter_from_model()
        return cf_loss, kg_loss


def bench_main(args, metric, unit, workload, make_workload, config_dict, ClockSampler):
    """``bench.py --gpus N`` under torchrun: strong scaling of the epoch on the fixed C3-shaped CKG."""
    import json
    import os

    from . import _lib
    from .engine import TrainEngine
    from .trainer import build_model

    import sys

    rank, world = dist.get_rank(), dist.get_world_size()
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    # NCCL prints its version banner on stdout: keep stdout clean for the single JSON line
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    g, data = make_workload(workload)
    model = build_model(g, dev)
    part = CyclicPartition(g.node_num, world, rank)
    holder = TrainEngine(model, use_graphs=False).bind_resident(data.tensors())
    # the first refresh swaps the attentive structure: do it before building the sharded graph
    from .model import KGATMode

    model(*holder.edges, mode=KGATMode.UPDATE_ATTENTION)
    eng = ShardedEngine(model, part)
    for _ in range(2):  # set-up (never timed): capture the step graphs on two 2-step mini-epochs
        eng.run_epoch(holder, n_cf=2, n_kg=2)
    for _ in range(max(args.warmup, 0)):
        eng.run_epoch(holder)
    torch.cuda.synchronize()
    dist.barrier()
    _lib.LaunchCounter.count = 0
    with ClockSampler(dev.index or 0) as clocks:
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        losses = None
        for _ in range(args.steps):
            losses = eng.run_epoch(holder)
        t1.record()
        torch.cuda.synchronize()
        dist.barrier()
    ms = torch.tensor([t0.elapsed_time(t1)], device=dev)
    dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    epoch_s = float(ms.item()) / 1e3 / max(args.steps, 1)
    launches = _lib.LaunchCounter.count
    # end to end at N GPUs: every bench step (= epoch) first copies its inputs -- the pre-sampled batch blocks and the
    # refresh edge list -- from pinned host memory to the device, and the epoch's losses are read back
    e2e = None
    try:
        host = data.tensors(pin=True)
        pairs = [(holder.cf, host.cf_block), (holder.kg, host.kg_block)] + list(zip(holder.edges, host.edges))
        h2d = sum(src.numel() * src.element_size() for _, src in pairs)
        torch.cuda.synchronize()
        dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            for dst, src in pairs:
                dst.copy_(src, non_blocking=True)
            eng.run_epoch(holder)
        e1.record()
        torch.cuda.synchronize()
        dist.barrier()
        ms2 = torch.tensor([e0.elapsed_time(e1)], device=dev)
        dist.all_reduce(ms2, op=dist.ReduceOp.MAX)
        e2e = {"value": float(ms2.item()) / 1e3 / max(args.steps, 1), "unit": unit, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 8,
               "api": "ShardedEngine.run_epoch after copying the epoch's pre-sampled batch blocks and edge list from pinned host memory "
                      "(every rank); the two mean losses are read back per epoch"}
    except Exception as e:  # noqa: BLE001 - never lose the bench line over the secondary measurement
        e2e = {"unavailable": f"{type(e).__name__}: {e}"[:200]}
    if rank == 0:
        graph = model._graph()
        line = {
            "metric": metric, "value": epoch_s, "unit": unit, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": epoch_s * 1e3, "higher_is_better": False, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": config_dict(g, data, world),
            "propagation_edges_per_s": graph.nnz * 3 * 2 * data.n_cf / epoch_s,
            "cf_loss": losses[0], "kg_loss": losses[1], "gpu_launches": launches, "clocks": clocks.summary(),
            "e2e": e2e, "roofline": None, "cpu_baseline": None,
            "exchange": eng.exchange_kind,
            "note": "CF phase row-sharded (cyclic): 7 row exchanges + 1 gradient all-reduce per step over NVLink peer memory (store kernel "
                    "into the peers' tables + flag handshake; exchange=nccl uses NCCL collectives instead), the whole "
                    "step captured as one CUDA graph per rank; KG phase and the refresh are replicated; timed on the device, max over ranks",
        }
        os.write(json_fd, (json.dumps(line) + "\n").encode())
    # tear-down: drop the captured graphs (they hold NCCL work) before the communicator, and do not let a
    # wedged communicator destructor hang the process after the result is out
    eng._cf_graph = None
    eng.single._graphs.clear()
    torch.cuda.synchronize()
    dist.barrier()
    if eng.exchange is not None:
        eng.exchange.close()
    sys.stderr.flush()
    os._exit(0)

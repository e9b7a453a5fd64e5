"""Thin tensor-level wrappers over the C ABI (one Python function per ``kgat_*`` entry point).

PyTorch is used here for device memory and streams only: every wrapper validates its tensors
(CUDA, dtype, contiguity), takes raw ``data_ptr()`` values and launches on torch's *current* CUDA
stream so the kernels compose with torch's stream/graph machinery.  Nothing falls back to a torch
op when the library or a GPU is missing -- the call raises.
"""

from __future__ import annotations

import ctypes as C
import operator

import torch

from . import _lib
from ._lib import AdamTensorsT, KgatLibraryError, MhaT, TablesT, check

f32, i32, i64, u8 = torch.float32, torch.int32, torch.int64, torch.uint8


def _stream() -> int:
    """Raw handle of torch's current stream on the current device (two C calls; ``torch.cuda.current_stream()`` builds a Stream
    object through several layers of Python and costs ~10 us, more than some of the launches it serves)."""
    return torch._C._cuda_getCurrentRawStream(torch._C._cuda_getDevice())


class KernelTimer:
    """Optional per-kernel CUDA-event timing on the launching stream (bench.py roofline leg).
    ``with ops.KernelTimer() as t: ...`` then ``t.summary()`` -> {name: (launches, total_ms)}."""

    active: "KernelTimer | None" = None

    def __init__(self):
        self.events: dict[str, list] = {}

    def __enter__(self):
        KernelTimer.active = self
        return self

    def __exit__(self, *exc):
        KernelTimer.active = None

    def summary(self) -> dict:
        torch.cuda.synchronize()
        return {k: (len(v), sum(a.elapsed_time(b) for a, b in v)) for k, v in self.events.items()}


def _timed(name_fn):
    def deco(fn):
        def wrapper(*args, **kwargs):
            t = KernelTimer.active
            if t is None:
                return fn(*args, **kwargs)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            out = fn(*args, **kwargs)
            b.record()
            t.events.setdefault(name_fn(*args, **kwargs) if callable(name_fn) else name_fn, []).append((a, b))
            return out

        wrapper.__name__ = fn.__name__
        wrapper.__doc__ = fn.__doc__
        return wrapper

    return deco


def _ptr(t: torch.Tensor | None, dtype=None, name: str = "tensor", row_strided: bool = False) -> int | None:
    if t is None:
        return None
    if not t.is_cuda:
        raise KgatLibraryError(f"{name} must be a CUDA tensor (no CPU fallback in kgat_b200)")
    if dtype is not None and t.dtype != dtype:
        raise KgatLibraryError(f"{name} must be {dtype}, got {t.dtype}")
    if row_strided:  # 2-D, unit inner stride, 16-byte aligned rows
        if t.dim() != 2 or t.stride(1) != 1 or t.stride(0) % 4 or t.data_ptr() % 16:
            raise KgatLibraryError(f"{name} must be 2-D with unit inner stride and 16-byte aligned rows")
    elif not t.is_contiguous():
        raise KgatLibraryError(f"{name} must be contiguous")
    return t.data_ptr()


def _tables(tensors, allow_none: bool = False) -> TablesT:
    t = TablesT()
    t.n_tables = len(tensors)
    if len(tensors) > _lib.KGAT_MAX_LAYERS:
        raise KgatLibraryError(f"at most {_lib.KGAT_MAX_LAYERS} layer tables are supported")
    for i, x in enumerate(tensors):
        if x is None:
            if not allow_none:
                raise KgatLibraryError("missing table")
            t.dims[i], t.tables[i], t.lds[i] = 0, None, 0
            continue
        t.dims[i] = x.shape[1]
        t.tables[i] = _ptr(x, f32, "table")
        t.lds[i] = x.stride(0)
    return t


def device_info() -> dict:
    lib = _lib.load()
    sm, ma, mi, l2 = C.c_int32(), C.c_int32(), C.c_int32(), C.c_int64()
    check(lib.kgat_device_info(C.byref(sm), C.byref(ma), C.byref(mi), C.byref(l2)), "device_info")
    return {"sm_count": sm.value, "cc": (ma.value, mi.value), "l2_bytes": l2.value}


# ----------------------------------------------------------------------------------------------
# graph containers
# ----------------------------------------------------------------------------------------------


def group_by_key(keys: torch.Tensor, key_bits: int = 64):
    """Stable grouping of int64 keys (treated as unsigned).  Returns
    (order i32[n], group_of i32[n], group_ptr i32[g+1], unique_keys i64[g])."""
    lib = _lib.load()
    n = keys.numel()
    dev = keys.device
    ws_bytes = lib.kgat_group_by_key_workspace_bytes(n)
    if ws_bytes < 0:
        raise KgatLibraryError("group_by_key: too many keys")
    ws = torch.empty(ws_bytes, dtype=u8, device=dev)
    order = torch.empty(n, dtype=i32, device=dev)
    group_of = torch.empty(n, dtype=i32, device=dev)
    group_ptr = torch.empty(n + 1, dtype=i32, device=dev)
    uniq = torch.empty(max(n, 1), dtype=i64, device=dev)
    ng = C.c_int64(0)
    check(
        lib.kgat_group_by_key(
            _ptr(keys, i64, "keys"), n, key_bits, ws.data_ptr(), ws_bytes, order.data_ptr(), group_of.data_ptr(),
            group_ptr.data_ptr(), uniq.data_ptr(), C.byref(ng), _stream(),
        ),
        "group_by_key",
    )
    g = ng.value
    return order, group_of, group_ptr[: g + 1].clone(), uniq[:g].clone()


def decode_sorted_keys(unique_keys: torch.Tensor, n_major: int, n_minor: int):
    lib = _lib.load()
    n = unique_keys.numel()
    dev = unique_keys.device
    major_ptr = torch.empty(n_major + 1, dtype=i32, device=dev)
    minor_idx = torch.empty(n, dtype=i32, device=dev)
    check(
        lib.kgat_decode_sorted_keys(_ptr(unique_keys, i64), n, n_major, n_minor, major_ptr.data_ptr(), minor_idx.data_ptr(), _stream()),
        "decode_sorted_keys",
    )
    return major_ptr, minor_idx


def segment_sum(values: torch.Tensor, order: torch.Tensor, group_ptr: torch.Tensor, out: torch.Tensor | None = None):
    lib = _lib.load()
    g = group_ptr.numel() - 1
    if out is None:
        out = torch.empty(g, dtype=f32, device=values.device)
    check(lib.kgat_segment_sum_f32(_ptr(values, f32), _ptr(order, i32), _ptr(group_ptr, i32), g, _ptr(out, f32), _stream()), "segment_sum")
    return out


def gather_f32(src: torch.Tensor, index: torch.Tensor, out: torch.Tensor | None = None):
    lib = _lib.load()
    n = index.numel()
    if out is None:
        out = torch.empty(n, dtype=f32, device=src.device)
    check(lib.kgat_gather_f32(_ptr(src, f32), _ptr(index, i32), n, _ptr(out, f32), _stream()), "gather_f32")
    return out


def select_batch(src: torch.Tensor, counter_dev: torch.Tensor, dst: torch.Tensor):
    """dst (flat int64) = src[counter % n_batches] where src is [n_batches, ...] int64 on the device."""
    lib = _lib.load()
    n_batches = src.shape[0]
    elems = src[0].numel()
    if dst.numel() != elems:
        raise KgatLibraryError("select_batch: dst size mismatch")
    check(lib.kgat_select_batch_i64(_ptr(src, i64), n_batches, elems, _ptr(counter_dev, i64), _ptr(dst, i64), _stream()), "select_batch")
    return dst


def step_begin(src: torch.Tensor, step_dev: torch.Tensor, dst: torch.Tensor, lr, beta1, beta2, eps, hyper: torch.Tensor):
    """``select_batch`` + ``adam_advance`` on the same counter in one launch: dst = src[step % n_batches], then step += 1 and
    ``hyper`` holds the new step's Adam scalars."""
    lib = _lib.load()
    elems = src[0].numel()
    if dst.numel() != elems:
        raise KgatLibraryError("step_begin: dst size mismatch")
    check(lib.kgat_step_begin_i64(_ptr(src, i64), src.shape[0], elems, _ptr(step_dev, i64), _ptr(dst, i64), float(lr), float(beta1), float(beta2),
                                  float(eps), _ptr(hyper, f32), _stream()), "step_begin")


def fill_(t: torch.Tensor, value: float = 0.0):
    lib = _lib.load()
    check(lib.kgat_fill_f32(_ptr(t, f32), t.numel(), float(value), _stream()), "fill")
    return t


# ----------------------------------------------------------------------------------------------
# K1 SpMM
# ----------------------------------------------------------------------------------------------


def _spmm_name(plan, col_idx, vals, x, out, addend=None, partials=None, row_mask=None, edge_mask=None, rows=None, n_rows_dev=None, tag=""):
    kind = "_rows" if rows is not None else ("_edges" if edge_mask is not None else ("_pruned" if row_mask is not None else ""))
    return f"spmm{'T' if addend is not None else ''}_d{x.shape[1]}{kind}{tag}"


@_timed(_spmm_name)
def spmm(plan, col_idx, vals, x: torch.Tensor, out: torch.Tensor, addend: torch.Tensor | None = None, partials=None,
         row_mask: torch.Tensor | None = None, edge_mask: torch.Tensor | None = None, rows: torch.Tensor | None = None,
         n_rows_dev: torch.Tensor | None = None, tag: str = ""):
    """out = A @ x (+ addend); ``plan`` is a graph.SpmmPlan.  ``row_mask`` / ``edge_mask``: node bitmaps of a
    ``frontier.Frontier`` level (only the rows in ``row_mask`` are computed; edges / addend rows outside ``edge_mask`` are
    dropped).  With the level's row list (``rows``, ``n_rows_dev``; needs ``row_mask`` too) or with an ``edge_mask`` alone the
    persistent row-list kernel runs; a ``row_mask`` without a list uses the grid-per-task kernel."""
    d = x.shape[1]
    # the kernels write d floats at row * ld of every plan row: a narrower or shorter output would be written out of bounds
    for name, t in (("out", out), ("addend", addend)):
        if t is not None and (t.dim() != 2 or t.shape[1] != d or t.shape[0] < plan.n_rows):
            raise KgatLibraryError(f"spmm: {name} of shape {tuple(t.shape)} does not cover {plan.n_rows} rows of width {d}")
    lib = _lib.load()
    if plan.n_heavy > 0:
        need = plan.n_partials * d
        if partials is None or partials.numel() < need:
            raise KgatLibraryError("spmm: partials scratch too small")
    args = (
        _ptr(plan.tasks, i32), plan.n_tasks, _ptr(plan.heavy, i32) if plan.n_heavy else None, plan.n_heavy,
        _ptr(col_idx, i32), _ptr(vals, f32), _ptr(x, f32, "x", True), x.shape[0], x.stride(0), _ptr(out, f32, "out", True), out.stride(0),
        _ptr(addend, f32, "addend", True) if addend is not None else None, addend.stride(0) if addend is not None else 0, d,
        _ptr(partials, f32) if partials is not None else None,
    )
    use_rows_kernel = (rows is not None or (edge_mask is not None and row_mask is None)) and d in (16, 32, 64, 128)
    if use_rows_kernel:
        n_bits = max(x.shape[0], out.shape[0])
        for m in (row_mask, edge_mask):
            if m is not None and m.numel() * 32 < n_bits:
                raise KgatLibraryError("spmm: node bitmap too small")
        if rows is not None and (row_mask is None or n_rows_dev is None or plan.light_rank is None):
            raise KgatLibraryError("spmm: a row list needs its bitmap, its device-side count and a plan with light_rank")
        check(
            lib.kgat_spmm_csr_rows(
                _ptr(plan.tasks, i32), plan.n_tasks, plan.n_partials, _ptr(plan.light_rank, i32) if plan.light_rank is not None else None,
                _ptr(plan.heavy, i32) if plan.n_heavy else None, plan.n_heavy, *args[4:],
                _ptr(rows, i32) if rows is not None else None, _ptr(n_rows_dev, i32) if rows is not None else None,
                _ptr(row_mask, i32) if row_mask is not None else None, _ptr(edge_mask, i32) if edge_mask is not None else None, n_bits, _stream(),
            ),
            "spmm_csr_rows",
        )
    elif row_mask is None and edge_mask is None:
        check(lib.kgat_spmm_csr(*args, _stream()), "spmm_csr")
    else:
        words = (max(x.shape[0], out.shape[0]) + 31) // 32
        for m in (row_mask, edge_mask):
            if m is not None and m.numel() < words:
                raise KgatLibraryError("spmm: node bitmap too small")
        check(lib.kgat_spmm_csr_masked(*args, _ptr(row_mask, i32) if row_mask is not None else None,
                                       _ptr(edge_mask, i32) if edge_mask is not None else None, _stream()), "spmm_csr_masked")
    return out


@_timed(lambda plan, col_idx, vals, g, out, *a, **k: f"spmmT_d{g.shape[1]}_scatter{k.get('tag', '')}")
def spmm_scatter_rows(plan, col_idx, vals, g: torch.Tensor, out: torch.Tensor, rows, n_rows_dev, max_rows: int, row_mask, addend=None,
                      tag: str = ""):
    """out[c] += A[r, c] * g[r] over the listed rows r (and out[r] += addend[r]); ``plan`` / ``col_idx`` / ``vals`` of A itself.
    The destination rows of ``out`` must have been zeroed (frontier_zero_rows)."""
    d = g.shape[1]
    for name, t in (("out", out), ("addend", addend)):
        if t is not None and (t.dim() != 2 or t.shape[1] != d):
            raise KgatLibraryError(f"spmm_scatter_rows: {name} of shape {tuple(t.shape)} does not have the width {d} of g")
    lib = _lib.load()
    check(
        lib.kgat_spmm_scatter_rows(
            _ptr(plan.tasks, i32), plan.n_partials, _ptr(plan.light_rank, i32), _ptr(rows, i32), _ptr(n_rows_dev, i32), int(max_rows),
            _ptr(row_mask, i32), _ptr(col_idx, i32), _ptr(vals, f32), _ptr(g, f32, "g", True), g.stride(0),
            _ptr(addend, f32, "addend", True) if addend is not None else None, addend.stride(0) if addend is not None else 0,
            _ptr(out, f32, "out", True), out.stride(0), d, _stream(),
        ),
        "spmm_scatter_rows",
    )
    return out


# ----------------------------------------------------------------------------------------------
# needed-row frontier of a TRAIN_CF step (csrc/frontier.cu)
# ----------------------------------------------------------------------------------------------


def frontier_scratch_ints(n_nodes: int) -> int:
    return int(_lib.load().kgat_frontier_scratch_ints(int(n_nodes)))


def frontier_mark_ids(ids: torch.Tensor, n_nodes: int, flags: torch.Tensor, bad_count: torch.Tensor | None = None):
    """flags (uint8, one byte per node, zero between builds)[ids] = 1"""
    lib = _lib.load()
    if flags.numel() < (n_nodes + 31) // 32 * 32:
        raise KgatLibraryError("frontier_mark_ids: flag array too small")
    check(lib.kgat_frontier_mark_ids(_ptr(ids, i64, "ids"), ids.numel(), int(n_nodes), _ptr(flags, u8),
                                     _ptr(bad_count, i32) if bad_count is not None else None, _stream()), "frontier_mark_ids")


def frontier_expand(plan, col_idx, rows, count_dev, max_rows: int, level_bitmap, flags):
    """flags[r] = flags[c] = 1 for the listed rows r and the columns c of their CSR rows; ``plan``: the graph's SpmmPlan."""
    lib = _lib.load()
    check(lib.kgat_frontier_expand(_ptr(plan.tasks, i32), plan.n_partials, _ptr(plan.light_rank, i32), _ptr(col_idx, i32), _ptr(rows, i32),
                                   _ptr(count_dev, i32), int(max_rows), _ptr(level_bitmap, i32), _ptr(flags, u8), plan.light_rank.numel(),
                                   _stream()), "frontier_expand")


def frontier_list(flags, bitmap, n_nodes: int, scratch, rows, count_dev):
    """bitmap <- flags (flags cleared), rows <- ascending set bits, count_dev <- their number"""
    lib = _lib.load()
    if scratch.numel() < frontier_scratch_ints(n_nodes) or bitmap.numel() * 32 < n_nodes or flags.numel() < (n_nodes + 31) // 32 * 32:
        raise KgatLibraryError("frontier_list: scratch / bitmap / flags too small")
    check(lib.kgat_frontier_list(_ptr(flags, u8), _ptr(bitmap, i32), int(n_nodes), _ptr(scratch, i32), _ptr(rows, i32), _ptr(count_dev, i32),
                                 _stream()), "frontier_list")


def frontier_segment(rows, count_dev, bitmap, n_nodes: int, lo: int, hi: int, out_rows, out_count_dev, out_bitmap):
    """The part of a frontier level inside the node range [lo, hi): its row-list segment, count and bitmap words."""
    lib = _lib.load()
    if out_rows.numel() < hi - lo or out_bitmap.numel() * 32 < n_nodes:
        raise KgatLibraryError("frontier_segment: output buffers too small")
    check(lib.kgat_frontier_segment(_ptr(rows, i32), _ptr(count_dev, i32), _ptr(bitmap, i32), int(n_nodes), int(lo), int(hi), _ptr(out_rows, i32),
                                    _ptr(out_count_dev, i32), _ptr(out_bitmap, i32), _stream()), "frontier_segment")


def frontier_zero_rows(table: torch.Tensor, rows, count_dev, max_rows: int):
    lib = _lib.load()
    check(lib.kgat_frontier_zero_rows(_ptr(table, f32, "table", True), table.stride(0), table.shape[1], _ptr(rows, i32), _ptr(count_dev, i32),
                                      int(max_rows), _stream()), "frontier_zero_rows")


# ----------------------------------------------------------------------------------------------
# K2/K3 bi-interaction aggregator
# ----------------------------------------------------------------------------------------------


@_timed(lambda E, S, W1, *a, **k: f"biagg_fwd_{E.shape[1]}x{W1.shape[0]}{'_rows' if k.get('rows') is not None else ''}{k.get('tag', '')}")
def biagg_forward(E, S, W1, b1, W2, b2, out, inv_norm, flags, dropout_p=0.0, seed=0, offset=0, keep_bits=None, seed_dev=None,
                  peer_out=None, rows=None, n_rows_dev=None, max_rows=None, tag: str = ""):
    """``peer_out``: int64 device tensor of pointers to this rank's rows in every peer's copy of ``out`` (peer.PeerArena).
    ``rows`` / ``n_rows_dev`` / ``max_rows``: needed-row list of a ``frontier.Frontier`` level (arrays stay node-indexed)."""
    lib = _lib.load()
    n, d_in = E.shape
    d_out = W1.shape[0]
    if rows is not None:
        if peer_out is not None:
            raise KgatLibraryError("biagg_forward: a row list and peer stores are mutually exclusive")
        check(
            lib.kgat_biagg_forward_rows(
                _ptr(E, f32, "E"), _ptr(S, f32, "S"), _ptr(rows, i32, "rows"), _ptr(n_rows_dev, i32), int(max_rows), d_in, d_out,
                _ptr(W1, f32), _ptr(b1, f32), _ptr(W2, f32), _ptr(b2, f32), float(dropout_p), int(seed), int(offset),
                _ptr(seed_dev, i64) if seed_dev is not None else None, _ptr(keep_bits, i32) if keep_bits is not None else None,
                _ptr(out, f32, "out"), out.stride(0), _ptr(inv_norm, f32) if inv_norm is not None else None,
                _ptr(flags, u8) if flags is not None else None, _stream(),
            ),
            f"biagg_forward_rows({d_in}->{d_out})",
        )
        return out
    check(
        lib.kgat_biagg_forward(
            _ptr(E, f32, "E"), _ptr(S, f32, "S"), n, d_in, d_out, _ptr(W1, f32), _ptr(b1, f32), _ptr(W2, f32), _ptr(b2, f32),
            float(dropout_p), int(seed), int(offset), _ptr(seed_dev, i64) if seed_dev is not None else None,
            _ptr(keep_bits, i32) if keep_bits is not None else None,
            _ptr(out, f32, "out"), out.stride(0), _ptr(inv_norm, f32) if inv_norm is not None else None,
            _ptr(flags, u8) if flags is not None else None,
            _ptr(peer_out, i64) if peer_out is not None else None, peer_out.numel() if peer_out is not None else 0, _stream(),
        ),
        f"biagg_forward({d_in}->{d_out})",
    )
    return out


def biagg_backward_ctas(n: int, d_in: int, d_out: int, rows: bool = False) -> int:
    lib = _lib.load()
    return lib.kgat_biagg_backward_rows_ctas(n, d_in, d_out) if rows else lib.kgat_biagg_backward_ctas(n, d_in, d_out)


@_timed(lambda g_out, out, inv_norm, flags, E, S, W1, *a, **k: f"biagg_bwd_{E.shape[1]}x{W1.shape[0]}{'_rows' if k.get('rows') is not None else ''}{k.get('tag', '')}")
def biagg_backward(g_out, out, inv_norm, flags, E, S, W1, W2, dropout_p, g_S, g_E, partials, n_ctas, peer_out=None, rows=None,
                   n_rows_dev=None, max_rows=None, tag: str = ""):
    lib = _lib.load()
    n, d_in = E.shape
    d_out = W1.shape[0]
    if partials.numel() < n_ctas * (2 * d_in * d_out + 2 * d_out):
        raise KgatLibraryError("biagg_backward: partials scratch too small")
    if rows is not None:
        if peer_out is not None:
            raise KgatLibraryError("biagg_backward: a row list and peer stores are mutually exclusive")
        check(
            lib.kgat_biagg_backward_rows(
                _ptr(g_out, f32, "g_out"), g_out.stride(0), _ptr(out, f32), out.stride(0), _ptr(inv_norm, f32), _ptr(flags, u8),
                _ptr(E, f32), _ptr(S, f32), _ptr(rows, i32, "rows"), _ptr(n_rows_dev, i32), int(max_rows), d_in, d_out, _ptr(W1, f32),
                _ptr(W2, f32), float(dropout_p), _ptr(g_S, f32), _ptr(g_E, f32), _ptr(partials, f32), n_ctas, _stream(),
            ),
            f"biagg_backward_rows({d_in}->{d_out})",
        )
        return
    check(
        lib.kgat_biagg_backward(
            _ptr(g_out, f32, "g_out"), g_out.stride(0), _ptr(out, f32), out.stride(0), _ptr(inv_norm, f32), _ptr(flags, u8),
            _ptr(E, f32), _ptr(S, f32), n, d_in, d_out, _ptr(W1, f32), _ptr(W2, f32), float(dropout_p), _ptr(g_S, f32),
            _ptr(g_E, f32), _ptr(partials, f32), n_ctas,
            _ptr(peer_out, i64) if peer_out is not None else None, peer_out.numel() if peer_out is not None else 0, _stream(),
        ),
        f"biagg_backward({d_in}->{d_out})",
    )


@_timed("biagg_reduce")
def biagg_reduce_param_grads(partials, n_ctas, d_in, d_out, gW1, gb1, gW2, gb2, accumulate=False):
    lib = _lib.load()
    check(
        lib.kgat_biagg_reduce_param_grads(
            _ptr(partials, f32), n_ctas, d_in, d_out, _ptr(gW1, f32), _ptr(gb1, f32), _ptr(gW2, f32), _ptr(gb2, f32),
            1 if accumulate else 0, _stream(),
        ),
        "biagg_reduce_param_grads",
    )


# ----------------------------------------------------------------------------------------------
# K4 BPR, K5 TransR
# ----------------------------------------------------------------------------------------------


def zero_rows_(table: torch.Tensor, ids: torch.Tensor):
    """table[ids] = 0 (int64 ids; out-of-range ones ignored)."""
    lib = _lib.load()
    check(lib.kgat_zero_rows_i64(_ptr(table, f32, "table", True), table.shape[0], table.stride(0), table.shape[1], _ptr(ids, i64, "ids"),
                                 ids.numel(), _stream()), "zero_rows")
    return table


@_timed("bpr_fwd")
def bpr_forward(tables, users, pos, neg, reg, loss, scratch, loss_sum=None, publish=None):
    lib = _lib.load()
    b = users.numel()
    if scratch.numel() < 2 * b:
        raise KgatLibraryError("bpr_forward: scratch needs 2*batch floats")
    t = _tables(tables)
    check(
        lib.kgat_bpr_forward(C.byref(t), _ptr(users, i64, "users"), _ptr(pos, i64, "pos"), _ptr(neg, i64, "neg"), b, float(reg),
                             _ptr(loss, f32), _ptr(loss_sum, f32) if loss_sum is not None else None, _ptr(scratch, f32),
                             C.byref(publish) if publish is not None else None, _stream()),
        "bpr_forward",
    )


@_timed("bpr_bwd")
def bpr_backward(tables, grad_tables, users, pos, neg, reg, scratch, g_loss):
    lib = _lib.load()
    t = _tables(tables)
    g = _tables(grad_tables, allow_none=True)
    for i, x in enumerate(grad_tables):
        if x is not None:
            g.dims[i] = tables[i].shape[1]
    check(
        lib.kgat_bpr_backward(C.byref(t), C.byref(g), _ptr(users, i64), _ptr(pos, i64), _ptr(neg, i64), users.numel(), float(reg),
                              _ptr(scratch, f32), _ptr(g_loss, f32), _stream()),
        "bpr_backward",
    )


@_timed("transr_fwd")
def transr_forward(emb, rel_emb, W, heads, rels, pos_t, neg_t, reg, loss, scratch):
    lib = _lib.load()
    b = heads.numel()
    if scratch.numel() < 2 * b:
        raise KgatLibraryError("transr_forward: scratch needs 2*batch floats")
    check(
        lib.kgat_transr_forward(_ptr(emb, f32), _ptr(rel_emb, f32), _ptr(W, f32), emb.shape[1], rel_emb.shape[1], _ptr(heads, i64),
                                _ptr(rels, i64), _ptr(pos_t, i64), _ptr(neg_t, i64), b, float(reg), _ptr(loss, f32),
                                _ptr(scratch, f32), _stream()),
        f"transr_forward(d={emb.shape[1]}, k={rel_emb.shape[1]})",
    )


@_timed("transr_bwd")
def transr_claim_rows(heads, pos_t, neg_t, d: int, row_slot, g_rows):
    """Compact gradient rows for a TransR batch: one slot per distinct node in ``row_slot`` (int32 [n_nodes], -1 = free),
    ``g_rows`` (3B x d) zeroed."""
    lib = _lib.load()
    if g_rows.numel() < 3 * heads.numel() * d:
        raise KgatLibraryError("transr_claim_rows: g_rows needs 3 * batch * d floats")
    check(lib.kgat_transr_claim_rows(_ptr(heads, i64), _ptr(pos_t, i64), _ptr(neg_t, i64), heads.numel(), int(d), _ptr(row_slot, i32),
                                     _ptr(g_rows, f32), _stream()), "transr_claim_rows")


def transr_scratch_numel(batch: int, k: int) -> int:
    """Floats of the ``scratch`` a fused TransR step needs: the per-sample margin and L2 term, then the per-sample projection
    gradients its second launch reduces in sample order (bit-identical gradients from run to run)."""
    return 2 * batch + 4 * batch * k


@_timed("transr_step")
def transr_step(emb, rel_emb, W, heads, rels, pos_t, neg_t, reg, loss, loss_sum, scratch, row_slot, g_rows, g_rel, g_W, publish=None):
    """Claim compact gradient rows + zero the gradient buffers, TransR forward and backward in one pass, loss value
    (added to ``loss_sum`` when given): the KG half-step of the epoch engine in three launches."""
    lib = _lib.load()
    if g_rows.numel() < 3 * heads.numel() * emb.shape[1] or scratch.numel() < transr_scratch_numel(heads.numel(), rel_emb.shape[1]):
        raise KgatLibraryError("transr_step: g_rows needs 3 * batch * d floats, scratch transr_scratch_numel(batch, k)")
    check(lib.kgat_transr_step(_ptr(emb, f32), _ptr(rel_emb, f32), _ptr(W, f32), emb.shape[1], rel_emb.shape[1], rel_emb.shape[0],
                               _ptr(heads, i64), _ptr(rels, i64), _ptr(pos_t, i64), _ptr(neg_t, i64), heads.numel(), float(reg),
                               _ptr(loss, f32), _ptr(loss_sum, f32) if loss_sum is not None else None, _ptr(scratch, f32),
                               _ptr(row_slot, i32), _ptr(g_rows, f32), _ptr(g_rel, f32), _ptr(g_W, f32),
                               C.byref(publish) if publish is not None else None, _stream()), "transr_step")


def transr_rows_to_dense(g_rows, row_slot, heads, pos_t, neg_t, dense, keep_ids=None):
    """dense[id] = g_rows[row_slot[id]] for the batch's ids (the dense ``embedding.weight.grad`` of a TransR step).
    ``keep_ids``: three int64 [B] tensors that receive copies of heads / pos_t / neg_t in the same launch."""
    lib = _lib.load()
    check(lib.kgat_transr_rows_to_dense(_ptr(g_rows, f32), _ptr(row_slot, i32), _ptr(heads, i64), _ptr(pos_t, i64), _ptr(neg_t, i64),
                                        heads.numel(), dense.shape[1], _ptr(dense, f32, "dense", True), dense.stride(0),
                                        *((_ptr(keep_ids[0], i64), _ptr(keep_ids[1], i64), _ptr(keep_ids[2], i64)) if keep_ids is not None
                                          else (None, None, None)), _stream()),
          "transr_rows_to_dense")


def transr_release_rows(dense, ids, row_slot):
    """dense[ids] = 0 and row_slot[ids] = -1 (the previous batch's rows)."""
    lib = _lib.load()
    check(lib.kgat_transr_release_rows(_ptr(dense, f32, "dense", True), dense.shape[0], dense.stride(0), dense.shape[1], _ptr(ids, i64),
                                       ids.numel(), _ptr(row_slot, i32), _stream()), "transr_release_rows")


def transr_backward(emb, rel_emb, W, heads, rels, pos_t, neg_t, reg, scratch, g_loss, g_emb, g_rel, g_W, row_slot=None):
    lib = _lib.load()
    check(
        lib.kgat_transr_backward(_ptr(emb, f32), _ptr(rel_emb, f32), _ptr(W, f32), emb.shape[1], rel_emb.shape[1], _ptr(heads, i64),
                                 _ptr(rels, i64), _ptr(pos_t, i64), _ptr(neg_t, i64), heads.numel(), float(reg), _ptr(scratch, f32),
                                 _ptr(g_loss, f32), _ptr(g_emb, f32), _ptr(g_rel, f32), _ptr(g_W, f32),
                                 _ptr(row_slot, i32) if row_slot is not None else None, _stream()),
        "transr_backward",
    )


# ----------------------------------------------------------------------------------------------
# K6-K8 attention refresh
# ----------------------------------------------------------------------------------------------


def _mha(mha_params: dict, n_heads: int, eps: float):
    m = MhaT()
    keep = []
    for field, key in (("Wv", "Wv"), ("bv", "bv"), ("Wo", "Wo"), ("bo", "bo"), ("ln_gamma", "gamma"), ("ln_beta", "beta")):
        t = mha_params[key]
        keep.append(t)
        setattr(m, field, _ptr(t, f32, key))
    m.ln_eps = eps
    m.n_heads = n_heads
    return m, keep


def mha_forward(x_tail, mha_params, dropout_p=0.0, head_bits=None, seed=0, offset=0, n_heads=8, eps=1e-5):
    """MultiHeadAttention.forward's value path: LayerNorm(Wo drop(Wv x + bv) + bo) for every row of ``x_tail`` (n x d)."""
    lib = _lib.load()
    n, d = x_tail.shape
    m, _keep = _mha(mha_params, n_heads, eps)
    out = torch.empty(n, d, dtype=f32, device=x_tail.device)
    check(lib.kgat_mha_forward(_ptr(x_tail, f32, "tail_embedding"), n, d, C.byref(m), float(dropout_p),
                               _ptr(head_bits, u8) if head_bits is not None else None, int(seed), int(offset), _ptr(out, f32), _stream()),
          f"mha_forward(d={d})")
    return out


def att_pair_scores(emb, W, pair_tail, pair_rel, mha_params, n_heads=8, eps=1e-5, want_v=False, want_score=True):
    lib = _lib.load()
    n_pairs = pair_tail.numel()
    d = emb.shape[1]
    m, _keep = _mha(mha_params, n_heads, eps)
    v_out = torch.empty(n_pairs, d, dtype=f32, device=emb.device) if want_v else None
    s_out = torch.empty(n_pairs, dtype=f32, device=emb.device) if want_score else None
    check(
        lib.kgat_att_pair_scores(_ptr(emb, f32), _ptr(W, f32), d, _ptr(pair_tail, i32), _ptr(pair_rel, i32), n_pairs, C.byref(m),
                                 _ptr(v_out, f32) if want_v else None, _ptr(s_out, f32) if want_score else None, _stream()),
        f"att_pair_scores(d={d})",
    )
    return v_out, s_out


def att_pair_project(emb, W, pair_node, pair_rel):
    """x[p] = emb[pair_node[p]] @ W[pair_rel[p]] for unique (node, relation) pairs (canonical-KGAT score mode)."""
    lib = _lib.load()
    n_pairs, d = pair_node.numel(), emb.shape[1]
    out = torch.empty(n_pairs, d, dtype=f32, device=emb.device)
    check(lib.kgat_att_pair_project(_ptr(emb, f32), _ptr(W, f32), d, _ptr(pair_node, i32), _ptr(pair_rel, i32), n_pairs, _ptr(out, f32), _stream()),
          f"att_pair_project(d={d})")
    return out


def att_edge_scores_kgat(x_head, head_pair, x_tail, tail_pair, rel_emb, edge_rel):
    """score[e] = <x_tail[tail_pair[e]], tanh(x_head[head_pair[e]] + rel_emb[edge_rel[e]])>  -- the KGAT paper's pi(h, r, t)."""
    lib = _lib.load()
    n_edges, d = head_pair.numel(), x_head.shape[1]
    out = torch.empty(n_edges, dtype=f32, device=x_head.device)
    check(lib.kgat_att_edge_scores_kgat(_ptr(x_head, f32), _ptr(head_pair, i32), _ptr(x_tail, f32), _ptr(tail_pair, i32), _ptr(rel_emb, f32),
                                        _ptr(edge_rel, i32), n_edges, d, _ptr(out, f32), _stream()), "att_edge_scores_kgat")
    return out


def att_edge_scores_dropout(pair_v, pair_of_edge, mha_params, dropout_p, head_bits=None, seed=0, offset=0, n_heads=8, eps=1e-5, seed_dev=None):
    lib = _lib.load()
    n_edges = pair_of_edge.numel()
    d = pair_v.shape[1]
    m, _keep = _mha(mha_params, n_heads, eps)
    out = torch.empty(n_edges, dtype=f32, device=pair_v.device)
    check(
        lib.kgat_att_edge_scores_dropout(_ptr(pair_v, f32), _ptr(pair_of_edge, i32), n_edges, d, C.byref(m), float(dropout_p),
                                         _ptr(head_bits, u8) if head_bits is not None else None, int(seed), int(offset),
                                         _ptr(seed_dev, i64) if seed_dev is not None else None, _ptr(out, f32), _stream()),
        "att_edge_scores_dropout",
    )
    return out


def att_row_softmax(row_ptr, slot_ptr, edge_weight, vals_out, pair_score=None, pair_of_edge=None, edge_score=None):
    lib = _lib.load()
    check(
        lib.kgat_att_row_softmax(_ptr(row_ptr, i32), row_ptr.numel() - 1, _ptr(slot_ptr, i32),
                                 _ptr(pair_score, f32) if pair_score is not None else None,
                                 _ptr(pair_of_edge, i32) if pair_of_edge is not None else None,
                                 _ptr(edge_score, f32) if edge_score is not None else None, _ptr(edge_weight, f32),
                                 _ptr(vals_out, f32), _stream()),
        "att_row_softmax",
    )
    return vals_out


def att_edge_weights(deg_head, deg_tail, mult=None):
    lib = _lib.load()
    n = deg_head.numel()
    out = torch.empty(n, dtype=f32, device=deg_head.device)
    check(lib.kgat_att_edge_weights(_ptr(deg_head, i32), _ptr(deg_tail, i32), _ptr(mult, f32) if mult is not None else None, n,
                                    _ptr(out, f32), _stream()), "att_edge_weights")
    return out


# ----------------------------------------------------------------------------------------------
# K9/K10 predict
# ----------------------------------------------------------------------------------------------


def gather_concat(tables, ids, out=None):
    lib = _lib.load()
    t = _tables(tables)
    n = ids.numel()
    width = sum(x.shape[1] for x in tables)
    if out is None:
        out = torch.empty(n, width, dtype=f32, device=tables[0].device)
    check(lib.kgat_gather_concat(C.byref(t), _ptr(ids, i64, "ids"), n, _ptr(out, f32), out.stride(0), _stream()), "gather_concat")
    return out


def sgemm_nt(A, B, out=None):
    lib = _lib.load()
    m, k = A.shape
    n = B.shape[0]
    if out is None:
        out = torch.empty(m, n, dtype=f32, device=A.device)
    if A.stride(1) != 1 or B.stride(1) != 1 or out.stride(1) != 1:
        raise KgatLibraryError("sgemm_nt: inner strides must be 1")
    for t_ in (A, B, out):
        if not t_.is_cuda or t_.dtype != f32:
            raise KgatLibraryError("sgemm_nt: CUDA fp32 tensors required")
    check(lib.kgat_sgemm_nt(A.data_ptr(), A.stride(0), B.data_ptr(), B.stride(0), out.data_ptr(), out.stride(0), m, n, k, _stream()), "sgemm_nt")
    return out


def mask_scores_(scores, mask_ptr, mask_items):
    lib = _lib.load()
    m, n = scores.shape
    check(lib.kgat_mask_scores(_ptr(scores, f32), scores.stride(0), m, n, _ptr(mask_ptr, i32), _ptr(mask_items, i32), _stream()), "mask_scores")
    return scores


def topk_rows(scores, k: int, want_values: bool = False):
    lib = _lib.load()
    m, n = scores.shape
    idx = torch.empty(m, k, dtype=i32, device=scores.device)
    val = torch.empty(m, k, dtype=f32, device=scores.device) if want_values else None
    check(lib.kgat_topk_rows(_ptr(scores, f32), scores.stride(0), m, n, k, idx.data_ptr(), val.data_ptr() if want_values else None, _stream()), "topk_rows")
    return (idx, val) if want_values else idx


def explain_paths(graph, src: torch.Tensor, dst: torch.Tensor, k: int, max_hops: int):
    """Top-``k`` attention-weighted simple paths of 1 .. ``max_hops`` hops from ``src[j]`` to ``dst[j]`` through the attentive
    matrix of ``graph`` (an ``AttentiveGraph``), with the number and summed weight of all such paths per length
    (``kgat_explain_paths``).  ``src`` / ``dst``: node ids, any integer dtype, on the graph's device.
    Returns ``(nodes [P,k,H+1] int64, slots [P,k,H] int64, hops [P,k] int32, weight [P,k] fp32, count [P,H] int64,
    mass [P,H] fp32)``.  Raises ``ValueError`` for an id outside ``[0, graph.n)`` (read back after the launches)."""
    k, max_hops = int(k), int(max_hops)
    if not 1 <= k <= 64:
        raise ValueError(f"k must be in [1, 64], got {k}")
    if max_hops not in (1, 2, 3):
        raise ValueError(f"max_hops must be 1, 2 or 3, got {max_hops}")
    if src.dim() != 1 or dst.dim() != 1 or src.numel() != dst.numel():
        raise ValueError(f"src and dst must be 1-D of equal length, got {tuple(src.shape)} and {tuple(dst.shape)}")
    lib = _lib.load()
    dev = graph.col_idx.device
    P, H = src.numel(), max_hops
    nodes = torch.empty(P, k, H + 1, dtype=i64, device=dev)
    slots = torch.empty(P, k, H, dtype=i64, device=dev)
    hops = torch.empty(P, k, dtype=i32, device=dev)
    weight = torch.empty(P, k, dtype=f32, device=dev)
    count = torch.empty(P, H, dtype=i64, device=dev)
    mass = torch.empty(P, H, dtype=f32, device=dev)
    if P == 0:
        return nodes, slots, hops, weight, count, mass
    ids = torch.cat([src.to(device=dev, dtype=i64), dst.to(device=dev, dtype=i64)]).contiguous()
    ids32 = torch.empty(2 * P, dtype=i32, device=dev)
    bad = torch.zeros(1, dtype=i32, device=dev)
    check(lib.kgat_ids64_to_i32(_ptr(ids, i64), 2 * P, graph.n, ids32.data_ptr(), bad.data_ptr(), _stream()), "explain_paths ids")
    ws_bytes = int(lib.kgat_explain_paths_workspace_bytes(P, k, H))
    ws = torch.empty(max(ws_bytes, 1), dtype=u8, device=dev)
    check(lib.kgat_explain_paths(
        _ptr(graph.row_ptr, i32), _ptr(graph.col_idx, i32), _ptr(graph.vals, f32), _ptr(graph.t_ptr, i32), _ptr(graph.t_idx, i32),
        _ptr(graph.t_perm, i32), graph.n, ids32.data_ptr(), ids32.data_ptr() + 4 * P, P, k, H, nodes.data_ptr(), slots.data_ptr(),
        hops.data_ptr(), weight.data_ptr(), count.data_ptr(), mass.data_ptr(), ws.data_ptr(), ws_bytes, _stream()), "explain_paths")
    n_bad = int(bad.item())
    if n_bad:
        raise ValueError(f"{n_bad} node id(s) outside [0, {graph.n})")
    return nodes, slots, hops, weight, count, mass


def _ids64(ids: torch.Tensor, name: str, dev) -> torch.Tensor:
    """1-D ids of any integer dtype, CPU or CUDA -> contiguous int64 on ``dev``."""
    if ids.dim() != 1 or ids.dtype.is_floating_point or ids.dtype == torch.bool:
        raise ValueError(f"{name} must be a 1-D integer tensor, got {ids.dtype} of shape {tuple(ids.shape)}")
    return ids.to(device=dev, dtype=i64).contiguous()


def range_check(checks, dev, flags=(), values=()) -> list:
    """checks: (name, int64 ids on dev, bound >= 1); flags: (message, device integer scalar that is nonzero on failure);
    values: device integer scalars the caller needs on the host.  Converts every id list to int32 and reads the out-of-range
    counts, the flags and the values back in one synchronisation, before any kernel indexes with the ids; ValueError for the
    first check or flag that fails.  Returns the int32 id lists, followed by the values as ints."""
    lib = _lib.load()
    bad = torch.zeros(len(checks) + len(flags), dtype=i32, device=dev)
    outs = []
    for j, (name, ids, bound) in enumerate(checks):
        out = torch.empty(ids.numel(), dtype=i32, device=dev)
        if ids.numel():
            check(lib.kgat_ids64_to_i32(_ptr(ids, i64), ids.numel(), bound, out.data_ptr(), bad.data_ptr() + 4 * j, _stream()), name)
        outs.append(out)
    for j, (_, flag) in enumerate(flags):
        bad[len(checks) + j] = flag
    if values:
        got = torch.cat([bad.to(i64), torch.stack([torch.as_tensor(v, device=dev).to(i64).reshape(()) for v in values])]).tolist()
    else:
        got = bad.tolist()
    for (name, _, bound), n_bad in zip(checks, got):
        if n_bad:
            raise ValueError(f"{n_bad} {name} outside [0, {bound})")
    for (msg, _), n_bad in zip(flags, got[len(checks) :]):
        if n_bad:
            raise ValueError(msg)
    return outs + got[len(checks) + len(flags) :]


def require_groups(groups, n_ent: int):
    """``require`` groups as lists of ints; ValueError for an empty group or an entity id outside ``[0, n_ent)``."""
    groups = [list(map(int, g)) for g in groups]
    if any(len(g) == 0 for g in groups):
        raise ValueError("every group of `require` must hold at least one entity id")
    if any(not 0 <= e < n_ent for g in groups for e in g):
        raise ValueError(f"entity ids of `require` must lie in [0, {n_ent})")
    return groups


def recommend_filter(graph, items: torch.Tensor, groups, user_num: int):
    """Candidate filter of ``KGAT.recommend`` (``kgat_recommend_filter``): keeps the items ``p`` of ``items`` (entity ids) whose
    CKG node ``user_num + p`` has a stored entry of ``graph`` (an ``AttentiveGraph``) towards ``user_num + e`` for some ``e`` of
    every group.  ``groups``: list of non-empty lists of entity ids in ``[0, graph.n - user_num)``.
    Returns ``(positions int32 [len(items)], cand_items int32 [len(items)], n_cand int32 [1])``, all on the device: the first
    ``n_cand`` entries are the passing positions into ``items`` in input order and their item ids (``cand_items`` is 0 after them)."""
    user_num = int(user_num)
    if not 0 <= user_num < graph.n:
        raise ValueError(f"user_num {user_num} outside [0, {graph.n})")
    dev = graph.col_idx.device
    groups = require_groups(groups, graph.n - user_num)
    (items32,) = range_check([("item ids", _ids64(items, "items", dev), graph.n - user_num)], dev)
    return launch_recommend_filter(graph, items32, groups, user_num)


def _group_nodes(groups, user_num: int, dev):
    """Groups of entity ids as a CSR over CKG node ids: (group_ptr int32 [G + 1], group_nodes int32), on ``dev``."""
    gptr = torch.tensor([0] + [len(g) for g in groups], dtype=i64).cumsum(0).to(dtype=i32, device=dev)
    gnodes = torch.tensor([e for g in groups for e in g], dtype=i32).add_(user_num).to(dev)
    return gptr, gnodes


def launch_recommend_filter(graph, items32: torch.Tensor, groups, user_num: int):
    """``recommend_filter`` for int32 ``items32`` and ``groups`` already known to lie in range (no checks, no synchronisation)."""
    lib = _lib.load()
    dev = graph.col_idx.device
    gptr, gnodes = _group_nodes(groups, user_num, dev)
    n = items32.numel()
    positions = torch.empty(n, dtype=i32, device=dev)
    cand = torch.zeros(n, dtype=i32, device=dev)  # entries from n_cand on stay 0, a valid row for recommend_topk_fused's range check
    n_cand = torch.empty(1, dtype=i32, device=dev)
    check(lib.kgat_recommend_filter(_ptr(graph.row_ptr, i32), _ptr(graph.col_idx, i32), graph.n, user_num, _ptr(items32, i32, "items") if n else None,
                                    n, gptr.data_ptr(), gnodes.data_ptr() if gnodes.numel() else None, len(groups), positions.data_ptr() if n else None,
                                    cand.data_ptr() if n else None, n_cand.data_ptr(), _stream()), "recommend_filter")
    return positions, cand, n_cand


def recommend_topk_fused(tables, users: torch.Tensor, cand_items: torch.Tensor, k: int, exclude_ptr=None, exclude_items=None, slices=None,
                         n_cand=None):
    """Top-``k`` of ``cand_items`` for every row of ``users`` in one call, without a score matrix (``kgat_recommend_topk``).
    ``tables``: the propagated layer tables [E0, ..., EL]; ``users`` / ``cand_items``: 1-D table rows, any integer dtype, candidates
    unique; ``n_cand`` (device int32 [1], e.g. from ``recommend_filter``): only the first ``n_cand`` candidates count.
    ``exclude_ptr`` int32 [>= max(users) + 2] / ``exclude_items`` int32: per user row the excluded item ids, ascending.  Scores
    are bit-identical to ``sgemm_nt(gather_concat(...))``; order: score descending (``topk_rows`` key), then candidate index.
    ``slices`` (1 .. 64, None = automatic) splits the candidates over CTAs; it does not change the result.
    Returns ``(items int64 [U, k], scores fp32 [U, k], count int32 [U])`` padded with -1 / -inf after ``count``."""
    k = int(k)
    if not 1 <= k <= 128:
        raise ValueError(f"k must be in [1, 128], got {k}")
    if slices is not None and not 1 <= int(slices) <= 64:
        raise ValueError(f"slices must be in [1, 64], got {slices}")
    if (exclude_ptr is None) != (exclude_items is None):
        raise ValueError("exclude_ptr and exclude_items go together")
    dev = tables[0].device
    rows = tables[0].shape[0]
    users = _ids64(users, "users", dev)
    cand_items = _ids64(cand_items, "cand_items", dev)
    checks = [("user ids", users, rows), ("candidate ids", cand_items, rows)]
    if exclude_ptr is not None:
        if exclude_ptr.dim() != 1 or exclude_ptr.numel() < 2:
            raise ValueError("exclude_ptr must be 1-D with one entry per user row plus one")
        checks.append(("user ids (rows of exclude_ptr)", users, exclude_ptr.numel() - 1))
    users32, cand32 = range_check(checks, dev)[:2] if users.numel() else (users.to(i32), cand_items.to(i32))
    return launch_recommend_topk(tables, users32, cand32, k, exclude_ptr, exclude_items, slices, n_cand)


def launch_recommend_topk(tables, users32: torch.Tensor, cand32: torch.Tensor, k: int, exclude_ptr=None, exclude_items=None, slices=None,
                          n_cand=None):
    """``recommend_topk_fused`` for int32 ids and arguments already known to be valid (no checks, no synchronisation)."""
    lib = _lib.load()
    dev = tables[0].device
    t = _tables(tables)
    U, n = users32.numel(), cand32.numel()
    out_items = torch.empty(U, k, dtype=i64, device=dev)
    out_scores = torch.empty(U, k, dtype=f32, device=dev)
    out_count = torch.empty(U, dtype=i32, device=dev)
    if U == 0:
        return out_items, out_scores, out_count
    s = 0 if slices is None else int(slices)
    ws_bytes = int(lib.kgat_recommend_workspace_bytes(C.byref(t), U, n, k, s))
    if ws_bytes < 0:
        raise KgatLibraryError(f"recommend_topk: tables of width {sum(x.shape[1] for x in tables)} rejected (not multiples of 4, or too wide for shared memory at k = {k})")
    ws = torch.empty(max(ws_bytes, 1), dtype=u8, device=dev)
    check(lib.kgat_recommend_topk(
        C.byref(t), _ptr(users32, i32, "users"), U, _ptr(cand32, i32, "cand_items") if n else None, n,
        None if n_cand is None else _ptr(n_cand, i32, "n_cand"), k,
        None if exclude_ptr is None else _ptr(exclude_ptr, i32, "exclude_ptr"), None if exclude_items is None else _ptr(exclude_items, i32, "exclude_items"),
        s, out_items.data_ptr(), out_scores.data_ptr(), out_count.data_ptr(), ws.data_ptr(), ws_bytes, _stream()), "recommend_topk")
    return out_items, out_scores, out_count


def cap_groups(caps, n_ent: int):
    """``caps`` of ``recommend_capped``, a list of ``(group, cap)`` pairs, as (groups: lists of ints, caps: ints); ValueError for
    more than 128 pairs, an empty group, an entity id outside ``[0, n_ent)``, or a cap that is not an integer >= 0."""
    try:
        pairs = [(list(g), c) for g, c in caps]
    except (TypeError, ValueError):
        raise ValueError("caps must be a list of (group, cap) pairs") from None
    if len(pairs) > 128:
        raise ValueError(f"at most 128 capped groups, got {len(pairs)}")
    groups, values = [], []
    for g, c in pairs:
        if isinstance(c, bool) or (isinstance(c, torch.Tensor) and c.dtype == torch.bool):
            raise ValueError(f"a cap must be an integer >= 0, got {c!r}")
        try:
            c = operator.index(c)
        except TypeError:
            raise ValueError(f"a cap must be an integer >= 0, got {c!r}") from None
        if c < 0:
            raise ValueError(f"a cap must be an integer >= 0, got {c}")
        if len(g) == 0:
            raise ValueError("every group of `caps` must hold at least one entity id")
        g = [int(e) for e in g]
        if any(not 0 <= e < n_ent for e in g):
            raise ValueError(f"entity ids of `caps` must lie in [0, {n_ent})")
        groups.append(g)
        values.append(c)
    return groups, values


def recommend_capped(tables, graph, users: torch.Tensor, cand_items: torch.Tensor, k: int, caps, user_num: int, exclude_ptr=None,
                     exclude_items=None, m=None, slices=None):
    """Top-``k`` of ``cand_items`` for every row of ``users`` with at most ``cap`` problems of each capped group, in one call
    (``kgat_recommend_group_masks`` + ``kgat_recommend_capped_round``).  ``tables``, ``users``, ``cand_items``, ``exclude_*`` and
    ``slices`` as for ``recommend_topk_fused``; ``graph``: the ``AttentiveGraph`` whose rows give group membership (problem ``p``
    is in a group when row ``user_num + p`` stores ``user_num + e`` for some ``e`` of it); ``caps``: list of ``(group, cap)``
    pairs (see ``cap_groups``); ``m`` (``k`` .. 128, None = ``max(k, 64)``): candidates per row and round.
    Each row walks its candidates in ``recommend_topk_fused``'s order and accepts one when all its groups are below their caps,
    until ``k`` are accepted.  Returns ``(items int64 [U, k], scores fp32 [U, k], count int32 [U], rounds)``, padded with
    -1 / -inf after ``count``; neither ``m`` nor ``slices`` changes the result."""
    k = int(k)
    if not 1 <= k <= 128:
        raise ValueError(f"k must be in [1, 128], got {k}")
    if m is not None and not k <= int(m) <= 128:
        raise ValueError(f"m must be in [k, 128] = [{k}, 128], got {m}")
    if slices is not None and not 1 <= int(slices) <= 64:
        raise ValueError(f"slices must be in [1, 64], got {slices}")
    if (exclude_ptr is None) != (exclude_items is None):
        raise ValueError("exclude_ptr and exclude_items go together")
    user_num = int(user_num)
    if not 0 <= user_num < graph.n:
        raise ValueError(f"user_num {user_num} outside [0, {graph.n})")
    groups, values = cap_groups(caps, graph.n - user_num)
    dev = tables[0].device
    rows = tables[0].shape[0]
    users = _ids64(users, "users", dev)
    cand_items = _ids64(cand_items, "cand_items", dev)
    checks = [("user ids", users, rows), ("candidate ids", cand_items, min(rows, graph.n - user_num))]
    if exclude_ptr is not None:
        if exclude_ptr.dim() != 1 or exclude_ptr.numel() < 2:
            raise ValueError("exclude_ptr must be 1-D with one entry per user row plus one")
        checks.append(("user ids (rows of exclude_ptr)", users, exclude_ptr.numel() - 1))
    users32, cand32 = range_check(checks, dev)[:2]
    return launch_recommend_capped(tables, graph, users32, cand32, k, groups, values, user_num, exclude_ptr, exclude_items, m, slices)


def launch_recommend_capped(tables, graph, users32: torch.Tensor, cand32: torch.Tensor, k: int, groups, caps, user_num: int, exclude_ptr=None,
                            exclude_items=None, m=None, slices=None, n_cand=None, active_rows=None):
    """``recommend_capped`` for int32 ids and arguments already known to be valid (``groups`` / ``caps`` from ``cap_groups``);
    ``n_cand`` (device int32 [1], e.g. from ``recommend_filter``): only the first ``n_cand`` candidates count; ``active_rows``: a
    list that receives the number of rows of each round.  No checks; one host synchronisation per round, to read the number
    of rows still active."""
    lib = _lib.load()
    dev = tables[0].device
    t = _tables(tables)
    U, n, G = users32.numel(), cand32.numel(), len(groups)
    m = max(k, 64) if m is None else int(m)
    out_items = torch.empty(U, k, dtype=i64, device=dev)
    out_scores = torch.empty(U, k, dtype=f32, device=dev)
    out_count = torch.empty(U, dtype=i32, device=dev)
    if U == 0:
        return out_items, out_scores, out_count, 0
    s = 0 if slices is None else int(slices)
    ws_bytes = int(lib.kgat_recommend_capped_workspace_bytes(C.byref(t), U, n, G, k, m, s))
    if ws_bytes < 0:
        raise KgatLibraryError(f"recommend_capped: tables of width {sum(x.shape[1] for x in tables)} rejected (not multiples of 4, or too wide for shared memory at m = {m})")
    ws = torch.empty(max(ws_bytes, 1), dtype=u8, device=dev)
    gptr, gnodes = _group_nodes(groups, user_num, dev)
    caps_dev = torch.tensor(caps, dtype=i32).to(dev)
    masks = torch.empty(n, 4, dtype=i32, device=dev)
    n_cand_p = None if n_cand is None else _ptr(n_cand, i32, "n_cand")
    check(lib.kgat_recommend_group_masks(_ptr(graph.row_ptr, i32), _ptr(graph.col_idx, i32), graph.n, user_num, _ptr(cand32, i32, "cand_items") if n else None,
                                         n, n_cand_p, gptr.data_ptr(), gnodes.data_ptr() if G else None, G, masks.data_ptr() if n else None, _stream()),
          "recommend_group_masks")
    ex_p = None if exclude_ptr is None else _ptr(exclude_ptr, i32, "exclude_ptr")
    ex_i = None if exclude_items is None else _ptr(exclude_items, i32, "exclude_items")
    n_next = torch.zeros(1, dtype=i32, device=dev)
    n_active, rounds = U, 0
    while n_active:
        if active_rows is not None:
            active_rows.append(n_active)
        check(lib.kgat_recommend_capped_round(
            C.byref(t), _ptr(users32, i32, "users"), U, _ptr(cand32, i32, "cand_items") if n else None, n, n_cand_p, masks.data_ptr() if n else None,
            caps_dev.data_ptr() if G else None, G, k, m, ex_p, ex_i, s, rounds, n_active, n_next.data_ptr(), out_items.data_ptr(),
            out_scores.data_ptr(), out_count.data_ptr(), ws.data_ptr(), ws_bytes, _stream()), "recommend_capped_round")
        rounds += 1
        n_active = int(n_next.item())
    return out_items, out_scores, out_count, rounds


def duplicate_count(ids: torch.Tensor) -> torch.Tensor:
    """Device scalar: the number of repeated entries of the 1-D ``ids`` (0 when they are unique)."""
    if ids.numel() < 2:
        return torch.zeros((), dtype=i64, device=ids.device)
    return (torch.sort(ids).values.diff() == 0).sum()


def target_rows(target_ptr: torch.Tensor, users: torch.Tensor) -> torch.Tensor:
    """Row pointer (int64 [U + 1], on the device) of the targets of ``users`` (int64) under the CSR pointer ``target_ptr``.  Ids
    outside the pointer's rows are clamped, so this is safe before the range check; the pointer is meaningful after it."""
    cnt = (target_ptr[1:] - target_ptr[:-1]).to(i64)
    out = torch.zeros(users.numel() + 1, dtype=i64, device=users.device)
    if users.numel() and cnt.numel():
        torch.cumsum(cnt[users.clamp(0, cnt.numel() - 1)], 0, out=out[1:])
    return out


def rank_targets(tables, users: torch.Tensor, cand_items, target_ptr: torch.Tensor, target_items: torch.Tensor, exclude_ptr=None,
                 exclude_items=None, slices=None):
    """Exact rank of every target of every row of ``users`` among ``cand_items`` in one call, without a score matrix
    (``kgat_rank_targets``).  ``tables``: the propagated layer tables [E0, ..., EL]; ``users``: 1-D table rows, any integer dtype,
    repeats allowed; ``cand_items``: an int ``n`` (= ``arange(n)``) or 1-D unique table rows, whose order breaks score ties;
    ``target_ptr`` int32 [>= max(users) + 2] / ``target_items`` int32: per user row the targets, ascending;
    ``exclude_ptr`` / ``exclude_items``: per user row the excluded item ids, ascending (an excluded item is not eligible).
    ``rank`` = the number of eligible candidates whose (score, position) key beats the target's, the order of
    ``recommend_topk_fused``; -1 when the target is not an eligible candidate.  ``slices`` (1 .. 64, None = automatic) does not
    change the result.  Returns ``(ptr int64 [U+1], items int64 [M], scores fp32 [M], rank int64 [M], eligible int64 [U])``."""
    if slices is not None and not 1 <= int(slices) <= 64:
        raise ValueError(f"slices must be in [1, 64], got {slices}")
    if (exclude_ptr is None) != (exclude_items is None):
        raise ValueError("exclude_ptr and exclude_items go together")
    if target_ptr.dim() != 1 or target_ptr.numel() < 2:
        raise ValueError("target_ptr must be 1-D with one entry per user row plus one")
    dev = tables[0].device
    rows = tables[0].shape[0]
    users = _ids64(users, "users", dev)
    arange = isinstance(cand_items, int)
    if arange and not 0 <= cand_items <= rows:
        raise ValueError(f"cand_items = {cand_items} must lie in [0, {rows}]")
    cand = torch.arange(cand_items, device=dev) if arange else _ids64(cand_items, "cand_items", dev)
    target_ptr, target_items = target_ptr.to(dev), target_items.to(dev)
    checks = [("user ids", users, rows), ("candidate ids", cand, rows), ("user ids (rows of target_ptr)", users, target_ptr.numel() - 1)]
    if exclude_ptr is not None:
        if exclude_ptr.dim() != 1 or exclude_ptr.numel() < 2:
            raise ValueError("exclude_ptr must be 1-D with one entry per user row plus one")
        checks.append(("user ids (rows of exclude_ptr)", users, exclude_ptr.numel() - 1))
    bad_targets = ((target_items < 0) | (target_items >= rows)).sum()
    out_ptr = target_rows(target_ptr, users)
    got = range_check(checks, dev, flags=[("cand_items holds duplicate ids", duplicate_count(cand)), (f"target ids outside [0, {rows})", bad_targets)],
                      values=[out_ptr[-1]])
    return launch_rank(tables, got[0], got[1], target_ptr, target_items, out_ptr, got[-1], exclude_ptr, exclude_items, slices, arange=arange,
                       n_pos=rows)


def launch_rank(tables, users32: torch.Tensor, cand32: torch.Tensor, target_ptr, target_items, out_ptr, n_targets: int, exclude_ptr=None,
                exclude_items=None, slices=None, arange: bool = False, n_pos: int = 0):
    """``rank_targets`` for int32 ids and arguments already known to be valid (no checks, no synchronisation).  ``out_ptr``
    from ``target_rows`` with ``n_targets = out_ptr[-1]``; ``arange``: ``cand32`` is ``0 .. n - 1``, positions are the ids;
    otherwise an int32 [n_pos] position map is built (every candidate id below ``n_pos``)."""
    lib = _lib.load()
    dev = tables[0].device
    t = _tables(tables)
    U, n, M = users32.numel(), cand32.numel(), int(n_targets)
    items = torch.empty(M, dtype=i64, device=dev)
    scores = torch.empty(M, dtype=f32, device=dev)
    rank = torch.empty(M, dtype=i64, device=dev)
    eligible = torch.empty(U, dtype=i64, device=dev)
    if U == 0:
        return out_ptr, items, scores, rank, eligible
    if exclude_items is not None and exclude_items.numel() == 0:
        exclude_ptr = exclude_items = None  # nothing is excluded
    pos_map = None
    if not arange:
        pos_map = torch.full((max(int(n_pos), 1),), -1, dtype=i32, device=dev)
        pos_map[cand32.long()] = torch.arange(n, dtype=i32, device=dev)
    s = 0 if slices is None else int(slices)
    ws_bytes = int(lib.kgat_rank_workspace_bytes(C.byref(t), U, M))
    if ws_bytes < 0:
        raise KgatLibraryError(f"rank_targets: tables of width {sum(x.shape[1] for x in tables)} rejected (not multiples of 4, or too wide for shared memory)")
    ws = torch.empty(max(ws_bytes, 1), dtype=u8, device=dev)
    check(lib.kgat_rank_targets(
        C.byref(t), _ptr(users32, i32, "users"), U, _ptr(cand32, i32, "cand_items") if n else None, n,
        None if pos_map is None else pos_map.data_ptr(), 0 if pos_map is None else pos_map.numel(), _ptr(target_ptr, i32, "target_ptr"),
        _ptr(target_items, i32, "target_items") if M else None, _ptr(out_ptr, i64, "out_ptr"), M,
        None if exclude_ptr is None else _ptr(exclude_ptr, i32, "exclude_ptr"), None if exclude_items is None else _ptr(exclude_items, i32, "exclude_items"),
        s, items.data_ptr() if M else None, scores.data_ptr() if M else None, rank.data_ptr() if M else None, eligible.data_ptr(), ws.data_ptr(),
        ws_bytes, _stream()), "rank_targets")
    return out_ptr, items, scores, rank, eligible


def _completion_queries(emb, rel_emb, W, heads, rels, tails, candidates, exclude_keys, slices):
    """Shared checks of ``complete_topk`` / ``kg_rank``; the queries sorted by relation (stable) and one read-back of the ranges,
    duplicates and per-relation query counts.  Returns a dict of what the launch needs."""
    if slices is not None and not 1 <= int(slices) <= 64:
        raise ValueError(f"slices must be in [1, 64], got {slices}")
    if emb.dim() != 2 or rel_emb.dim() != 2 or W.dim() != 3 or W.shape != (rel_emb.shape[0], emb.shape[1], rel_emb.shape[1]):
        raise ValueError("emb [N, d], rel_emb [R, k] and W [R, d, k] do not fit together")
    N, R = emb.shape[0], rel_emb.shape[0]
    if not (emb.shape[1] == rel_emb.shape[1] and emb.shape[1] in (32, 64, 128)):
        raise KgatLibraryError(f"complete: TransR widths d = {emb.shape[1]}, k = {rel_emb.shape[1]} unsupported (d = k in 32, 64, 128)")
    dev = emb.device
    heads, rels = _ids64(heads, "heads", dev), _ids64(rels, "relations", dev)
    if heads.numel() != rels.numel() or (tails is not None and tails.numel() != heads.numel()):
        raise ValueError("heads, relations (and tails) differ in length")
    arange = isinstance(candidates, int)
    if arange and not 0 <= candidates <= N:
        raise ValueError(f"candidates = {candidates} must lie in [0, {N}]")
    if not arange and not isinstance(candidates, torch.Tensor):
        raise ValueError("candidates must be an int or a 1-D integer tensor of node ids")
    cand = torch.arange(candidates, device=dev) if arange else _ids64(candidates, "candidates", dev)
    if exclude_keys is not None and (exclude_keys.dim() != 1 or exclude_keys.dtype != i64 or exclude_keys.device != dev):
        raise ValueError("exclude must hold int64 keys on the parameters' device")
    order = torch.sort(rels, stable=True).indices
    counts = torch.zeros(R, dtype=i64, device=dev).index_add_(0, rels.clamp(0, R - 1), torch.ones_like(rels))
    checks = [("head ids", heads, N), ("relation ids", rels, R), ("candidate ids", cand, N)]
    if tails is not None:
        checks.append(("tail ids", _ids64(tails, "tails", dev), N))
    got = range_check(checks, dev, flags=[("candidates hold duplicate ids", duplicate_count(cand))], values=list(counts))
    ids = [got[j][order].contiguous() if j != 2 else None for j in range(len(checks))]  # the queries in sorted order
    counts = got[len(checks) :]
    seg_rel = [r for r in range(R) if counts[r] > 0]
    seg_ptr = [0]
    for r in seg_rel:
        seg_ptr.append(seg_ptr[-1] + counts[r])
    pos_map = None
    if tails is not None and not arange:
        pos_map = torch.full((N,), -1, dtype=i32, device=dev)
        pos_map[got[2].long()] = torch.arange(got[2].numel(), dtype=i32, device=dev)
    ex = exclude_keys if exclude_keys is not None and exclude_keys.numel() else None
    return dict(N=N, R=R, d=emb.shape[1], kdim=rel_emb.shape[1], heads=ids[0], rels=ids[1], cand=got[2], tails=ids[3] if tails is not None else None,
                q_out=order.to(i32), seg_rel=torch.tensor(seg_rel, dtype=i32, device=dev), seg_ptr=seg_ptr,
                n_tiles=sum((seg_ptr[g + 1] - seg_ptr[g] + 63) // 64 for g in range(len(seg_rel))), pos_map=pos_map, ex=ex,
                slices=0 if slices is None else int(slices))


def _completion_workspace(q, k: int, count: bool):
    lib = _lib.load()
    ws_bytes = int(lib.kgat_complete_workspace_bytes(q["d"], q["kdim"], q["heads"].numel(), q["n_tiles"], q["cand"].numel(), len(q["seg_ptr"]) - 1,
                                                     k, q["slices"], int(count)))
    if ws_bytes < 0:
        raise KgatLibraryError(f"complete: width {q['kdim']} rejected (too wide for shared memory at k = {k})")
    return torch.empty(max(ws_bytes, 1), dtype=u8, device=q["heads"].device), ws_bytes


def complete_topk(emb, rel_emb, W, heads, rels, candidates, k: int, exclude_keys=None, slices=None):
    """Top-``k`` tails of the queries ``(heads[q], rels[q], ?)`` among ``candidates`` under the TransR parameters, lowest energy
    first, without an energy matrix (``kgat_complete_topk``).  ``emb`` [N, d] / ``rel_emb`` [R, k] / ``W`` [R, d, k]: the
    entity table, relation embeddings and projection matrices; ``heads`` / ``rels``: 1-D ids, any integer dtype;
    ``candidates``: an int ``n`` (= ``arange(n)``) or 1-D unique node ids, whose order breaks energy ties;
    ``exclude_keys``: ``metrics.TripleSet.keys`` of known triples (not returned).  ``slices`` (1 .. 64, None = automatic) does
    not change the result.  One host synchronisation.  Returns ``(tails int64 [Q, k], energy fp32 [Q, k], count int32 [Q])``
    padded with -1 / +inf after ``count``."""
    k = int(k)
    if not 1 <= k <= 128:
        raise ValueError(f"k must be in [1, 128], got {k}")
    q = _completion_queries(emb, rel_emb, W, heads, rels, None, candidates, exclude_keys, slices)
    dev, Q = emb.device, q["heads"].numel()
    tails = torch.empty(Q, k, dtype=i64, device=dev)
    energy = torch.empty(Q, k, dtype=f32, device=dev)
    count = torch.empty(Q, dtype=i32, device=dev)
    if Q == 0:
        return tails, energy, count
    ws, ws_bytes = _completion_workspace(q, k, False)
    seg_ptr = (C.c_int64 * len(q["seg_ptr"]))(*q["seg_ptr"])
    n = q["cand"].numel()
    check(_lib.load().kgat_complete_topk(
        _ptr(emb, f32, "emb"), _ptr(rel_emb, f32, "rel_emb"), _ptr(W, f32, "W"), q["d"], q["kdim"], q["N"], q["R"], q["heads"].data_ptr(),
        q["rels"].data_ptr(), q["q_out"].data_ptr(), Q, seg_ptr, q["seg_rel"].data_ptr(), len(q["seg_ptr"]) - 1, q["cand"].data_ptr() if n else None,
        n, None if q["ex"] is None else q["ex"].data_ptr(), 0 if q["ex"] is None else q["ex"].numel(), k, q["slices"], tails.data_ptr(),
        energy.data_ptr(), count.data_ptr(), ws.data_ptr(), ws_bytes, _stream()), "complete_topk")
    return tails, energy, count


def kg_rank(emb, rel_emb, W, heads, rels, tails, candidates, exclude_keys=None, slices=None):
    """Filtered rank of the tail of every triple ``(heads[q], rels[q], tails[q])`` among ``candidates`` (``kgat_complete_rank``):
    ``rank`` = the eligible candidates other than the target whose (energy, position) key beats the target's, -1 when the
    target is not a candidate; the target stays eligible when its own triple is in ``exclude_keys``.  Arguments as for
    ``complete_topk``.  One host synchronisation.  Returns ``(energy fp32 [Q], rank int64 [Q], eligible int64 [Q])``."""
    q = _completion_queries(emb, rel_emb, W, heads, rels, tails, candidates, exclude_keys, slices)
    dev, Q = emb.device, q["heads"].numel()
    energy = torch.empty(Q, dtype=f32, device=dev)
    rank = torch.empty(Q, dtype=i64, device=dev)
    eligible = torch.empty(Q, dtype=i64, device=dev)
    if Q == 0:
        return energy, rank, eligible
    ws, ws_bytes = _completion_workspace(q, 1, True)
    seg_ptr = (C.c_int64 * len(q["seg_ptr"]))(*q["seg_ptr"])
    n = q["cand"].numel()
    check(_lib.load().kgat_complete_rank(
        _ptr(emb, f32, "emb"), _ptr(rel_emb, f32, "rel_emb"), _ptr(W, f32, "W"), q["d"], q["kdim"], q["N"], q["R"], q["heads"].data_ptr(),
        q["rels"].data_ptr(), q["tails"].data_ptr(), q["q_out"].data_ptr(), Q, seg_ptr, q["seg_rel"].data_ptr(), len(q["seg_ptr"]) - 1,
        q["cand"].data_ptr() if n else None, n, None if q["pos_map"] is None else q["pos_map"].data_ptr(),
        None if q["ex"] is None else q["ex"].data_ptr(), 0 if q["ex"] is None else q["ex"].numel(), q["slices"], energy.data_ptr(),
        rank.data_ptr(), eligible.data_ptr(), ws.data_ptr(), ws_bytes, _stream()), "kg_rank")
    return energy, rank, eligible


# ----------------------------------------------------------------------------------------------
# K11 Adam
# ----------------------------------------------------------------------------------------------


def adam_set_hyper(step: int, lr, beta1, beta2, eps, hyper: torch.Tensor):
    lib = _lib.load()
    check(lib.kgat_adam_set_hyper(int(step), float(lr), float(beta1), float(beta2), float(eps), _ptr(hyper, f32), _stream()), "adam_set_hyper")


def adam_advance(step_dev: torch.Tensor, lr, beta1, beta2, eps, hyper: torch.Tensor):
    lib = _lib.load()
    check(lib.kgat_adam_advance(_ptr(step_dev, i64), float(lr), float(beta1), float(beta2), float(eps), _ptr(hyper, f32), _stream()), "adam_advance")


@_timed("adam_apply")
def adam_apply(params, grads, exp_avgs, exp_avg_sqs, hyper: torch.Tensor, peer_param0=None, row_slot0=None):
    """``peer_param0``: int64 device tensor of pointers; the updated ``params[0]`` is mirrored behind each of them.
    ``row_slot0``: int32 [rows of params[0]]; ``grads[0]`` then holds compact rows (ops.transr_claim_rows)."""
    lib = _lib.load()
    n = len(params)
    for start in range(0, n, _lib.KGAT_MAX_TENSORS):
        t = AdamTensorsT()
        chunk = range(start, min(n, start + _lib.KGAT_MAX_TENSORS))
        t.n_tensors = len(chunk)
        for j, i in enumerate(chunk):
            t.param[j] = _ptr(params[i], f32, "param")
            t.grad[j] = _ptr(grads[i], f32, "grad")
            if grads[i].numel() != params[i].numel() and not (i == 0 and row_slot0 is not None):
                raise KgatLibraryError("adam_apply: gradient / parameter size mismatch")
            t.exp_avg[j] = _ptr(exp_avgs[i], f32, "exp_avg")
            t.exp_avg_sq[j] = _ptr(exp_avg_sqs[i], f32, "exp_avg_sq")
            t.numel[j] = params[i].numel()
        if start == 0 and peer_param0 is not None:
            t.peer_param0, t.n_peers = _ptr(peer_param0, i64), peer_param0.numel()
        if start == 0 and row_slot0 is not None:
            if row_slot0.numel() * params[0].shape[-1] != params[0].numel():
                raise KgatLibraryError("adam_apply: row_slot0 needs one entry per row of params[0]")
            t.row_slot0, t.row_dim0 = _ptr(row_slot0, i32), params[0].shape[-1]
        check(lib.kgat_adam_apply(C.byref(t), _ptr(hyper, f32), _stream()), "adam_apply")


@_timed("adam_rolling_prepare")
def adam_rolling_prepare(heads, pos_t, neg_t, row_slot, g_rows, zero_a, zero_b, param, exp_avg, exp_avg_sq, row_step, cur_step_dev, s0, table, hyper,
                         advanced: bool = False, prev_ids=None, dense=None):
    """Rolling-window KG Adam, before the forward: claim compact gradient rows, zero ``g_rows`` / ``zero_a`` / ``zero_b``, bring
    the batch rows of ``param`` up to the steps done so far."""
    lib = _lib.load()
    if g_rows.numel() < 3 * heads.numel() * param.shape[1]:
        raise KgatLibraryError("adam_rolling_prepare: g_rows needs 3 * batch * d floats")
    check(lib.kgat_adam_rolling_prepare(_ptr(heads, i64), _ptr(pos_t, i64), _ptr(neg_t, i64), heads.numel(), param.shape[1], _ptr(row_slot, i32),
                                        _ptr(g_rows, f32), _ptr(zero_a, f32) if zero_a is not None else None, zero_a.numel() if zero_a is not None else 0,
                                        _ptr(zero_b, f32) if zero_b is not None else None, zero_b.numel() if zero_b is not None else 0,
                                        _ptr(param, f32), _ptr(exp_avg, f32), _ptr(exp_avg_sq, f32), _ptr(row_step, i32), _ptr(cur_step_dev, i64),
                                        int(bool(advanced)), _ptr(s0, i64), _ptr(table, f32), _ptr(hyper, f32),
                                        *((_ptr(prev_ids[0], i64), _ptr(prev_ids[1], i64), _ptr(prev_ids[2], i64), _ptr(dense, f32, "dense", True),
                                           dense.stride(0)) if dense is not None else (None, None, None, None, 0)),
                                        _stream()), "adam_rolling_prepare")


@_timed("transr_step_claimed")
def transr_step_claimed(emb, rel_emb, W, heads, rels, pos_t, neg_t, reg, loss, loss_sum, scratch, row_slot, g_rows, g_rel, g_W, publish=None):
    """``transr_step`` for rows claimed (and buffers zeroed) by ``adam_rolling_prepare``."""
    lib = _lib.load()
    if g_rows.numel() < 3 * heads.numel() * emb.shape[1] or scratch.numel() < transr_scratch_numel(heads.numel(), rel_emb.shape[1]):
        raise KgatLibraryError("transr_step_claimed: g_rows needs 3 * batch * d floats, scratch transr_scratch_numel(batch, k)")
    check(lib.kgat_transr_step_claimed(_ptr(emb, f32), _ptr(rel_emb, f32), _ptr(W, f32), emb.shape[1], rel_emb.shape[1], _ptr(heads, i64),
                                       _ptr(rels, i64), _ptr(pos_t, i64), _ptr(neg_t, i64), heads.numel(), float(reg), _ptr(loss, f32),
                                       _ptr(loss_sum, f32) if loss_sum is not None else None, _ptr(scratch, f32), _ptr(row_slot, i32),
                                       _ptr(g_rows, f32), _ptr(g_rel, f32), _ptr(g_W, f32), C.byref(publish) if publish is not None else None,
                                       _stream()), "transr_step_claimed")


@_timed("adam_rolling_apply")
def adam_rolling_apply(heads, pos_t, neg_t, row_slot, g_rows, param, exp_avg, exp_avg_sq, row_step, window, dense_params, dense_grads,
                       dense_exp_avgs, dense_exp_avg_sqs, cur_step_dev, s0, table, hyper, parts: int = 3):
    """Rolling-window KG Adam, after ``adam_advance``: claimed rows take their gradient, the small dense tensors a plain step, and the
    window's current slice of ``param`` is replayed (zero-gradient updates) to the previous step."""
    lib = _lib.load()
    n = len(dense_params)
    if n > _lib.KGAT_MAX_TENSORS:
        raise KgatLibraryError("adam_rolling_apply: too many dense tensors")
    t = AdamTensorsT()
    t.n_tensors = n
    for j in range(n):
        if dense_grads[j].numel() != dense_params[j].numel():
            raise KgatLibraryError("adam_rolling_apply: gradient / parameter size mismatch")
        t.param[j] = _ptr(dense_params[j], f32, "param")
        t.grad[j] = _ptr(dense_grads[j], f32, "grad")
        t.exp_avg[j] = _ptr(dense_exp_avgs[j], f32, "exp_avg")
        t.exp_avg_sq[j] = _ptr(dense_exp_avg_sqs[j], f32, "exp_avg_sq")
        t.numel[j] = dense_params[j].numel()
    check(lib.kgat_adam_rolling_apply(_ptr(heads, i64), _ptr(pos_t, i64), _ptr(neg_t, i64), heads.numel(), param.shape[1], _ptr(row_slot, i32),
                                      _ptr(g_rows, f32), _ptr(param, f32), _ptr(exp_avg, f32), _ptr(exp_avg_sq, f32), _ptr(row_step, i32),
                                      param.shape[0], int(window), C.byref(t), int(parts), _ptr(cur_step_dev, i64), _ptr(s0, i64), _ptr(table, f32),
                                      _ptr(hyper, f32), _stream()), "adam_rolling_apply")


def selftest_adam_arith(m, v, inv_sqrt_bc2: float, eps: float):
    """(mismatches vs the IEEE builtins, elements on the fast sequences) for q = m / (sqrt(v) * inv_sqrt_bc2 + eps)."""
    lib = _lib.load()
    counts = torch.zeros(2, dtype=torch.int32, device=m.device)
    check(lib.kgat_selftest_adam_arith(_ptr(m, f32), _ptr(v, f32), m.numel(), float(inv_sqrt_bc2), float(eps), _ptr(counts, i32), _stream()),
          "selftest_adam_arith")
    c = counts.tolist()
    return c[0], c[1]


def adam_hyper_table(s0_dev: torch.Tensor, n_steps: int, lr, beta1, beta2, table: torch.Tensor):
    lib = _lib.load()
    if table.numel() < 2 * n_steps:
        raise KgatLibraryError("adam_hyper_table: table needs 2*n_steps floats")
    check(lib.kgat_adam_hyper_table(_ptr(s0_dev, i64), int(n_steps), float(lr), float(beta1), float(beta2), _ptr(table, f32), _stream()), "adam_hyper_table")


@_timed("adam_lazy_catchup")
def adam_lazy_catchup(param, exp_avg, exp_avg_sq, row_step, ids, cur_step_dev, s0, table, hyper):
    lib = _lib.load()
    check(lib.kgat_adam_lazy_catchup(_ptr(param, f32), _ptr(exp_avg, f32), _ptr(exp_avg_sq, f32), _ptr(row_step, i32), _ptr(ids, i64),
                                     ids.numel(), param.shape[1], _ptr(cur_step_dev, i64), _ptr(s0, i64), _ptr(table, f32), _ptr(hyper, f32),
                                     _stream()), "adam_lazy_catchup")


@_timed("adam_sparse_rows")
def adam_sparse_rows(param, grad, exp_avg, exp_avg_sq, row_step, ids, cur_step_dev, s0, hyper):
    lib = _lib.load()
    check(lib.kgat_adam_sparse_rows(_ptr(param, f32), _ptr(grad, f32), _ptr(exp_avg, f32), _ptr(exp_avg_sq, f32), _ptr(row_step, i32),
                                    _ptr(ids, i64), ids.numel(), param.shape[1], _ptr(cur_step_dev, i64), _ptr(s0, i64), _ptr(hyper, f32),
                                    _stream()), "adam_sparse_rows")


def adam_lazy_flush(param, exp_avg, exp_avg_sq, row_step, cur_step_dev, s0, table, hyper):
    lib = _lib.load()
    check(lib.kgat_adam_lazy_flush(_ptr(param, f32), _ptr(exp_avg, f32), _ptr(exp_avg_sq, f32), _ptr(row_step, i32), param.shape[0],
                                   param.shape[1], _ptr(cur_step_dev, i64), _ptr(s0, i64), _ptr(table, f32), _ptr(hyper, f32), _stream()),
          "adam_lazy_flush")


def publish_args(serial_dev: torch.Tensor, ring_pinned: torch.Tensor):
    """kgat_publish_t for the ``publish=`` argument of bpr_forward / transr_step / transr_step_claimed (keep it alive with the
    tensors: the loss kernel itself then writes (serial, loss) into the pinned ring, no launch of its own)."""
    if ring_pinned.is_cuda or not ring_pinned.is_pinned() or ring_pinned.dtype != i64:
        raise KgatLibraryError("publish_args: the ring must be a pinned int64 host tensor")
    p = _lib.PublishT()
    p.serial_dev, p.ring_host_mapped, p.n_slots = _ptr(serial_dev, i64), ring_pinned.data_ptr(), ring_pinned.numel()
    return p


def publish_loss(loss: torch.Tensor, serial_dev: torch.Tensor, ring_pinned: torch.Tensor):
    """ring[s % len] = (s << 32) | bits(loss) with s = ++serial_dev, written by the GPU into pinned host memory (the pointer
    of a pinned allocation is device-visible under unified addressing)."""
    lib = _lib.load()
    if ring_pinned.is_cuda or not ring_pinned.is_pinned() or ring_pinned.dtype != i64:
        raise KgatLibraryError("publish_loss: the ring must be a pinned int64 host tensor")
    check(lib.kgat_publish_loss(_ptr(loss, f32), _ptr(serial_dev, i64), ring_pinned.data_ptr(), ring_pinned.numel(), _stream()), "publish_loss")


def sample_cf_batch(user_ptr, user_items, active_users, item_num: int, seed: int, step_dev, out):
    """out: int64 [3, B] <- (users, pos, neg), drawn on the device (csrc/sampler.cu)."""
    lib = _lib.load()
    check(lib.kgat_sample_cf_batch(_ptr(user_ptr, i32), _ptr(user_items, i32), _ptr(active_users, i32), active_users.numel(), int(item_num),
                                   out.shape[1], int(seed), _ptr(step_dev, i64), _ptr(out, i64), _stream()), "sample_cf_batch")
    return out


def sample_kg_batch(head_ptr, edge_rel, edge_tail, active_heads, node_num: int, seed: int, step_dev, out):
    """out: int64 [4, B] <- (heads, rels, pos tails, neg tails), drawn on the device."""
    lib = _lib.load()
    check(lib.kgat_sample_kg_batch(_ptr(head_ptr, i32), _ptr(edge_rel, i32), _ptr(edge_tail, i32), _ptr(active_heads, i32),
                                   active_heads.numel(), int(node_num), out.shape[1], int(seed), _ptr(step_dev, i64), _ptr(out, i64),
                                   _stream()), "sample_kg_batch")
    return out

"""The attentive SpMM (csrc/spmm.cu) and the needed-row frontier (csrc/frontier.cu) against float64 references, on every route
and across the sizes at which their code switches.

Two references, both computed on the host with scipy / numpy from the CSR the test built:

* **Exact.**  X and Z hold integers in [-8, 8], edge weights are +-2^-k (k = 0..3).  Every product and partial sum is then a
  multiple of 1/8 below 2^21 in magnitude (rows have fewer than 2^18 edges), so fp32 gives the exact result in any summation
  order -- the atomic scatter kernel's included -- and the kernel output must equal the float64 product cast to fp32 bit for
  bit.  One dropped, duplicated or misrouted edge, a partial counted twice or left stale, or a wrong addend row fails.
* **Rounding bound.**  Gaussian X and Z; attention-like weights (positive, rows summing to 1, Zipf row lengths) for A and
  signed Gaussian weights for A^T.  Per element ``|y - ref| <= 1.01 (L + 2) 2^-24 (sum_k |a_k x_k| + |z|)`` with L the row's
  length: true for any summation order, so it needs no measurement to set.

Routes: ``AttentiveGraph.matmul`` / ``matmul_t`` plain (task kernel), with a row mask (masked task kernel), row + edge mask
(masked task kernel), row list (rows kernel) with and without an edge mask, edge mask alone (rows kernel, dense output);
``ops.spmm`` with a plan from ``graph.make_plan`` over a row range in the sharded layout (full X, ``out`` a row slice of a
larger table); ``ops.spmm_scatter_rows``.  d = 16, 32, 64, 128 on every route, the generic kernel at d = 4 .. 256, chunk = 8
and 256, contiguous and strided X / Y / Z, with and without an addend.  Edge-masked routes read NaN from every dead source and
addend row.  The "big" graph has more tasks and listed rows than one pass of the rows and scatter kernels' grids covers; the
"small" one fewer.  The 4 GiB case crosses the 32-bit offset, ``WIDE`` and shared-memory edge-bitmap thresholds.

``KGAT_SPMM_U``, ``KGAT_SPMM_CTAS`` and ``KGAT_EXPAND_PLAIN`` are read once per process: the d = 64 and 128 cases, the
threshold cases and the frontier cases run again in a child process under ``KGAT_SPMM_U=4 KGAT_SPMM_CTAS=6
KGAT_EXPAND_PLAIN=1``.

Measured maxima of |y - ref| / bound on a B200 (1,000 W), default instances (U = 8 at d = 64, five CTAs per SM), over both
graphs and both chunks, for d = 16 / 32 / 64 / 128:
  plain, row mask, row list, plan (sharded layout)   A: 0.53 / 0.64 / 0.64 / 0.64   A^T: 0.56 / 0.64 / 0.60 / 0.60
  edge-masked (row + edge, list + edge, edge only)   A: 0.51 / 0.51 / 0.54 / 0.52   A^T: 0.50 / 0.55 / 0.58 / 0.56
  scatter (A^T)                                          0.61 / 0.60 / 0.63 / 0.60
The largest ratios are on the shortest rows, where one or two roundings already use most of the (L + 2) units.  The
module, its child process included, runs in about two minutes on one B200.
"""

from __future__ import annotations

import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import scipy.sparse as sp
import torch

from conftest import elem_err

ROOT = Path(__file__).resolve().parents[1]

pytestmark = pytest.mark.gpu

IN_CHILD = os.environ.get("KGAT_SPMM_TEST_CHILD") == "1"
CHILD_ENV = {"KGAT_SPMM_U": "4", "KGAT_SPMM_CTAS": "6", "KGAT_EXPAND_PLAIN": "1", "KGAT_SPMM_TEST_CHILD": "1"}
DIMS = [16, 32, 64, 128]
GENERIC_DIMS = [4, 8, 12, 48, 96, 132, 252, 256]
CHUNKS = [8, 256]
SIZES = {"small": 4096, "big": 24000}
ROUTES = ["plain", "row_mask", "row_edge", "rows", "rows_edge", "edge", "plan", "plan_rows", "scatter"]
EDGE_ROUTES = ("row_edge", "rows_edge", "edge")
# row lengths every graph holds: 0, 1, EPI +- 1 for EPI = 4, 8, 16, 31..33, 63..65, chunk - 1 .. chunk + 1, 2 chunk, 2 chunk + 1
SPECIAL_LENS = [0, 1, 3, 4, 5, 7, 8, 9, 15, 16, 17, 31, 32, 33, 63, 64, 65, 255, 256, 257, 512, 513]
# rows of four 32-edge batches with these live-edge counts under the edge mask (0, 1, EPI +- 1 live edges: the padding path)
LIVE_BATCHES = [(0, 1, 3, 4), (5, 7, 8, 9), (15, 16, 17, 32), (31, 2, 0, 1)]
HEAVY_ROWS = (1000, 1001, 1002)  # adjacent heavy rows (finish_heavy_row finds its row by binary search)
HUB_COL = 7  # a column in > 32 chunks of A^T at chunk 256 (big graph)
SENTINEL = 1234.5
RATIOS: dict = {}  # (route, d, direction) -> largest |y - ref| / bound seen


def epi(d: int) -> int:
    """Edges per unrolled step of the templated kernels: (32 / (d / 4)) * U."""
    u = {16: 2, 32: 4, 64: 4 if os.environ.get("KGAT_SPMM_U") == "4" else 8, 128: 4}[d]
    return 32 // (d // 4) * u


@pytest.fixture(scope="module")
def kb():
    if not torch.cuda.is_available():
        pytest.skip("needs CUDA")
    import kgat_b200

    kgat_b200._lib.load()
    return kgat_b200


@pytest.fixture(scope="module")
def sms(kb):
    return torch.cuda.get_device_properties(0).multi_processor_count


def _bits(mask: np.ndarray, n_bits: int | None = None) -> torch.Tensor:
    """bool [n] -> int32 bitmap of ceil(n_bits / 32) words on the device (bit i of word i >> 5)."""
    words = ((n_bits or mask.size) + 31) // 32
    pad = np.zeros(words * 32, dtype=bool)
    pad[: mask.size] = mask
    return torch.from_numpy(np.packbits(pad, bitorder="little").view(np.int32).copy()).cuda()


def exact_weights(rng, m: int) -> np.ndarray:
    return (rng.choice([-1.0, 1.0], m) * 2.0 ** -rng.integers(0, 4, m)).astype(np.float32)


def attention_weights(rng, indptr: np.ndarray) -> np.ndarray:
    lens = np.diff(indptr)
    row = np.repeat(np.arange(lens.size), lens)
    w = rng.random(row.size) + 0.05
    return (w / np.bincount(row, weights=w, minlength=lens.size)[row]).astype(np.float32)


def structure(size: str):
    """Host CSR (row_ptr int64 [n + 1], col int32) of a square n x n graph and the live set of its edge mask.
    Row 0 and row n - 1 are heavy at both chunks, rows 1000-1002 are adjacent heavy rows, rows 10.. hold SPECIAL_LENS, rows 40..
    the LIVE_BATCHES compositions; the other rows have Zipf lengths (many empty).  Columns 0, n - 1, 500, 501 and HUB_COL are
    popular, so A^T has heavy rows at both ends, adjacent ones and (big graph) one of more than 32 chunks of 256."""
    n = SIZES[size]
    rng = np.random.default_rng(n)
    live = rng.random(n) < 0.5
    hub = 33 * 256 + 5 if size == "big" else 3000
    fixed = {0: hub, n - 1: 513, HEAVY_ROWS[0]: 300, HEAVY_ROWS[1]: 257, HEAVY_ROWS[2]: 600}
    fixed.update({10 + i: k for i, k in enumerate(SPECIAL_LENS)})
    keys = [np.int64(r) * n + rng.choice(n, k, replace=False) for r, k in fixed.items()]
    for i, comp in enumerate(LIVE_BATCHES):  # batch q draws from the q-th quarter of the columns, so it is the q-th 32 of the row
        for q, m in enumerate(comp):
            idx = np.arange(q * n // 4, (q + 1) * n // 4)
            keys.append(np.int64(40 + i) * n + rng.choice(idx[live[idx]], m, replace=False))
            keys.append(np.int64(40 + i) * n + rng.choice(idx[~live[idx]], 32 - m, replace=False))
    special = list(fixed) + [40 + i for i in range(len(LIVE_BATCHES))]
    bulk = np.setdiff1d(np.arange(n), special)
    br = np.repeat(bulk, np.minimum(rng.zipf(2.0, bulk.size) - 1, 200))
    bc = rng.integers(0, n, br.size)
    for c, k in ((HUB_COL, 9000 if size == "big" else 3000), (0, 600), (n - 1, 600), (500, 300), (501, 300)):
        pick = rng.choice(bulk, min(k, bulk.size), replace=False)
        br, bc = np.concatenate([br, pick]), np.concatenate([bc, np.full(pick.size, c)])
    keys.append(np.unique(br.astype(np.int64) * n + bc))
    keys = np.sort(np.concatenate(keys))
    assert np.unique(keys).size == keys.size
    rows, cols = keys // n, (keys % n).astype(np.int32)
    row_ptr = np.concatenate([[0], np.cumsum(np.bincount(rows, minlength=n))]).astype(np.int64)
    return row_ptr, cols, live


@pytest.fixture(scope="module")
def graphs(kb, sms):
    """(size, chunk) -> (AttentiveGraph, host CSR of A, live set, row mask).  Asserts the shapes the module docstring promises."""
    from kgat_b200.graph import AttentiveGraph

    out = {}
    for size, n in SIZES.items():
        row_ptr, cols, live = structure(size)
        lens = np.diff(row_ptr)
        A = sp.csr_matrix((np.ones(cols.size), cols, row_ptr), shape=(n, n))
        At = A.T.tocsr()
        t_lens = np.diff(At.indptr)
        assert set(SPECIAL_LENS) <= set(lens.tolist()) and (lens == 0).sum() > 100
        for d_ in DIMS:
            assert {epi(d_) - 1, epi(d_), epi(d_) + 1} <= set(lens.tolist())
        for i, comp in enumerate(LIVE_BATCHES):
            c = cols[row_ptr[40 + i] : row_ptr[41 + i]]
            assert [int(live[c[32 * q : 32 * q + 32]].sum()) for q in range(4)] == list(comp)
        rng = np.random.default_rng(n + 1)
        rmask = rng.random(n) < (0.9 if size == "big" else 0.5)
        rmask[[0, n - 1, HEAVY_ROWS[0], HEAVY_ROWS[2]] + list(range(10, 44))] = True
        rmask[[HEAVY_ROWS[1], 5, 6]] = False  # a heavy row and some others outside the row mask
        for chunk in CHUNKS:
            for ln in (lens, t_lens):  # heavy rows at row 0, row n - 1 and adjacent ids, in both directions
                assert ln[0] > chunk and ln[n - 1] > chunk
            assert all(lens[r] > chunk for r in HEAVY_ROWS) and t_lens[500] > chunk and t_lens[501] > chunk
            d = torch.from_numpy
            g = AttentiveGraph(n, d(row_ptr.astype(np.int32)).cuda(), d(cols).cuda(), torch.zeros(cols.size, device="cuda"), chunk=chunk)
            assert torch.equal(g.t_ptr.cpu(), d(At.indptr.astype(np.int32))) and torch.equal(g.t_idx.cpu(), d(At.indices.astype(np.int32)))
            warps = sms * 8  # 256-thread CTAs of the rows kernel: sms * 5 (or 6) of them, the scatter kernel sms * 8
            if size == "big":
                assert g.plan.n_tasks >= 20000 and g.t_plan.n_tasks >= 20000 and g.plan.n_tasks > 6 * warps
                assert rmask.sum() >= 20000 and rmask.sum() > 8 * warps
                if chunk == 256:
                    assert lens[0] > 32 * chunk and t_lens[HUB_COL] > 32 * chunk
            elif chunk == 256:
                assert g.plan.n_tasks < 5 * warps and g.t_plan.n_tasks < 5 * warps
            out[(size, chunk)] = (g, A, live, rmask)
    return out


def _direction(g, A: sp.csr_matrix, t: bool):
    """(matmul method, host CSR of the operator, plan, col_idx, vals) of A (t = False) or A^T."""
    if t:
        return g.matmul_t, A.T.tocsr(), g.t_plan, g.t_idx, g.t_vals
    return g.matmul, A, g.plan, g.col_idx, g.vals


def _counters_zero(*plans):
    for p in plans:
        if p.n_heavy:
            assert int(p.heavy[:, 3].abs().max()) == 0, "heavy-row arrival counters not back at 0"


def _table(rows: int, d: int, strided: bool, fill=None, values=None) -> torch.Tensor:
    """[rows, d] on the device, or a column slice [:, 4:4 + d] of a [rows, d + 8] table when strided (the other columns hold
    SENTINEL)."""
    if not strided:
        t = torch.full((rows, d), SENTINEL, device="cuda")
        if values is not None:
            t.copy_(values)
        return t
    w = torch.full((rows, d + 8), SENTINEL, device="cuda")
    if values is not None:
        w[:, 4 : 4 + d] = values
    return w[:, 4 : 4 + d]


def run_route(route: str, g, A: sp.csr_matrix, t: bool, live, rmask, x64, z64, strided: bool):
    """Launch one route; returns (y float64 [m, d] on the host over the output rows, reference float64, sum |a x| + |z|,
    row lengths, rows written (bool)).  Dead rows of X and Z (outside the edge mask) hold NaN on the edge-masked routes, the
    unlisted rows of G and Z on the scatter route."""
    from kgat_b200 import ops
    from kgat_b200.graph import make_plan

    n = g.n
    d = x64.shape[1]
    mm, M, plan, col, vals = _direction(g, A, t)
    edge = route in EDGE_ROUTES
    xin, zin = x64.copy(), None if z64 is None else z64.copy()
    if edge:
        xin[~live] = np.nan
        if zin is not None:
            zin[~live] = np.nan
    if route == "scatter":
        M = A.T.tocsr()
        xin[~rmask] = np.nan
        if zin is not None:
            zin[~rmask] = np.nan
    x = _table(n, d, strided, values=torch.from_numpy(xin).float().cuda())
    z = None if zin is None else _table(n, d, strided, values=torch.from_numpy(zin).float().cuda())
    listed = np.flatnonzero(rmask).astype(np.int32)
    rows = torch.from_numpy(np.concatenate([listed, np.flatnonzero(~rmask).astype(np.int32)])).cuda()  # unlisted ids past the count
    cnt = torch.tensor([listed.size], dtype=torch.int32, device="cuda")
    rb, eb = _bits(rmask), _bits(live)
    r0, r1 = 960, n  # the sharded layout: the plan covers rows [r0, r1), out is big[r0:r1]
    m_rows = n
    if route in ("plan", "plan_rows"):
        sub = M[r0:r1]
        ptr = torch.from_numpy(sub.indptr.astype(np.int32)).cuda()
        plan = make_plan(ptr)
        scol = torch.from_numpy(sub.indices.astype(np.int32)).cuda()
        svals = vals[int(M.indptr[r0]) : int(M.indptr[r1])]
        big = _table(n + 40, d, strided)
        out = big[r0:r1]
        zs = None if z is None else z[r0:r1]
        partials = torch.empty(max(plan.n_partials, 1) * d, device="cuda")
        kw = {}
        if route == "plan_rows":
            loc = rmask[r0:r1]
            ll = np.flatnonzero(loc).astype(np.int32)
            kw = dict(row_mask=_bits(loc, max(n, r1 - r0)), rows=torch.from_numpy(ll).cuda(),
                      n_rows_dev=torch.tensor([ll.size], dtype=torch.int32, device="cuda"))
        ops.spmm(plan, scol, svals, x, out, zs, partials, **kw)
        _counters_zero(plan)
        outside = torch.cat([big[:r0], big[r1:]])
        assert bool((outside == SENTINEL).all()), "rows outside the plan's range were written"
        M, m_rows, written = sub, r1 - r0, (rmask[r0:r1] if route == "plan_rows" else np.ones(r1 - r0, bool))
        z64 = None if z64 is None else z64[r0:r1]
    elif route == "scatter":
        out = _table(n, d, strided)
        out.zero_()
        ops.spmm_scatter_rows(g.plan, g.col_idx, g.vals, x, out, rows, cnt, n, rb, addend=z)
        written = np.ones(n, bool)
    else:
        out = _table(n, d, strided)
        kw = {"plain": {}, "row_mask": dict(row_mask=rb), "row_edge": dict(row_mask=rb, edge_mask=eb),
              "rows": dict(row_mask=rb, rows=rows, n_rows_dev=cnt), "rows_edge": dict(row_mask=rb, edge_mask=eb, rows=rows, n_rows_dev=cnt),
              "edge": dict(edge_mask=eb)}[route]
        mm(x, out=out, addend=z, **kw)
        written = rmask if "row_mask" in kw else np.ones(n, bool)
    _counters_zero(g.plan, g.t_plan)
    if strided:
        w = out.as_strided((out.shape[0], d + 8), (out.stride(0), 1), out.storage_offset() - 4)
        assert bool((w[:, :4] == SENTINEL).all()) and bool((w[:, 4 + d :] == SENTINEL).all()), "columns outside the slice were written"
    y = out.cpu().double().numpy()
    # reference: dead sources (edge mask) or unlisted sources (scatter) contribute nothing; the addend counts for rows in the
    # edge mask (edge routes) or in the list (scatter) only
    src = live if edge else (rmask if route == "scatter" else np.ones(n, bool))
    xs = np.where(src[:, None], x64, 0.0)
    Mabs = abs(M)
    ref, absum = M @ xs, Mabs @ np.abs(xs)
    if z64 is not None:
        gate = src[r0:r1] if route in ("plan", "plan_rows") else src
        zg = np.where(gate[: m_rows, None], z64, 0.0) if (edge or route == "scatter") else z64
        ref, absum = ref + zg, absum + np.abs(zg)
    lens = np.diff(M.indptr)
    assert bool((y[~written] == SENTINEL).all()), f"{route}: rows outside the row mask were written"
    return y[written], ref[written], absum[written], lens[written]


def _set_values(g, A: sp.csr_matrix, kind: str, seed: int):
    rng = np.random.default_rng(seed)
    if kind == "exact":
        v = exact_weights(rng, A.nnz)
    elif kind == "attention":
        v = attention_weights(rng, A.indptr)
    else:
        v = rng.standard_normal(A.nnz).astype(np.float32)
    g.set_values(torch.from_numpy(v).cuda())
    A.data = v.astype(np.float64)


def _route_params():
    return [pytest.param(size, chunk, d, route, id=f"{size}-c{chunk}-d{d}-{route}") for size in SIZES for chunk in CHUNKS for d in DIMS
            for route in ROUTES]


@pytest.mark.parametrize("size,chunk,d,route", _route_params())
def test_exact(graphs, size, chunk, d, route):
    """Integer X / Z and +-2^-k weights: bit-exact against the float64 product, both directions, contiguous with an addend,
    strided with a strided addend, and without an addend (empty rows: exactly 0)."""
    g, A, live, rmask = graphs[(size, chunk)]
    _set_values(g, A, "exact", seed=d + chunk)
    rng = np.random.default_rng(d * chunk)
    n = g.n
    for t in ((True,) if route == "scatter" else (False, True)):
        for strided, with_z in ((False, True), (True, True), (False, False)):
            x64 = rng.integers(-8, 9, (n, d)).astype(np.float64)
            z64 = rng.integers(-8, 9, (n, d)).astype(np.float64) if with_z else None
            y, ref, _, lens = run_route(route, g, A, t, live, rmask, x64, z64, strided)
            bad = np.flatnonzero((y != ref.astype(np.float32)).any(axis=1))
            assert bad.size == 0, (f"{route} t={t} strided={strided} addend={with_z}: {bad.size} rows differ, first (length "
                                   f"{lens[bad[0]]}): got {y[bad[0], :4]} expected {ref[bad[0], :4]}")


@pytest.mark.parametrize("size,chunk,d,route", _route_params())
def test_rounding_bound(graphs, size, chunk, d, route):
    """Gaussian X / Z, attention-like weights for A and signed weights for A^T: every element within the a-priori fp32
    summation bound 1.01 (L + 2) 2^-24 (sum |a x| + |z|)."""
    g, A, live, rmask = graphs[(size, chunk)]
    rng = np.random.default_rng(7 * d + chunk)
    n = g.n
    for t in ((True,) if route == "scatter" else (False, True)):
        _set_values(g, A, "signed" if t else "attention", seed=d + chunk + t)
        x64 = rng.standard_normal((n, d)).astype(np.float32).astype(np.float64)
        z64 = rng.standard_normal((n, d)).astype(np.float32).astype(np.float64)
        y, ref, absum, lens = run_route(route, g, A, t, live, rmask, x64, z64, strided=bool(t))
        bound = 1.01 * (lens[:, None] + 2) * 2.0**-24 * absum
        err = np.abs(y - ref)
        bad = ~(err <= bound)
        assert not bad.any(), f"{route} t={t}: {int(bad.sum())} elements outside the bound (per element {elem_err(y, ref):.3g})"
        key = (route, d, "AT" if t else "A")
        RATIOS[key] = max(RATIOS.get(key, 0.0), float((err / np.where(bound > 0, bound, 1.0)).max()))


@pytest.mark.parametrize("size,chunk", [(s, c) for s in SIZES for c in CHUNKS])
@pytest.mark.parametrize("d", GENERIC_DIMS)
def test_generic_d(graphs, size, chunk, d):
    """The generic-d kernel and its separate heavy-row reduce: exact and within the bound on the plain and plan routes; the
    masked, edge-mask and scatter routes raise KgatLibraryError and leave out untouched."""
    from kgat_b200._lib import KgatLibraryError

    g, A, live, rmask = graphs[(size, chunk)]
    rng = np.random.default_rng(d + chunk)
    n = g.n
    for route in ("plain", "plan"):
        for t in (False, True):
            _set_values(g, A, "exact", seed=d)
            x64 = rng.integers(-8, 9, (n, d)).astype(np.float64)
            z64 = rng.integers(-8, 9, (n, d)).astype(np.float64)
            y, ref, _, _ = run_route(route, g, A, t, live, rmask, x64, z64, strided=t)
            assert np.array_equal(y, ref.astype(np.float32)), f"generic d={d} {route} t={t}"
            _set_values(g, A, "signed", seed=d)
            x64 = rng.standard_normal((n, d)).astype(np.float32).astype(np.float64)
            y, ref, absum, lens = run_route(route, g, A, t, live, rmask, x64, z64 / 8, strided=not t)
            assert (np.abs(y - ref) <= 1.01 * (lens[:, None] + 2) * 2.0**-24 * absum).all(), f"generic d={d} {route} t={t}"
    for route in ("row_mask", "row_edge", "rows", "rows_edge", "edge", "scatter"):
        with pytest.raises(KgatLibraryError, match="unsupported|failed"):
            run_route(route, g, A, False, live, rmask, np.zeros((n, d)), None, strided=False)


def test_unsupported_widths_rejected(graphs):
    """d = 2 (a column slice of a width-4 table, so the row stride is valid) and d = 260 never launch."""
    from kgat_b200._lib import KgatLibraryError

    g = graphs[("small", 256)][0]
    n = g.n
    for d, w in ((2, 4), (260, 260)):
        x = torch.zeros(n, w, device="cuda")[:, :d]
        big = torch.full((n, w), SENTINEL, device="cuda")
        with pytest.raises(KgatLibraryError):
            g.matmul(x, out=big[:, :d])
        torch.cuda.synchronize()
        assert bool((big == SENTINEL).all())


def test_wrong_output_shapes_rejected_before_launch(graphs):
    """ops.spmm / spmm_scatter_rows reject an out or addend of the wrong width or with fewer rows than the plan.  The bad
    tensors are views into larger buffers, so a launch that slipped through would still stay in bounds and show as a written
    SENTINEL."""
    from kgat_b200 import ops
    from kgat_b200._lib import KgatLibraryError

    g, A, live, rmask = graphs[("small", 8)]
    n, d = g.n, 32
    x = torch.ones(n, d, device="cuda")
    buf = torch.full((n, 2 * d), SENTINEL, device="cuda")
    partials = g.partials(d)
    cases = {
        "narrow out": dict(out=buf[:, : d - 4]),
        "short out": dict(out=buf[: n - 1, :d]),
        "narrow addend": dict(out=buf[:, :d], addend=torch.zeros(n, 2 * d, device="cuda")[:, : d - 4]),
        "short addend": dict(out=buf[:, :d], addend=torch.zeros(n - 1, d, device="cuda")),
    }
    for what, kw in cases.items():
        for extra in ({}, dict(row_mask=_bits(rmask)), dict(edge_mask=_bits(live))):
            with pytest.raises(KgatLibraryError, match="does not cover"):
                ops.spmm(g.plan, g.col_idx, g.vals, x, kw["out"], kw.get("addend"), partials, **extra)
            torch.cuda.synchronize()
            assert bool((buf == SENTINEL).all()), what
    listed = np.flatnonzero(rmask).astype(np.int32)
    rows, cnt = torch.from_numpy(listed).cuda(), torch.tensor([listed.size], dtype=torch.int32, device="cuda")
    for what, out, z in (("narrow out", buf[:, : d - 4], None), ("narrow addend", buf[:, :d], torch.zeros(n, 2 * d, device="cuda")[:, : d - 4])):
        with pytest.raises(KgatLibraryError, match="width"):
            ops.spmm_scatter_rows(g.plan, g.col_idx, g.vals, x, out, rows, cnt, n, _bits(rmask), addend=z)
        torch.cuda.synchronize()
        assert bool((buf == SENTINEL).all()), what


@pytest.mark.parametrize("d", [pytest.param(d, id=f"d{d}") for d in DIMS])
def test_graph_replay_and_repeat_calls(graphs, d):
    """matmul + matmul_t + matmul captured in one CUDA graph (the two directions share AttentiveGraph.partials), replayed three
    times with X changed in place: exact every time and the arrival counters back at 0.  Two eager calls of a gather route give
    identical bytes."""
    from kgat_b200 import functions

    g, A, live, rmask = graphs[("small", 8)]
    n = g.n
    _set_values(g, A, "exact", seed=3)
    At = A.T.tocsr()
    x1, x2 = torch.zeros(n, d, device="cuda"), torch.zeros(n, d, device="cuda")
    o1, o2, o3 = (torch.empty(n, d, device="cuda") for _ in range(3))

    def step():
        g.matmul(x1, out=o1)
        g.matmul_t(x1, out=o2)
        g.matmul(x2, out=o3)

    step()
    torch.cuda.synchronize()
    cg = torch.cuda.CUDAGraph()
    with functions.capture_graph(cg):
        step()
    gen = torch.Generator().manual_seed(d)
    for _ in range(3):
        a = torch.randint(-8, 9, (n, d), generator=gen).double()
        b = torch.randint(-8, 9, (n, d), generator=gen).double()
        x1.copy_(a)
        x2.copy_(b)
        cg.replay()
        torch.cuda.synchronize()
        _counters_zero(g.plan, g.t_plan)
        for got, M, xv in ((o1, A, a), (o2, At, a), (o3, A, b)):
            assert np.array_equal(got.cpu().numpy(), (M @ xv.numpy()).astype(np.float32))
    del cg
    _set_values(g, A, "attention", seed=4)
    x = torch.randn(n, d, device="cuda", generator=torch.Generator(device="cuda").manual_seed(d))
    rows = torch.from_numpy(np.flatnonzero(rmask).astype(np.int32)).cuda()
    cnt = torch.tensor([rows.numel()], dtype=torch.int32, device="cuda")
    for kw in ({}, dict(row_mask=_bits(rmask), edge_mask=_bits(live), rows=rows, n_rows_dev=cnt)):
        for mm in (g.matmul, g.matmul_t):
            a, b = mm(x, out=torch.zeros(n, d, device="cuda"), **kw), mm(x, out=torch.zeros(n, d, device="cuda"), **kw)
            assert torch.equal(a.view(torch.int32), b.view(torch.int32))


# ---------------------------------------------------------------------------------------------
# the 32-bit offset, WIDE and edge-bitmap thresholds, from one 4 GiB table
# ---------------------------------------------------------------------------------------------
FULL_ROWS, FULL_COLS = 262_145, 4096
VIEW_ROWS = [262_143, 262_144, 262_145]


def _pattern(r: torch.Tensor, c: torch.Tensor) -> torch.Tensor:
    """X[r, c] = ((131 r + 7 c) mod 17) - 8: a wrapped byte offset reads a valid row with different values."""
    return ((r[:, None] * 131 + c[None, :] * 7) % 17 - 8).to(torch.float32)


def test_threshold_offsets_and_edge_bitmap_4gib(kb, sms):
    """X_full of 262,145 x 4,096 fp32 (4 GiB + 16 KiB) and its views X_full[:R, 4096 - d:]: R = 262,143 (32-bit offsets up to
    ~2^32, 32 KiB edge bitmap in shared memory), 262,144 (WIDE at exactly 2^32, bitmap still in shared memory), 262,145 (WIDE,
    bitmap read from global memory).  Edges point mostly at rows >= 131,072 (byte offsets >= 2^31) and at the last rows."""
    from kgat_b200 import ops
    from kgat_b200.graph import make_plan

    if torch.cuda.mem_get_info()[0] < 8 * 2**30:
        pytest.skip("needs 8 GiB of free device memory")
    X = torch.empty(FULL_ROWS, FULL_COLS, device="cuda")
    try:
        assert X.numel() * 4 == 2**32 + 16 * 1024
        cols_used = torch.arange(FULL_COLS - 128, FULL_COLS, device="cuda")
        for r0 in range(0, FULL_ROWS, 32768):  # only the last 128 columns are read by any view
            r = torch.arange(r0, min(r0 + 32768, FULL_ROWS), device="cuda")
            X[r0 : r0 + r.numel(), FULL_COLS - 128 :] = _pattern(r, cols_used)
        m = 3000
        rng = np.random.default_rng(5)
        for R in VIEW_ROWS:
            # rows: a heavy row of 2,000 edges (chunks of 256), rows of 1 .. 300 edges, empty rows; the last rows in every 7th row
            lens = np.concatenate([[2000], rng.integers(0, 300, m - 1)])
            rows = np.repeat(np.arange(m, dtype=np.int64), lens)
            cols = rng.integers(131072, R, rows.size)
            last = np.repeat(np.arange(0, m, 7, dtype=np.int64), 3)  # every 7th row also reads the last two rows and row 131,072
            rows = np.concatenate([rows, last])
            cols = np.concatenate([cols, np.tile([R - 1, R - 2, 131072], last.size // 3)])
            keys = np.unique(rows * R + cols)
            rows, cols = keys // R, keys % R
            A = sp.csr_matrix((exact_weights(rng, keys.size).astype(np.float64), cols, np.concatenate([[0], np.cumsum(np.bincount(rows, minlength=m))])),
                              shape=(m, R))
            assert A.indices.max() == R - 1 and (A.indices >= 131072).mean() > 0.99
            plan = make_plan(torch.from_numpy(A.indptr.astype(np.int32)).cuda())
            assert plan.n_heavy > 0
            col = torch.from_numpy(A.indices.astype(np.int32)).cuda()
            vals = torch.from_numpy(A.data.astype(np.float32)).cuda()
            used = np.unique(A.indices)
            live = rng.random(R) < 0.6
            rmask = rng.random(m) < 0.7
            rmask[0] = True
            listed = np.flatnonzero(rmask).astype(np.int32)
            rows_t, cnt = torch.from_numpy(listed).cuda(), torch.tensor([listed.size], dtype=torch.int32, device="cuda")
            for d in DIMS:
                xv = X[:R, FULL_COLS - d :]
                bytes_ = xv.shape[0] * xv.stride(0) * 4
                assert (bytes_ < 2**32) == (R == 262_143) and (bytes_ == 2**32) == (R == 262_144)
                assert (((R + 31) // 32) * 4 <= 32 * 1024) == (R <= 262_144)
                xh = np.zeros((R, d))
                xh[used] = _pattern(torch.from_numpy(used), torch.arange(FULL_COLS - d, FULL_COLS)).double().numpy()
                z64 = rng.integers(-8, 9, (m, d)).astype(np.float64)
                z = torch.from_numpy(z64).float().cuda()
                partials = torch.empty(plan.n_partials * d, device="cuda")
                for route, kw in (("plain", {}), ("row_mask", dict(row_mask=_bits(rmask, R))),
                                  ("rows", dict(row_mask=_bits(rmask, R), rows=rows_t, n_rows_dev=cnt)),
                                  ("rows_edge", dict(row_mask=_bits(rmask, R), edge_mask=_bits(live), rows=rows_t, n_rows_dev=cnt)),
                                  ("edge", dict(edge_mask=_bits(live)))):
                    out = torch.full((m, d), SENTINEL, device="cuda")
                    ops.spmm(plan, col, vals, xv, out, z, partials, **kw)
                    _counters_zero(plan)
                    edge = "edge_mask" in kw
                    ref = A @ (np.where(live[:, None], xh, 0.0) if edge else xh) + (np.where(live[:m, None], z64, 0.0) if edge else z64)
                    w = rmask if "row_mask" in kw else np.ones(m, bool)
                    y = out.cpu().numpy()
                    assert (y[~w] == SENTINEL).all(), f"R={R} d={d} {route}: unmasked rows written"
                    bad = np.flatnonzero((y[w] != ref[w].astype(np.float32)).any(axis=1))
                    assert bad.size == 0, f"R={R} d={d} {route}: {bad.size} rows differ"
    finally:
        del X
        torch.cuda.empty_cache()


# ---------------------------------------------------------------------------------------------
# the needed-row frontier at scale
# ---------------------------------------------------------------------------------------------
def frontier_graph(n: int, seed: int):
    """Zipf row lengths, Zipf-popular columns, and a hub row of 60,000 edges (or n / 4 on small graphs) at id 123."""
    rng = np.random.default_rng(seed)
    lens = np.minimum(rng.zipf(2.0, n), 2000)
    lens[123] = min(60000, n // 4)
    rows = np.repeat(np.arange(n, dtype=np.int64), lens)
    perm = rng.permutation(n)
    cols = perm[(rng.zipf(1.3, rows.size) - 1) % n]
    cols[rows == 123] = rng.choice(n, lens[123], replace=False)
    keys = np.unique(rows * n + cols)
    row_ptr = np.concatenate([[0], np.cumsum(np.bincount(keys // n, minlength=n))])
    return row_ptr, (keys % n).astype(np.int32)


def bfs_levels(ptr, idx, n: int, ids: np.ndarray, layers: int) -> dict:
    """level -> bool [n]: F_L = ids, F_{l-1} = F_l | cols(A[F_l, :]) (vectorised over the CSR)."""
    level = np.zeros(n, bool)
    level[ids] = True
    out = {layers: level}
    for lv in range(layers - 1, 0, -1):
        rows = np.flatnonzero(level)
        lens = ptr[rows + 1] - ptr[rows]
        slots = np.repeat(ptr[rows] - (np.cumsum(lens) - lens), lens) + np.arange(int(lens.sum()))
        level = level.copy()
        level[idx[slots]] = True
        out[lv] = level
    return out


FRONTIER_N = [1_700_000, 1_638_400, 8_193]


@pytest.fixture(scope="module", params=FRONTIER_N, ids=[f"n{n}" for n in FRONTIER_N])
def fgraph(request, kb):
    from kgat_b200.graph import AttentiveGraph

    n = request.param
    ptr, idx = frontier_graph(n, seed=n % 1000)
    g = AttentiveGraph(n, torch.from_numpy(ptr.astype(np.int32)).cuda(), torch.from_numpy(idx).cuda(), torch.zeros(idx.size, device="cuda"))
    return n, ptr, idx, g


def _check_frontier(f, ptr, idx, n, ids, layers):
    ref = bfs_levels(ptr, idx, n, ids, layers)
    for lv in range(layers, 0, -1):
        rows = np.flatnonzero(ref[lv])
        assert int(f.count(lv).item()) == rows.size, f"level {lv}: count"
        np.testing.assert_array_equal(f.rows(lv)[: rows.size].cpu().numpy(), rows, err_msg=f"level {lv}: rows")
        words = f.mask(lv).cpu().numpy().view(np.uint32)
        expect = np.packbits(np.pad(ref[lv], (0, words.size * 32 - n)), bitorder="little").view(np.uint32)
        np.testing.assert_array_equal(words, expect, err_msg=f"level {lv}: bitmap")
    assert int(f.flags.max()) == 0, "flags not cleared by the listing pass"
    return ref


def test_frontier_levels_at_scale(fgraph, sms):
    """Frontier levels (bitmaps, row lists, counts) against the numpy BFS, bit for bit; a second build leaves nothing of the
    first.  n = 1,700,000: the global-store expand kernel (bitmap > 200 KiB) and 208 listing CTAs; n = 1,638,400: the
    shared-memory kernel at its 200 KiB limit; n = 8,193: a second listing CTA holding one word."""
    from kgat_b200.frontier import Frontier

    n, ptr, idx, g = fgraph
    words = (n + 31) // 32
    if n == 1_700_000:
        assert words * 4 > 200 * 1024 and (words + 255) // 256 == 208
    elif n == 1_638_400:
        assert words * 4 == 200 * 1024
    else:
        assert (words + 255) // 256 == 2 and words - 256 == 1
    rng = np.random.default_rng(n)
    layers = 3
    f = Frontier(g, layers, 768)
    ids = rng.integers(0, n, 768)
    ids[:3] = [123, n - 1, 8192 if n > 8192 else 0]
    t = torch.from_numpy(ids).cuda()
    f.build([t[:256], t[256:]])
    ref = _check_frontier(f, ptr, idx, n, ids, layers)
    assert ref[1].sum() >= ref[2].sum() > ref[3].sum()
    ids2 = rng.integers(0, n, 500)  # the second build: nothing of the first may survive
    f.build([torch.from_numpy(ids2).cuda()])
    _check_frontier(f, ptr, idx, n, ids2, layers)


def test_frontier_segment(fgraph):
    """ops.frontier_segment against numpy: [0, 32), a middle range, the last range (ending at n, not a multiple of 32 for
    n = 8,193), an empty range, [0, n), and a level with count 0."""
    from kgat_b200 import ops
    from kgat_b200.frontier import Frontier

    n, ptr, idx, g = fgraph
    f = Frontier(g, 2, 512)
    ids = np.random.default_rng(1).integers(0, n, 512)
    ids[0] = n - 1
    f.build([torch.from_numpy(ids).cuda()])
    level = bfs_levels(ptr, idx, n, ids, 2)[1]
    words = (n + 31) // 32
    mid, mid2, last = (n // 3) // 32 * 32, (2 * n // 3) // 32 * 32, (n - 100) // 32 * 32
    empty_rows, empty_cnt = torch.zeros(n, dtype=torch.int32, device="cuda"), torch.zeros(1, dtype=torch.int32, device="cuda")
    empty_mask = torch.zeros(f.words, dtype=torch.int32, device="cuda")
    for lvl_rows, lvl_cnt, lvl_mask, lvl in ((f.rows(1), f.count(1), f.mask(1), level), (empty_rows, empty_cnt, empty_mask, np.zeros(n, bool))):
        all_rows = np.flatnonzero(lvl)
        for lo, hi in ((0, 32), (mid, mid2), (last, n), (mid, mid), (0, n)):
            out_rows = torch.full((n,), -7, dtype=torch.int32, device="cuda")
            out_cnt = torch.full((1,), 99, dtype=torch.int32, device="cuda")
            out_mask = torch.full((words,), -1, dtype=torch.int32, device="cuda")
            ops.frontier_segment(lvl_rows, lvl_cnt, lvl_mask, n, lo, hi, out_rows, out_cnt, out_mask)
            seg = all_rows[(all_rows >= lo) & (all_rows < hi)]
            assert int(out_cnt.item()) == seg.size, (lo, hi)
            np.testing.assert_array_equal(out_rows[: seg.size].cpu().numpy(), seg)
            assert bool((out_rows[seg.size :] == -7).all())
            inside = np.zeros(words * 32, bool)
            inside[: n] = lvl
            inside[: lo] = False
            inside[(hi + 31) // 32 * 32 :] = False
            np.testing.assert_array_equal(out_mask.cpu().numpy().view(np.uint32), np.packbits(inside, bitorder="little").view(np.uint32))


@pytest.mark.parametrize("d", [16, 128])
def test_frontier_zero_rows(kb, sms, d):
    """ops.frontier_zero_rows on a strided table (ld > d) with more rows than one pass of its grid: listed rows zeroed in the
    d columns only, every other row and column unchanged, list entries past the count ignored."""
    from kgat_b200 import ops

    n, cnt = 100_000, 40_000
    assert cnt * d // 4 > sms * 4 * 256
    rng = np.random.default_rng(d)
    perm = rng.permutation(n).astype(np.int32)
    wide = torch.randn(n, d + 12, device="cuda")
    before = wide.clone()
    T = wide[:, :d]
    ops.frontier_zero_rows(T, torch.from_numpy(perm).cuda(), torch.tensor([cnt], dtype=torch.int32, device="cuda"), n)
    expect = before.clone()
    expect[torch.from_numpy(perm[:cnt]).long().cuda(), :d] = 0.0
    assert torch.equal(wide, expect)


# ---------------------------------------------------------------------------------------------
# the env-latched instances
# ---------------------------------------------------------------------------------------------
def test_env_latched_variants_in_child(kb):
    """The d = 64 and 128 cases, the threshold cases and the frontier cases of this module again, in one child process under
    KGAT_SPMM_U=4 (d = 64 at U = 4), KGAT_SPMM_CTAS=6 (six CTAs per SM of the unmasked rows kernel) and KGAT_EXPAND_PLAIN=1 (the
    global-store frontier expand at every size)."""
    if IN_CHILD:
        pytest.skip("already the child")
    r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-x", "-p", "no:cacheprovider", "-m", "gpu", str(Path(__file__).resolve()), "-k",
                        "d64 or d128 or threshold or frontier"], env=dict(os.environ, **CHILD_ENV), cwd=str(ROOT), capture_output=True, text=True,
                       timeout=1800)
    assert r.returncode == 0, f"child failed ({r.returncode}):\n{r.stdout[-4000:]}\n{r.stderr[-2000:]}"

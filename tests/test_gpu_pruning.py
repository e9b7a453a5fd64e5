"""GPU tests of the needed-row pruning of the TRAIN_CF step (frontier.py, csrc/frontier.cu, the masked SpMM and the
row-list bi-interaction kernels).  The pruned step must equal the reference's full-graph propagation
(model.py:165-202) on everything the loss reads and on every gradient.

Tolerances: frontier bitmaps / row lists / counts bit-exact vs a numpy breadth-first restatement; the row-masked SpMM
bit-exact vs the unmasked kernel on the surviving rows (2e-6 when edges are masked too: the survivors are packed, which
changes the fp32 summation order); pruned vs full step: loss 1e-6, gradients 2e-6 normwise
(identical per-row arithmetic; only the summation order of the weight-gradient partials differs)."""

from __future__ import annotations

import numpy as np
import pytest
import torch

from conftest import Golden, rel_err
from oracle import kgat_oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def kb():
    if not torch.cuda.is_available():
        pytest.skip("needs CUDA")
    import kgat_b200

    kgat_b200._lib.load()
    return kgat_b200


def _random_graph(n, m, seed, chunk=256, heavy=()):
    from kgat_b200.graph import AttentiveGraph

    rng = np.random.default_rng(seed)
    rows = rng.integers(0, n, m)
    cols = rng.integers(0, n, m)
    for r, k in heavy:
        rows = np.concatenate([rows, np.full(k, r)])
        cols = np.concatenate([cols, rng.integers(0, n, k)])
    vals = rng.standard_normal(rows.size).astype(np.float32)
    g = AttentiveGraph.from_coo(torch.from_numpy(rows).cuda(), torch.from_numpy(cols).cuda(), torch.from_numpy(vals).cuda(), n, chunk=chunk)
    return g


def _bits(mask_np, words):
    """bool [n] -> int32 [words] bitmap (bit i of word i >> 5)."""
    pad = np.zeros(words * 32, dtype=bool)
    pad[: mask_np.size] = mask_np
    return torch.from_numpy(np.packbits(pad, bitorder="little").view(np.int32).copy()).cuda()


def _unbits(t, n):
    return np.unpackbits(t.cpu().numpy().view(np.uint8), bitorder="little")[:n].astype(bool)


@pytest.mark.parametrize("n,m,layers,n_ids", [(1000, 3000, 3, 12), (5000, 40000, 2, 64), (257, 600, 4, 5), (64, 10, 3, 3)])
def test_frontier_levels_match_numpy_bfs(kb, n, m, layers, n_ids):
    from kgat_b200.frontier import Frontier

    g = _random_graph(n, m, seed=n + layers, heavy=[(7, 900)])
    rng = np.random.default_rng(n_ids)
    ids = rng.integers(0, n, n_ids)
    ids[-1] = ids[0]  # a duplicate id
    ptr, idx = g.row_ptr.cpu().numpy(), g.col_idx.cpu().numpy()
    f = Frontier(g, layers, 2 * n_ids)
    t = torch.from_numpy(ids).cuda()
    f.build([t[: n_ids // 2], t[n_ids // 2 :]])
    level = np.zeros(n, bool)
    level[ids] = True
    for l in range(layers, 0, -1):
        rows = np.nonzero(level)[0]
        assert int(f.count(l).item()) == rows.size
        np.testing.assert_array_equal(f.rows(l)[: rows.size].cpu().numpy(), rows)
        np.testing.assert_array_equal(_unbits(f.mask(l), n), level)
        nxt = level.copy()
        for r in rows:
            nxt[idx[ptr[r] : ptr[r + 1]]] = True
        level = nxt
    # rebuilding for another batch leaves nothing behind from the first one
    ids2 = rng.integers(0, n, 3)
    f.build([torch.from_numpy(ids2).cuda()])
    assert int(f.count(layers).item()) == np.unique(ids2).size
    assert int(f.bad_ids.item()) == 0
    f.build([torch.tensor([0, n, -1, 5]).cuda()])  # out-of-range ids are skipped and counted
    assert int(f.count(layers).item()) == 2
    with pytest.raises(IndexError):
        f.check_ids()
    f.check_ids()  # the counter was reset


@pytest.mark.parametrize("d", [16, 32, 64, 128])
@pytest.mark.parametrize("chunk", [8, 256])
def test_masked_spmm_equals_dense_on_live_rows_and_never_reads_dead_ones(kb, d, chunk):
    n = 700
    g = _random_graph(n, 9000, seed=d + chunk, chunk=chunk, heavy=[(17, 800), (250, 40)])
    rng = np.random.default_rng(d)
    words = (n + 31) // 32
    for p_row, p_col in [(0.3, 0.6), (1.0, 0.1), (0.05, 1.0), (0.5, 0.0)]:
        rmask, cmask = rng.random(n) < p_row, rng.random(n) < p_col
        rmask[17] = True
        x = torch.randn(n, d, device="cuda")
        z = torch.randn(n, d, device="cuda")
        xz, zz = x.clone(), z.clone()
        live = torch.from_numpy(cmask).cuda()
        xz[~live] = 0.0  # reference: dead source rows contribute nothing ...
        zz[~live] = 0.0  # ... and the addend counts only for rows in the edge mask
        x[~live] = float("nan")  # the masked kernel must never touch them
        z[~live] = float("nan")
        for t in (False, True):
            mm = g.matmul_t if t else g.matmul
            ref = mm(xz, addend=zz)
            out = torch.full((n, d), 7.0, device="cuda")
            mm(x, out=out, addend=z, row_mask=_bits(rmask, words), edge_mask=_bits(cmask, words))
            rm = torch.from_numpy(rmask).cuda()
            # surviving edges are packed before the gather, so they meet the lane groups in another order: fp32 rounding only
            assert rel_err(out[rm], ref[rm]) < 2e-6 and bool(torch.isfinite(out[rm]).all())
            assert bool((out[~rm] == 7.0).all())  # rows outside the row mask are not written
        # the persistent row-list kernel: same masks plus the ascending list of the live rows and a device-side count
        listed = np.nonzero(rmask)[0].astype(np.int32)
        rows = torch.zeros(n, dtype=torch.int32, device="cuda")
        rows[: listed.size] = torch.from_numpy(listed).cuda()
        cnt = torch.tensor([listed.size], dtype=torch.int32, device="cuda")
        rm = torch.from_numpy(rmask).cuda()
        for t in (False, True):
            mm = g.matmul_t if t else g.matmul
            ref = mm(xz, addend=zz)
            out = torch.full((n, d), 7.0, device="cuda")
            mm(x, out=out, addend=z, row_mask=_bits(rmask, words), edge_mask=_bits(cmask, words), rows=rows, n_rows_dev=cnt)
            assert rel_err(out[rm], ref[rm]) < 2e-6 and bool(torch.isfinite(out[rm]).all())
            assert bool((out[~rm] == 7.0).all())
            out = torch.full((n, d), 7.0, device="cuda")
            mm(xz, out=out, row_mask=_bits(rmask, words), rows=rows, n_rows_dev=cnt)  # forward use: rows only
            assert torch.equal(out[rm], mm(xz)[rm]) and bool((out[~rm] == 7.0).all())
            out = torch.full((n, d), 7.0, device="cuda")
            mm(x, out=out, addend=z, edge_mask=_bits(cmask, words))  # dense output, masked sources (the embedding gradient)
            assert rel_err(out, ref) < 2e-6 and bool(torch.isfinite(out).all())
        # row mask only (the forward use): no edge filtering, no addend gating
        ref = g.matmul(xz)
        out = torch.full((n, d), 7.0, device="cuda")
        g.matmul(xz, out=out, row_mask=_bits(rmask, words))
        rm = torch.from_numpy(rmask).cuda()
        assert torch.equal(out[rm], ref[rm]) and bool((out[~rm] == 7.0).all())


@pytest.mark.parametrize("d", [16, 32, 64, 128])
@pytest.mark.parametrize("chunk", [8, 256])
def test_scatter_rows_equals_transposed_gather(kb, d, chunk):
    """Y[c] += A[r, c] G[r] over a row list (vector reductions) == the masked gather over A^T, up to fp32 summation order."""
    from kgat_b200 import ops

    n = 700
    g = _random_graph(n, 9000, seed=3 * d + chunk, chunk=chunk, heavy=[(17, 800), (250, 40)])
    rng = np.random.default_rng(d + 1)
    words = (n + 31) // 32
    for p_src in (0.02, 0.3, 1.0):
        src = rng.random(n) < p_src
        src[17] = True
        listed = np.nonzero(src)[0].astype(np.int32)
        rows = torch.zeros(n, dtype=torch.int32, device="cuda")
        rows[: listed.size] = torch.from_numpy(listed).cuda()
        cnt = torch.tensor([listed.size], dtype=torch.int32, device="cuda")
        live = torch.from_numpy(src).cuda()
        G, Z = torch.randn(n, d, device="cuda"), torch.randn(n, d, device="cuda")
        Gz, Zz = G.clone(), Z.clone()
        Gz[~live] = 0.0
        Zz[~live] = 0.0
        ref = g.matmul_t(Gz, addend=Zz)
        G[~live] = float("nan")
        Z[~live] = float("nan")
        out = torch.zeros(n, d, device="cuda")
        ops.spmm_scatter_rows(g.plan, g.col_idx, g.vals, G, out, rows, cnt, n, _bits(src, words), addend=Z)
        assert bool(torch.isfinite(out).all()) and rel_err(out, ref) < 2e-6


@pytest.mark.parametrize("d_in,d_out", [(64, 64), (64, 32), (32, 16), (128, 64)])
@pytest.mark.parametrize("p", [0.0, 0.1])
def test_biagg_row_list_equals_dense_kernels_on_listed_rows(kb, d_in, d_out, p):
    from kgat_b200 import ops

    n = 1500
    rng = np.random.default_rng(d_in * d_out)
    torch.manual_seed(d_in + d_out)
    listed = np.sort(rng.choice(n, size=333, replace=False)).astype(np.int32)
    rows = torch.zeros(n, dtype=torch.int32, device="cuda")
    rows[: listed.size] = torch.from_numpy(listed).cuda()
    cnt = torch.tensor([listed.size], dtype=torch.int32, device="cuda")
    E, S = torch.randn(n, d_in, device="cuda"), torch.randn(n, d_in, device="cuda")
    W1, W2 = torch.randn(d_out, d_in, device="cuda") * 0.2, torch.randn(d_out, d_in, device="cuda") * 0.2
    b1, b2 = torch.randn(d_out, device="cuda") * 0.1, torch.randn(d_out, device="cuda") * 0.1
    li = torch.from_numpy(listed).long().cuda()
    dead = torch.ones(n, dtype=torch.bool, device="cuda")
    dead[li] = False

    def fwd(rows_kw, Ein, Sin):
        out = torch.full((n, d_out), 3.0, device="cuda")
        inv = torch.full((n,), 3.0, device="cuda")
        flags = torch.full((n, d_out), 9, dtype=torch.uint8, device="cuda")
        ops.biagg_forward(Ein, Sin, W1, b1, W2, b2, out, inv, flags, dropout_p=p, seed=11, offset=1 << 40, **rows_kw)
        return out, inv, flags

    kw = {"rows": rows, "n_rows_dev": cnt, "max_rows": n}
    Ep, Sp = E.clone(), S.clone()
    Ep[dead] = float("nan")
    Sp[dead] = float("nan")
    o_d, i_d, f_d = fwd({}, E, S)
    o_r, i_r, f_r = fwd(kw, Ep, Sp)
    # same kernel, same per-row arithmetic, dropout keyed by node id: bit-exact on the listed rows
    assert torch.equal(o_r[li], o_d[li]) and torch.equal(i_r[li], i_d[li]) and torch.equal(f_r[li], f_d[li])
    assert bool((o_r[dead] == 3.0).all()) and bool((i_r[dead] == 3.0).all()) and bool((f_r[dead] == 9).all())

    g_out = torch.randn(n, d_out, device="cuda")
    g_zero = g_out.clone()
    g_zero[dead] = 0.0  # dense reference: rows outside the list carry a zero upstream gradient

    def bwd(rows_kw, gin, out, inv, flags, Ein, Sin):
        n_ctas = ops.biagg_backward_ctas(n, d_in, d_out, rows=bool(rows_kw))
        partials = torch.empty(n_ctas * (2 * d_in * d_out + 2 * d_out), device="cuda")
        g_s = torch.full((n, d_in), 5.0, device="cuda")
        g_e = torch.full((n, d_in), 5.0, device="cuda")
        ops.biagg_backward(gin, out, inv, flags, Ein, Sin, W1, W2, p, g_s, g_e, partials, n_ctas, **rows_kw)
        gw1, gb1, gw2, gb2 = torch.empty_like(W1), torch.empty_like(b1), torch.empty_like(W2), torch.empty_like(b2)
        ops.biagg_reduce_param_grads(partials, n_ctas, d_in, d_out, gw1, gb1, gw2, gb2)
        return g_s, g_e, (gw1, gb1, gw2, gb2)

    gs_d, ge_d, pg_d = bwd({}, g_zero, o_d, i_d, f_d, E, S)
    gp = g_out.clone()
    gp[dead] = float("nan")
    o_p, i_p = o_r.clone(), i_r.clone()
    o_p[dead] = float("nan")
    i_p[dead] = float("nan")
    gs_r, ge_r, pg_r = bwd(kw, gp, o_p, i_p, f_r, Ep, Sp)
    assert rel_err(gs_r[li], gs_d[li]) < 1e-6 and rel_err(ge_r[li], ge_d[li]) < 1e-6
    assert bool((gs_r[dead] == 5.0).all()) and bool((ge_r[dead] == 5.0).all())
    for a, b in zip(pg_r, pg_d):
        assert rel_err(a, b) < 5e-6  # different tile composition -> different fp32 summation order
    # empty list: nothing is written, parameter gradients are zero
    cnt0 = torch.zeros(1, dtype=torch.int32, device="cuda")
    gs0, ge0, pg0 = bwd({"rows": rows, "n_rows_dev": cnt0, "max_rows": n}, gp, o_p, i_p, f_r, Ep, Sp)
    assert bool((gs0 == 5.0).all()) and all(float(t.abs().max()) == 0.0 for t in pg0)


def _small_model(kb, layer_size, seed=3):
    from kgat_b200 import synthetic
    from kgat_b200.trainer import build_model

    g = synthetic.make_ckg("small", seed=seed)
    kw = {"layer_size": layer_size, "message_dropout": [0.1] * len(layer_size)}
    return g, build_model(g, "cuda", seed=seed, **kw)


@pytest.mark.parametrize("layer_size", [[64, 32, 16], [64], [32, 32, 16, 16]])
@pytest.mark.parametrize("mode", ["eval", "train-masks", "train-philox", "eval-gather"])
def test_pruned_cf_step_equals_full_propagation(kb, layer_size, mode):
    """model.cf_pruning on / off: same loss, same gradients; with every stale row poisoned by NaN.
    ("eval-gather": the upper layers' backward as the deterministic masked gather instead of the edge scatter.)"""
    from kgat_b200 import functions
    from kgat_b200.model import KGATMode

    g, model = _small_model(kb, layer_size)
    model.api_graphs = False
    if mode in ("eval", "eval-gather"):  # the edge scatter is no longer the default: select each backward explicitly
        model._frontier(model.cuda()._graph(), 3 * 6).scatter_backward = mode == "eval"
        mode = "eval"
    rng = np.random.default_rng(len(layer_size))
    b = 6
    u = torch.from_numpy(rng.integers(0, g.user_num, b)).cuda()
    p = torch.from_numpy(rng.integers(0, g.item_num, b)).cuda()
    q = torch.from_numpy(rng.integers(0, g.item_num, b)).cuda()
    n = g.node_num
    if mode == "eval":
        model.eval()
    else:
        model.train()
    if mode == "train-masks":
        keep = [rng.random((n, d)) < 0.9 for d in layer_size]
        model._injected_message_keep_bits = [
            torch.from_numpy(np.packbits(np.pad(k, ((0, 0), (0, (-k.shape[1]) % 32))), axis=1, bitorder="little").view(np.int32).copy()).cuda()
            for k in keep
        ]
    results = []
    for pruning in (False, True):
        model.cf_pruning = pruning
        model.zero_grad()
        functions.POISON_STALE_ROWS = pruning
        try:
            if mode == "train-philox":
                torch.manual_seed(77)  # the dropout seed is drawn from torch's CPU generator per forward
            loss = model(u, p, q, mode=KGATMode.TRAIN_CF)
            loss.backward()
        finally:
            functions.POISON_STALE_ROWS = False
        grads = {k: v.grad.detach().clone() for k, v in model.named_parameters() if v.grad is not None}
        results.append((float(loss), grads))
    (l0, g0), (l1, g1) = results
    assert np.isfinite(l1) and abs(l1 - l0) <= 1e-6 * max(abs(l0), 1.0)
    assert g0.keys() == g1.keys() and len(g0) == 1 + 4 * len(layer_size)
    for k in g0:
        assert bool(torch.isfinite(g1[k]).all()), k
        assert rel_err(g1[k], g0[k]) < 2e-6, k
    # the frontier really pruned something on this graph for the shallow configurations
    f = model._frontier(model._graph(), 3 * b)
    counts = f.counts.cpu().tolist()
    assert counts[-1] == np.unique(np.concatenate([u.cpu().numpy(), p.cpu().numpy(), q.cpu().numpy()])).size
    assert all(counts[i] >= counts[i + 1] for i in range(len(counts) - 1))
    assert counts[-1] < n


def test_pruned_cf_against_reference_golden_and_oracle(kb, golden_model):
    """The pruned step against the unmodified reference's outputs (golden) -- the default path of every other test in
    test_gpu_parity.py, restated here with small batches so that the frontier is a strict subset of the graph."""
    from kgat_b200.model import KGAT, KGATArgs, KGATMode

    g = golden_model
    m = KGAT(KGATArgs(user_num=int(g["user_num"]), entity_num=int(g["entity_num"]), relation_num=int(g["relation_num"]), attentive_matrix=g.att_coo()))
    m.load_state_dict(g.params(), strict=False)
    m = m.cuda().eval()
    m.api_graphs = False
    u, p, q = (torch.from_numpy(g[k][:3].copy()) for k in ("cf_users", "cf_pos", "cf_neg"))
    loss = m(u.cuda(), p.cuda(), q.cuda(), mode=KGATMode.TRAIN_CF)
    loss.backward()
    leaves = {k: v.clone().requires_grad_(True) for k, v in g.params().items()}
    ref = O.cf_loss(leaves, g.att_coo(), u, p, q)
    ref.backward()
    assert rel_err(loss, ref) < 1e-5
    for k, v in m.named_parameters():
        if v.grad is not None:
            assert rel_err(v.grad, leaves[k].grad) < 5e-5, k


@pytest.mark.parametrize("use_graphs", [False, True])
def test_engine_and_api_graph_paths_with_pruning_match_unpruned(kb, use_graphs):
    """Three CF steps (Adam included) through the captured engine / the captured API path, pruning on vs off."""
    from kgat_b200 import synthetic
    from kgat_b200.engine import TrainEngine
    from kgat_b200.trainer import EpochData, build_model, run_epoch

    g = synthetic.make_ckg("small", seed=5)
    data = EpochData.sample(g, seed=5, n_cf=3, n_kg=1)
    outs = {}
    for pruning in (False, True):
        for path in ("engine", "api"):
            model = build_model(g, "cuda", seed=5)
            model.eval()  # dropout off: the two settings must agree to rounding
            model.cf_pruning = pruning
            if path == "engine":
                eng = TrainEngine(model, use_graphs=use_graphs)
                eng.bind_resident(data.tensors())
                model.train = lambda *a, **k: model  # keep eval() semantics inside run_epoch
                cf, _, _, _ = eng.run_epoch(n_cf=3, n_kg=0, refresh=False)
            else:
                model.api_graphs = use_graphs
                model.train = lambda *a, **k: model
                cf, _, _, _ = run_epoch(model, data.tensors(device="cuda"), n_cf=3, n_kg=0, refresh=False)
            outs[(pruning, path)] = (cf, model._user_entity_embedding.weight.detach().clone(),
                                     model._aggregator_layers[0].linear1.weight.detach().clone())
    base = outs[(False, "api")]
    for k, v in outs.items():
        assert abs(v[0] - base[0]) < 1e-6 * max(1.0, abs(base[0])), k
        # three Adam steps of lr 1e-3 from identical states: parameters agree far inside one step size
        assert float((v[1] - base[1]).abs().max()) < 2e-5, k
        assert float((v[2] - base[2]).abs().max()) < 2e-5, k


def test_range_sharded_engine_world1_matches_single_gpu_engine(kb):
    """sharded_pruned.RangeShardedEngine with one rank (no exchange, but the same segment / range-mask / sliced-Adam code path)
    reproduces the single-GPU engine: two epochs (CF + KG + refresh), captured graphs."""
    from kgat_b200 import synthetic
    from kgat_b200.engine import TrainEngine
    from kgat_b200.model import KGATMode
    from kgat_b200.sharded_pruned import RangeShardedEngine, balanced_ranges
    from kgat_b200.trainer import EpochData, build_model

    g = synthetic.make_ckg("small", seed=11)
    data = EpochData.sample(g, seed=3, n_cf=4, n_kg=6)
    kw = dict(message_dropout=[0.0, 0.0, 0.0])
    models = [build_model(g, "cuda", seed=5, **kw) for _ in range(2)]
    for m in models:
        m._multi_head_attention._dropout.p = 0.0
    single = TrainEngine(models[0])
    holder = single.bind_resident(data.tensors())
    for m in models:
        m(*holder.edges, mode=KGATMode.UPDATE_ATTENTION)
    l_single = [single.run_epoch()[:2] for _ in range(2)]
    eng = RangeShardedEngine(models[1], 1, 0)
    eng.bind_resident(data.tensors())
    l_sharded = [eng.run_epoch(epoch_seed=i) for i in range(2)]
    for a, b in zip(l_single, l_sharded):
        assert abs(a[0] - b[0]) < 2e-6 and abs(a[1] - b[1]) < 2e-6
    a, b = models[0].state_dict(), models[1].state_dict()
    for k in a:
        if not a[k].is_sparse:
            assert float((b[k].double() - a[k].double()).norm() / a[k].double().norm().clamp_min(1e-30)) < 2e-5, k
    assert rel_err(b["attentive_matrix"]._values(), a["attentive_matrix"]._values()) < 1e-5
    # cost-balanced contiguous ranges: word-aligned, covering, ordered
    gr = models[1]._graph()
    for world in (2, 3, 8):
        r = balanced_ranges(gr.row_ptr.cpu().numpy(), gr.t_ptr.cpu().numpy(), world)
        assert r[0][0] == 0 and r[-1][1] == g.node_num and all(x[1] == y[0] for x, y in zip(r, r[1:]))
        assert all(lo % 32 == 0 and hi > lo for lo, hi in r)
    eng.close()


def test_range_sharded_engine_multi_gpu(kb):
    """World size 2 (or all visible GPUs up to 4) over NVLink peer memory against the single-GPU engine; skipped on a one-GPU box."""
    import subprocess
    import sys as _sys
    from pathlib import Path

    n = min(torch.cuda.device_count(), 4)
    if n < 2:
        pytest.skip("needs 2 GPUs")
    script = str(Path(__file__).with_name("sharded_pruned_check.py"))
    r = subprocess.run([_sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(n), "--master-addr", "127.0.0.1",
                        "--master-port", "29541", script], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-4000:]

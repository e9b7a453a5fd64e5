"""Path explanations (``kgat_explain_paths``, ``ops.explain_paths``, ``KGAT.explain``) against the torch reference
``oracle/explain_ref.py``.  Everything the kernel returns is compared bit for bit, except ``mass``: the kernel sums in fp64
in its own fixed order and rounds to fp32, the reference sums in fp64, so they agree to 1e-5 relative."""

from __future__ import annotations

import numpy as np
import pytest
import torch

from conftest import Golden
from oracle.explain_ref import explain_paths_ref

# ---------------------------------------------------------------------------------------------
# CPU: the reference on a hand-built graph whose paths are written out below
# ---------------------------------------------------------------------------------------------
#   row 0: 0 (self-loop) .5, 1 .5, 2 .5, 5 .25          slots 0-3
#   row 1: 0 .5, 2 .25, 3 .5, 5 .5                       slots 4-7
#   row 2: 1 1.0, 5 .5                                   slots 8-9
#   row 3: 5 1.0                                         slot 10
#   row 5: 5 (self-loop) .5                              slot 11
#   row 6: 7 1.0                                         slot 12
# All values are powers of two, so every product is exact and five paths 0 -> 5 tie at 0.25.
HAND_ROWS = [0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 3, 5, 6]
HAND_COLS = [0, 1, 2, 5, 0, 2, 3, 5, 1, 5, 5, 5, 7]
HAND_VALS = [.5, .5, .5, .25, .5, .25, .5, .5, 1., .5, 1., .5, 1.]
# 0 -> 5, H = 3, in rank order: (nodes, slots, weight)
HAND_PATHS_0_5 = [
    ([0, 5], [3], .25),
    ([0, 1, 5], [1, 7], .25),
    ([0, 2, 5], [2, 9], .25),
    ([0, 1, 3, 5], [1, 6, 10], .25),
    ([0, 2, 1, 5], [2, 8, 7], .25),
    ([0, 1, 2, 5], [1, 5, 9], .0625),
]


def _hand_csr():
    n = 8
    row_ptr = torch.from_numpy(np.concatenate([[0], np.cumsum(np.bincount(HAND_ROWS, minlength=n))]).astype(np.int32))
    return row_ptr, torch.tensor(HAND_COLS, dtype=torch.int32), torch.tensor(HAND_VALS, dtype=torch.float32)


def _padded(paths, k, H):
    nodes = np.full((k, H + 1), -1, np.int64)
    slots = np.full((k, H), -1, np.int64)
    hops = np.zeros(k, np.int32)
    weight = np.zeros(k, np.float32)
    for r, (nd, sl, w) in enumerate(paths[:k]):
        nodes[r, : len(nd)] = nd
        slots[r, : len(sl)] = sl
        hops[r] = len(sl)
        weight[r] = w
    return nodes, slots, hops, weight


@pytest.mark.parametrize("k", [1, 4, 7])
@pytest.mark.parametrize("H", [1, 2, 3])
def test_reference_on_hand_built_graph(k, H):
    rp, col, val = _hand_csr()
    src = torch.tensor([0, 3, 0, 6])  # a pair with ties, s == t, no path at all, one direct edge
    dst = torch.tensor([5, 3, 7, 7])
    nodes, slots, hops, weight, count, mass = explain_paths_ref(rp, col, val, src, dst, k, H)
    want = [p for p in HAND_PATHS_0_5 if len(p[1]) <= H]
    for j, paths in enumerate([want, [], [], [([6, 7], [12], 1.0)]]):
        n_, s_, h_, w_ = _padded(paths, k, H)
        np.testing.assert_array_equal(nodes[j].numpy(), n_)
        np.testing.assert_array_equal(slots[j].numpy(), s_)
        np.testing.assert_array_equal(hops[j].numpy(), h_)
        np.testing.assert_array_equal(weight[j].numpy(), w_)
    np.testing.assert_array_equal(count[0].numpy(), [1, 2, 3][:H])
    np.testing.assert_array_equal(mass[0].numpy(), [.25, .5, .5625][:H])
    np.testing.assert_array_equal(count[1:3].numpy(), 0)
    np.testing.assert_array_equal(count[3].numpy(), [1, 0, 0][:H])


def test_reference_chunking_does_not_change_the_result():
    rp, col, val = _hand_csr()
    src, dst = torch.tensor([0, 0, 1, 2, 6, 0]), torch.tensor([5, 3, 5, 0, 7, 1])
    a = explain_paths_ref(rp, col, val, src, dst, 5, 3)
    b = explain_paths_ref(rp, col, val, src, dst, 5, 3, max_probes=1)
    for x, y in zip(a, b):
        assert torch.equal(x, y)


# ---------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------


@pytest.fixture(scope="module")
def kb():
    if not torch.cuda.is_available():
        pytest.skip("needs CUDA")
    import kgat_b200

    kgat_b200._lib.load()
    return kgat_b200


def _model_from_golden(g: Golden):
    from kgat_b200.model import KGAT, KGATArgs

    m = KGAT(KGATArgs(user_num=int(g["user_num"]), entity_num=int(g["entity_num"]), relation_num=int(g["relation_num"]),
                      attentive_matrix=g.att_coo()))
    m.load_state_dict(g.params(), strict=False)
    return m.cuda()


def _refresh(m, g: Golden):
    from kgat_b200.model import KGATMode

    cuda = lambda key: torch.from_numpy(np.asarray(g[key])).cuda()  # noqa: E731
    m(cuda("heads"), cuda("relations"), cuda("tails"), cuda("adjacency_relations"), mode=KGATMode.UPDATE_ATTENTION)


def _assert_matches_reference(graph, src, dst, k, H, got):
    ref = explain_paths_ref(graph.row_ptr, graph.col_idx, graph.vals, src, dst, k, H)
    names = ("nodes", "slots", "hops", "weight", "count")
    for name, a, b in zip(names, got[:5], ref[:5]):
        assert a.dtype == b.dtype and torch.equal(a, b), name
    m_ref = ref[5]
    assert got[5].dtype == torch.float32
    assert float(((got[5].double() - m_ref).abs() / m_ref.abs().clamp_min(1e-30)).max()) <= 1e-5
    return ref


@pytest.mark.gpu
@pytest.mark.parametrize("refreshed", [False, True])
def test_golden_graphs_match_reference(kb, golden_model, refreshed):
    g = golden_model
    m = _model_from_golden(g).eval()
    if refreshed:
        _refresh(m, g)
    users, items = int(g["user_num"]), int(g["entity_num"])
    uu, ii = torch.meshgrid(torch.arange(users), torch.arange(items), indexing="ij")
    uu, ii = uu.flatten(), ii.flatten()
    if uu.numel() > 512:
        pick = torch.from_numpy(np.random.default_rng(0).choice(uu.numel(), 512, replace=False))
        uu, ii = uu[pick], ii[pick]
    graph = m._graph()
    for H in (1, 2, 3):
        for k in (1, 7, 64):
            ex = m.explain(uu, ii, k=k, max_hops=H)
            got = (ex.nodes, ex.slots, ex.hops, ex.weight, ex.count, ex.mass)
            _assert_matches_reference(graph, uu.cuda(), ii.cuda() + users, k, H, got)


@pytest.mark.gpu
def test_amazon_book_scale_with_hub_items(kb):
    from kgat_b200 import ops, synthetic
    from kgat_b200.graph import AttentiveGraph
    from kgat_b200.trainer import attentive_coo

    g = synthetic.make_ckg("amazon-book", with_dicts=False)
    graph = AttentiveGraph.from_sparse_coo(attentive_coo(g).cuda())
    in_deg = (graph.t_ptr[1:] - graph.t_ptr[:-1])[g.user_num : g.user_num + g.item_num]
    hubs = torch.topk(in_deg, 32).indices + g.user_num
    rng = np.random.default_rng(1)
    items = torch.cat([hubs.cpu(), torch.from_numpy(rng.integers(0, g.item_num, 224)) + g.user_num])
    users = torch.from_numpy(rng.integers(0, g.user_num, 256))
    src, dst = users.cuda(), items.cuda()
    got = ops.explain_paths(graph, src, dst, 10, 3)
    ref = _assert_matches_reference(graph, src, dst, 10, 3, got)
    assert int(ref[4].sum()) > 0


@pytest.mark.gpu
def test_slots_index_the_coo_view(kb, golden_small):
    g = golden_small
    m = _model_from_golden(g).eval()
    _refresh(m, g)
    users, items = int(g["user_num"]), int(g["entity_num"])
    u = torch.arange(users).repeat_interleave(4)
    i = torch.arange(4 * users) % items
    ex = m.explain(u, i, k=16, max_hops=3)
    idx, val = m.attentive_matrix.data.indices(), m.attentive_matrix.data.values()
    assert int((ex.hops > 0).sum()) > 0
    w = val[ex.slots[..., 0].clamp(min=0)]
    for j in range(3):
        has = ex.hops > j
        sl = ex.slots[..., j][has]
        assert torch.equal(idx[0, sl], ex.nodes[..., j][has]) and torch.equal(idx[1, sl], ex.nodes[..., j + 1][has])
        if j:
            w = torch.where(has, w * val[ex.slots[..., j].clamp(min=0)], w)
    found = ex.hops > 0
    assert torch.equal(w[found], ex.weight[found])


@pytest.mark.gpu
def test_invariants(kb, golden_tiny):
    g = golden_tiny
    m = _model_from_golden(g).eval()
    users, items = int(g["user_num"]), int(g["entity_num"])
    u = torch.arange(users).repeat_interleave(items)
    i = torch.arange(items).repeat(users)
    a, b = m.explain(u, i, k=64, max_hops=3), m.explain(u.cuda().int(), i.cuda(), k=64, max_hops=3)
    for f in ("nodes", "slots", "hops", "weight", "count", "mass"):
        assert torch.equal(getattr(a, f), getattr(b, f)), f
    # k above the number of paths: padded as specified
    n_paths = a.count.sum(1)
    assert int(n_paths.min()) < 64
    r = torch.arange(64, device=a.hops.device)
    missing = r[None, :] >= n_paths[:, None]
    assert bool((a.hops[missing] == 0).all() and (a.weight[missing] == 0).all())
    assert bool((a.nodes[missing] == -1).all() and (a.slots[missing] == -1).all())
    assert bool((a.hops[~missing] > 0).all())
    # default max_hops = min(3, layers)
    assert m.explain([0], [0]).count.shape == (1, min(3, len(m._aggregator_layers)))
    # empty
    e = m.explain(torch.zeros(0, dtype=torch.int64), torch.zeros(0, dtype=torch.int64), k=5, max_hops=2)
    assert e.nodes.shape == (0, 5, 3) and e.slots.shape == (0, 5, 2) and e.hops.shape == (0, 5)
    assert e.weight.shape == (0, 5) and e.count.shape == (0, 2) and e.mass.shape == (0, 2)
    # bad arguments
    for bad_u, bad_i in (([users], [0]), ([-1], [0]), ([0], [items]), ([0], [-1])):
        with pytest.raises(ValueError):
            m.explain(bad_u, bad_i)
    for k in (0, 65):
        with pytest.raises(ValueError):
            m.explain([0], [0], k=k)
    for h in (0, 4):
        with pytest.raises(ValueError):
            m.explain([0], [0], max_hops=h)
    with pytest.raises(ValueError):
        m.explain([0, 1], [0])
    from kgat_b200 import ops

    with pytest.raises(ValueError):
        ops.explain_paths(m._graph(), torch.tensor([0], device="cuda"), torch.tensor([m.node_num], device="cuda"), 3, 3)


@pytest.mark.gpu
def test_explain_does_not_disturb_training(kb):
    """CF steps, then KG steps with ``explain`` calls inside the deferred KG phase: parameters, losses and torch's RNG state
    are bitwise those of the same run without the calls."""
    from kgat_b200 import synthetic
    from kgat_b200.model import KGATMode
    from kgat_b200.trainer import EpochData, build_model

    g = synthetic.make_ckg("small", seed=11)
    data = EpochData.sample(g, seed=3, n_cf=4, n_kg=12).tensors(device="cuda")
    users = torch.arange(8)
    items = torch.arange(8) * 3
    out = {}
    for call in (False, True):
        m = build_model(g, "cuda", seed=5).train()
        losses = []
        for i in range(4):
            loss = m(*(t[i] for t in data.cf), mode=KGATMode.TRAIN_CF)
            loss.backward()
            m.update_cf_weights()
            losses.append(loss.detach().clone())
        for i in range(12):
            loss = m(*(t[i] for t in data.kg), mode=KGATMode.TRAIN_KG)
            loss.backward()
            m.update_kg_weights()
            losses.append(loss.detach().clone())
            if call and i % 3 == 1:
                d = m._kg_optimizer.deferred
                active = d is not None and d.active
                m.explain(users, items, k=5)
                assert (d is not None and d.active) == active
        rng = torch.get_rng_state().clone(), torch.cuda.get_rng_state().clone()
        sd = {k: v.clone() for k, v in m.state_dict().items() if not v.is_sparse}
        out[call] = (torch.stack(losses), sd, rng)
    a, b = out[False], out[True]
    assert torch.equal(a[0], b[0])
    for k in a[1]:
        assert torch.equal(a[1][k], b[1][k]), k
    assert torch.equal(a[2][0], b[2][0]) and torch.equal(a[2][1], b[2][1])

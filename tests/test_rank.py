"""Exact full ranking of held-out targets (``kgat_rank_targets``, ``ops.rank_targets``, ``KGAT.rank``) and the full-ranking
metrics built on it (``metrics.rank_metrics``), against the torch reference ``oracle/rank_ref.py`` fed the bit-exact
``PREDICT`` scores, against ``KGAT.recommend`` and against ``metrics.evaluate``."""

from __future__ import annotations

from types import SimpleNamespace

import numpy as np
import pytest
import torch

from conftest import Golden
from oracle import kgat_oracle as O
from oracle.rank_ref import auc_pairs, rank_ref

# ---------------------------------------------------------------------------------------------
# CPU: the reference on a hand-built case, the closed-form AUC, and the metrics
# ---------------------------------------------------------------------------------------------
NAN = float("nan")
# item ids 0-6; items = arange(6), so item 6 is never a candidate
SCORES = [[1.0, 1.0, 0.5, 0.0, -0.0, NAN, 3.0],  # user 0: NaN first, then 1 (pos 0) before 1 (pos 1), .5, +0, -0
          [0.0, 1.0, 2.0, 3.0, 4.0, 5.0, 6.0],   # user 1
          [1.0, 1.0, 1.0, 1.0, 1.0, 1.0, 1.0]]   # user 2: no targets


def _csr(lists):
    ptr = torch.tensor(np.concatenate([[0], np.cumsum([len(x) for x in lists])]), dtype=torch.int32)
    return ptr, torch.tensor([i for x in lists for i in x], dtype=torch.int32)


def _hand(users, items, exclude=True):
    s = torch.tensor(SCORES)[users]
    t_ptr, t_items = _csr([[1, 4, 6], [0, 2], []])
    e_ptr, e_items = _csr([[0], [2], []]) if exclude else (None, None)
    return rank_ref(s, users, items, t_ptr, t_items, e_ptr, e_items)


def test_reference_ties_nan_signed_zero_exclusion_and_repeats():
    ptr, items, scores, rank, eligible = _hand(torch.tensor([0, 1, 2, 0]), torch.arange(6))
    assert ptr.tolist() == [0, 3, 5, 5, 8]
    assert items.tolist() == [1, 4, 6, 0, 2, 1, 4, 6]
    # user 0: item 0 is excluded, so item 1 is beaten by the NaN only; -0 by NaN, 1, .5 and +0; item 6 is not a candidate.
    # user 1: its target 2 is excluded; target 0 is beaten by 5, 4, 3, 1.
    assert rank.tolist() == [1, 4, -1, 4, -1, 1, 4, -1]
    assert eligible.tolist() == [5, 5, 6, 5]
    assert scores.view(torch.int32).tolist() == torch.tensor([1.0, -0.0, 3.0, 0.0, 2.0, 1.0, -0.0, 3.0]).view(torch.int32).tolist()
    # without exclusion: item 0 (position 0) now ties item 1 and goes first
    _, _, _, rank, eligible = _hand(torch.tensor([0, 1]), torch.arange(6), exclude=False)
    assert rank.tolist() == [2, 5, -1, 5, 3] and eligible.tolist() == [6, 6]
    # the tie order is the position in `items`: item 1 before item 0 now; item 4 is missing from the candidates
    _, _, _, rank, eligible = _hand(torch.tensor([0]), torch.tensor([1, 0, 2, 3, 5]), exclude=False)
    assert rank.tolist() == [1, -1, -1] and eligible.tolist() == [5]


def _random_case(seed, U=30, n=200, per_train=10, per_test=6):
    rng = np.random.default_rng(seed)
    scores = torch.from_numpy((np.round(rng.standard_normal((U, n)) * 4) / 4 + 0.125).astype(np.float32))  # many ties, no zeros
    train = {u: sorted(set(rng.integers(0, n, per_train).tolist())) for u in range(U)}
    test = {u: sorted(set(rng.integers(0, n, rng.integers(0, per_test + 1)).tolist())) for u in range(U)}
    return scores, train, test


def test_closed_form_auc_equals_pair_counting():
    scores, train, test = _random_case(5)
    U, n = scores.shape
    tp, ti = _csr([test[u] for u in range(U)])
    ep, ei = _csr([train[u] for u in range(U)])
    for items in (torch.arange(n), torch.from_numpy(np.random.default_rng(6).permutation(n)[: n - 20])):
        ptr, _, _, rank, eligible = rank_ref(scores, torch.arange(U), items, tp, ti, ep, ei)
        n_checked = 0
        for b in range(U):
            r = torch.sort(rank[ptr[b] : ptr[b + 1]]).values
            r = r[r >= 0]
            P, N = r.numel(), int(eligible[b]) - r.numel()
            want = auc_pairs(scores[b], items, test[b], train[b])
            if P == 0 or N == 0:
                assert np.isnan(want)
                continue
            got = 1.0 - float((r - torch.arange(P)).sum()) / (P * N)
            assert abs(got - want) < 1e-12, (b, got, want)
            n_checked += 1
        assert n_checked > U // 2


def test_metrics_from_reference_ranks_equal_metrics_at_k():
    from kgat_b200.metrics import metrics_from_ranks

    scores, train, test = _random_case(7)
    U, n = scores.shape
    users = np.array([u for u in range(U) if test[u]])
    tp, ti = _csr([test[u] for u in range(U)])
    ep, ei = _csr([train[u] for u in range(U)])
    ptr, _, _, rank, eligible = rank_ref(scores[users], torch.from_numpy(users), torch.arange(n), tp, ti, ep, ei)
    k_list = [1, 5, 20, 150]
    got = metrics_from_ranks(SimpleNamespace(ptr=ptr, rank=rank, eligible=eligible), np.array([len(test[u]) for u in users]), k_list)
    ref = O.metrics_at_k(scores[users], train, test, users, n, k_list)
    idx = O.rank_items(scores[users], train, users).numpy()
    pos = np.zeros((len(users), n), bool)
    for i, u in enumerate(users):
        pos[i, test[int(u)]] = True
    hits = np.take_along_axis(pos, idx, axis=1)
    for j, k in enumerate(k_list):
        for m, name in enumerate(("precision", "recall", "ndcg")):
            want = float(np.mean(ref[k][name]))  # the restatement works in fp32
            assert abs(float(got[4 * j + m]) - want) <= 1e-6 * abs(want) + 1e-9, (k, name)
        assert float(got[4 * j + 3]) == float(np.mean(hits[:, :k].any(1)))
    # mrr and mean rank straight from the definition
    first, mean_rank = [], []
    for i, u in enumerate(users):
        r = rank[ptr[i] : ptr[i + 1]]
        r = r[r >= 0].double()
        first.append(1.0 / (1.0 + float(r.min())) if r.numel() else 0.0)
        if r.numel():
            mean_rank.append(float(r.mean()))
    assert abs(float(got[-3]) - np.mean(first)) < 1e-12
    assert abs(float(got[-1]) - np.mean(mean_rank)) < 1e-9


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
    return m.cuda().eval()


_CF = {}


def _codeforces_sm():
    if not _CF:
        from kgat_b200 import synthetic
        from kgat_b200.trainer import build_model

        g = synthetic.make_ckg("codeforces-sm")
        _CF["g"], _CF["m"] = g, build_model(g, "cuda").eval()
    return _CF["g"], _CF["m"]


def _csr_cuda(lists, user_num, item_num):
    from kgat_b200.metrics import InteractionCSR

    pairs = np.array([(u, i) for u, x in lists.items() for i in x], dtype=np.int64).reshape(-1, 2)
    return InteractionCSR(pairs, user_num, item_num, "cuda")


def _predict(m, users, n):
    from kgat_b200.model import KGATMode

    with torch.no_grad():
        return m(users.cuda(), torch.arange(n).cuda(), mode=KGATMode.PREDICT)


def _assert_equals_reference(m, users, items, targets, exclude, n_scores):
    got = m.rank(users, items, targets, exclude=exclude)
    cand = torch.arange(items) if isinstance(items, int) else items
    s = _predict(m, users, n_scores)
    want = rank_ref(s, users, cand, targets.ptr_dev, targets.items, *((exclude.ptr_dev, exclude.items) if exclude is not None else ()))
    assert torch.equal(got.ptr, want[0]) and torch.equal(got.items, want[1])
    assert torch.equal(got.scores.view(torch.int32), want[2].view(torch.int32))  # bit-identical to PREDICT
    assert torch.equal(got.rank, want[3])
    assert torch.equal(got.eligible, want[4])
    return got


@pytest.mark.gpu
def test_ranks_equal_reference_on_golden_models(kb, golden_model):
    g = golden_model
    m = _model_from_golden(g)
    U, n = int(g["user_num"]), int(g["item_num"])
    rng = np.random.default_rng(11)
    targets = _csr_cuda({u: rng.integers(0, n, 6).tolist() for u in range(U)}, U, n)
    exclude = _csr_cuda({u: rng.integers(0, n, 8).tolist() for u in range(U)}, U, n)
    users = torch.cat([torch.arange(U), torch.tensor([0, U - 1, 0])])
    subset = torch.from_numpy(rng.permutation(n)[: 3 * n // 4])
    for items in (n, subset):
        for ex in (None, exclude):
            got = _assert_equals_reference(m, users, items, targets, ex, n)
            assert bool((got.rank >= 0).any()) and bool((got.rank == -1).any() == (ex is not None or not isinstance(items, int)))


@pytest.mark.gpu
@pytest.mark.parametrize("subset", [False, True])
def test_ranks_equal_reference_on_codeforces_sm(kb, subset):
    g, m = _codeforces_sm()
    train = _csr_cuda(g.train_dict, g.user_num, g.item_num)
    test = _csr_cuda(g.test_dict, g.user_num, g.item_num)
    items = torch.from_numpy(np.random.default_rng(12).permutation(g.item_num)[:7000]) if subset else g.item_num
    for ex in (None, train):
        got = _assert_equals_reference(m, torch.arange(g.user_num), items, test, ex, g.item_num)
        assert int(got.items.numel()) == int(test.counts.sum())


@pytest.mark.gpu
def test_rank_is_the_position_in_recommend(kb):
    """rank < 128  <=>  the target sits at rec.items[b, rank] of recommend(k = 128), in both directions."""
    g, m = _codeforces_sm()
    train = _csr_cuda(g.train_dict, g.user_num, g.item_num)
    test = _csr_cuda(g.test_dict, g.user_num, g.item_num)
    users = torch.arange(g.user_num)
    for items in (g.item_num, torch.from_numpy(np.random.default_rng(13).permutation(g.item_num)[:5000])):
        r = m.rank(users, items, test, exclude=train)
        rec = m.recommend(users, items, k=128, exclude=train)
        b = torch.repeat_interleave(torch.arange(g.user_num, device="cuda"), r.ptr.diff())
        top = (r.rank >= 0) & (r.rank < 128)
        assert int(top.sum()) > 100
        assert torch.equal(rec.items[b[top], r.rank[top]], r.items[top])
        assert torch.equal(rec.scores[b[top], r.rank[top]].view(torch.int32), r.scores[top].view(torch.int32))
        listed = test.contains(users.cuda()[:, None].expand(-1, 128), rec.items) & (rec.items >= 0)
        assert int(listed.sum()) == int(top.sum())  # every target recommended has a rank < 128 (the ranks are then distinct)
        assert torch.equal(r.eligible.clamp(max=128), rec.count.long())


def _evaluate_hits(m, train, test, users, k_list):
    from kgat_b200.metrics import evaluate

    res, top = evaluate(m, train, test, k_list=k_list, users=users)
    u = torch.from_numpy(users).cuda()[:, None].expand_as(top)
    hits = test.contains(u, top)
    return res, {k: hits[:, :k].sum(1) for k in k_list}


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["golden_small", "codeforces-sm"])
def test_rank_metrics_match_evaluate(kb, which):
    from kgat_b200.metrics import rank_metrics

    if which == "golden_small":
        g = Golden("model_small.npz")
        m = _model_from_golden(g)
        U, n = int(g["user_num"]), int(g["item_num"])
        train, test = _csr_cuda(g.ragged("train_dict"), U, n), _csr_cuda(g.ragged("test_dict"), U, n)
        k_list = (20, 40, 100)
    else:
        cf, m = _codeforces_sm()
        U, n = cf.user_num, cf.item_num
        train, test = _csr_cuda(cf.train_dict, U, n), _csr_cuda(cf.test_dict, U, n)
        k_list = (20, 40, 60, 80, 100)
    counts = np.diff(test.ptr_host)
    elig = n - np.diff(train.ptr_host)
    users = np.nonzero((counts > 0) & (elig >= max(k_list)))[0]
    assert users.size > 10
    res, hits = _evaluate_hits(m, train, test, users, k_list)
    got = rank_metrics(m, train, test, k_list=k_list, users=users)
    r = m.rank(torch.from_numpy(users), n, test, exclude=train)
    b = torch.repeat_interleave(torch.arange(users.size, device="cuda"), r.ptr.diff())
    for k in k_list:
        h = torch.zeros(users.size, dtype=torch.int64, device="cuda").index_add_(0, b, ((r.rank >= 0) & (r.rank < k)).long())
        assert torch.equal(h, hits[k].long()), k  # hit counts exactly
        assert got[k]["hit"] == float((hits[k] > 0).double().mean())
        for name in ("precision", "recall", "ndcg"):
            assert abs(got[k][name] - res[k][name]) <= 1e-6 * abs(res[k][name]) + 1e-12, (k, name, got[k][name], res[k][name])
    assert 0.0 < got["mrr"] <= 1.0 and 0.0 < got["auc"] < 1.0 and got["mean_rank"] >= 0.0
    # the default user list is every user with a test item, as evaluate's; k beyond 128 is allowed
    all_users = rank_metrics(m, train, test, k_list=(20, 1000))
    assert 0.0 <= all_users[1000]["recall"] <= 1.0 and all_users[1000]["hit"] >= all_users[20]["hit"]


@pytest.mark.gpu
def test_result_does_not_depend_on_the_split(kb):
    from kgat_b200 import ops

    g, m = _codeforces_sm()
    train = _csr_cuda(g.train_dict, g.user_num, g.item_num)
    test = _csr_cuda(g.test_dict, g.user_num, g.item_num)
    tables = m._tables()
    users = torch.arange(130).repeat(2)
    cand = torch.from_numpy(np.random.default_rng(14).permutation(g.item_num))
    for items in (g.item_num, cand):
        outs = [ops.rank_targets(tables, users, items, test.ptr_dev, test.items, train.ptr_dev, train.items, slices=s)
                for s in (1, 2, 7, 64, None, None)]
        for o in outs[1:]:
            for a, b in zip(o, outs[0]):
                assert torch.equal(a.view(torch.int32) if a.dtype == torch.float32 else a, b.view(torch.int32) if b.dtype == torch.float32 else b)
        ptr, rank = outs[0][0], outs[0][3]
        assert torch.equal(rank[: ptr[130]], rank[ptr[130] :])
    got = [m.rank(users, g.item_num, test, exclude=train) for _ in range(2)]
    assert all(torch.equal(getattr(got[0], f), getattr(got[1], f)) for f in ("ptr", "items", "rank", "eligible"))
    from kgat_b200.metrics import rank_metrics

    assert rank_metrics(m, train, test) == rank_metrics(m, train, test)


@pytest.mark.gpu
def test_heavy_user_keeps_its_keys_in_global_memory(kb):
    """A user with more than 6,000 targets: the 64-user tile's keys do not fit in shared memory."""
    g, m = _codeforces_sm()
    rng = np.random.default_rng(15)
    lists = {u: list(v) for u, v in g.test_dict.items()}
    lists[3] = rng.choice(g.item_num, 6500, replace=False).tolist()
    targets = _csr_cuda(lists, g.user_num, g.item_num)
    train = _csr_cuda(g.train_dict, g.user_num, g.item_num)
    users = torch.arange(100)
    assert int(targets.counts[:64].sum()) > 6000
    for items in (g.item_num, torch.from_numpy(rng.permutation(g.item_num)[:8000])):
        got = _assert_equals_reference(m, users, items, targets, train, g.item_num)
        row = got.rank[got.ptr[3] : got.ptr[4]]
        assert int((row >= 0).sum()) > 4000 and torch.equal(torch.sort(row[row >= 0]).values.unique(), torch.sort(row[row >= 0]).values)


@pytest.mark.gpu
def test_argument_errors(kb, golden_tiny):
    from kgat_b200 import ops
    from kgat_b200.metrics import InteractionCSR, rank_metrics

    g = golden_tiny
    m = _model_from_golden(g)
    users, ent, items = int(g["user_num"]), int(g["entity_num"]), int(g["item_num"])
    t = _csr_cuda({0: [1, 2], 2: [5]}, users, items)
    u = torch.arange(3)
    bad = [
        dict(user_ids=torch.tensor([users]), items=items),
        dict(user_ids=torch.tensor([-1]), items=items),
        dict(user_ids=u, items=torch.tensor([0, ent])),
        dict(user_ids=u, items=torch.tensor([-1, 2])),
        dict(user_ids=u, items=ent + 1),
        dict(user_ids=u, items=-1),
        dict(user_ids=u, items=torch.tensor([3, 1, 3])),
        dict(user_ids=u, items=items, exclude=InteractionCSR(np.array([[0, 1]]), users + 1, items, "cuda")),
        dict(user_ids=u, items=items, targets=InteractionCSR(np.array([[0, 1]]), users + 1, items, "cuda")),
        dict(user_ids=u, items=items, targets=InteractionCSR(np.array([[0, 1]]), users, ent + 1, "cuda")),
        dict(user_ids=u[None, :], items=items),
        dict(user_ids=u, items=torch.arange(items)[None, :]),
        dict(user_ids=u.float(), items=items),
        dict(user_ids=u, items=torch.arange(4).float()),
    ]
    for kw in bad:
        kw.setdefault("targets", t)
        with pytest.raises(ValueError):
            m.rank(**kw)
    tables = m._tables()
    n = tables[0].shape[0]
    for args, kw in (((torch.tensor([n]), 4), {}), ((u, torch.tensor([n])), {}), ((u, torch.tensor([1, 1])), {}), ((u, 4), dict(slices=0)),
                     ((u, 4), dict(slices=65)), ((u, n + 1), {})):
        with pytest.raises(ValueError):
            ops.rank_targets(tables, *args, t.ptr_dev, t.items, **kw)
    with pytest.raises(ValueError):  # a user row beyond the target pointer
        ops.rank_targets(tables, torch.tensor([users]), 4, t.ptr_dev, t.items)
    with pytest.raises(ValueError):  # a target id beyond the tables
        ops.rank_targets(tables, u, 4, torch.tensor([0, 1, 1, 1], dtype=torch.int32, device="cuda"), torch.tensor([n], dtype=torch.int32, device="cuda"))
    with pytest.raises(ValueError):
        ops.rank_targets(tables, u, 4, t.ptr_dev, t.items, exclude_ptr=t.ptr_dev)
    with pytest.raises(ValueError):
        rank_metrics(m, t, t, k_list=(0, 20))
    # empty inputs
    r = m.rank(torch.zeros(0, dtype=torch.int64), items, t)
    assert r.ptr.tolist() == [0] and r.items.numel() == 0 and r.eligible.numel() == 0
    r = m.rank(torch.tensor([1]), items, t)  # a user without targets
    assert r.ptr.tolist() == [0, 0] and r.eligible.tolist() == [items]
    r = m.rank(torch.tensor([0, 2]), 0, t)  # no candidates at all
    assert r.rank.tolist() == [-1, -1, -1] and r.eligible.tolist() == [0, 0]


@pytest.mark.gpu
def test_yelp2018_shape_all_users_in_one_call(kb):
    """C4: every user with a test item, in one call; hit counts equal evaluate's top-100 at every k."""
    from kgat_b200 import synthetic
    from kgat_b200.metrics import InteractionCSR, rank_metrics
    from kgat_b200.trainer import build_model

    g = synthetic.make_ckg("yelp2018")
    m = build_model(g, "cuda").eval()
    train = InteractionCSR(g.train_interactions, g.user_num, g.item_num, "cuda")
    test = InteractionCSR(g.test_dict, g.user_num, g.item_num, "cuda")
    users = np.nonzero(np.diff(test.ptr_host) > 0)[0]
    k_list = (20, 40, 60, 80, 100)
    res, hits = _evaluate_hits(m, train, test, users, k_list)
    r = m.rank(torch.from_numpy(users), g.item_num, test, exclude=train)
    b = torch.repeat_interleave(torch.arange(users.size, device="cuda"), r.ptr.diff())
    for k in k_list:
        h = torch.zeros(users.size, dtype=torch.int64, device="cuda").index_add_(0, b, ((r.rank >= 0) & (r.rank < k)).long())
        assert torch.equal(h, hits[k].long()), k
    got = rank_metrics(m, train, test, k_list=k_list)
    for k in k_list:
        for name in ("precision", "recall", "ndcg"):
            assert abs(got[k][name] - res[k][name]) <= 1e-6 * abs(res[k][name]) + 1e-12, (k, name)

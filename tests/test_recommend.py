"""Filtered top-k recommendations (``kgat_recommend_filter`` / ``kgat_recommend_topk``, ``ops.recommend_filter`` /
``ops.recommend_topk_fused``, ``KGAT.recommend``) against the torch reference ``oracle/recommend_ref.py`` and against the
materialised path ``KGAT.recommend_topk``.  Scores must be bit-identical to ``recommend_topk``'s; the reference sums in
another order, so it is compared on indices away from near-ties."""

from __future__ import annotations

import numpy as np
import pytest
import torch

from conftest import Golden
from oracle.recommend_ref import filter_ref, recommend_ref

# ---------------------------------------------------------------------------------------------
# CPU: the reference on a hand-built CKG whose answers are written out below
# ---------------------------------------------------------------------------------------------
# 3 users (nodes 0-2); entities 0-4 are problems (nodes 3-7), 5-6 tags, 7-8 ratings, 9 a contest (nodes 8-12).
#   problem 0: tag 5, rating 7, contest 9      problem 1: tag 5, rating 8      problem 2: tag 6, rating 7
#   problem 3: tag 5 (no rating)               problem 4: tag 6, rating 8, contest 9
# Scores use table row p for problem p (quirk Q4), so problems 0-2 share the users' rows.  Power-of-two values make every
# score exact and give ties:
#   user 0 [1, 0]: p0 1, p1 0, p2 1, p3 .5, p4 2
#   user 1 [0, 1]: p0 0, p1 1, p2 1, p3 .5, p4 0
#   user 2 [1, 1]: p0 1, p1 1, p2 2, p3 1,  p4 2
USER_NUM, ENTITY_NUM = 3, 10
LINKS = {0: [5, 7, 9], 1: [5, 8], 2: [6, 7], 3: [5], 4: [6, 8, 9]}
TABLE = [[1, 0], [0, 1], [1, 1], [.5, .5], [2, 0]]


def _hand_ckg():
    n = USER_NUM + ENTITY_NUM
    edges = set()
    for p, ents in LINKS.items():
        for e in ents:
            edges.add((USER_NUM + p, USER_NUM + e))
            edges.add((USER_NUM + e, USER_NUM + p))
    edges |= {(0, USER_NUM + 0), (1, USER_NUM + 2), (2, USER_NUM + 4)}  # user -> problem entries play no part in the filter
    rows, cols = np.array(sorted(edges)).T
    row_ptr = torch.from_numpy(np.concatenate([[0], np.cumsum(np.bincount(rows, minlength=n))]).astype(np.int32))
    table = torch.zeros(n, 4)
    table[: len(TABLE), :2] = torch.tensor(TABLE)
    return row_ptr, torch.from_numpy(cols.astype(np.int32)), table


def _exclude(lists):
    ptr = torch.tensor(np.concatenate([[0], np.cumsum([len(x) for x in lists])]), dtype=torch.int32)
    return ptr, torch.tensor([i for x in lists for i in x], dtype=torch.int32)


def _check(got, items, scores):
    it, sc, cnt = got
    want_cnt = [sum(1 for x in row if x >= 0) for row in items]
    assert it.tolist() == items
    assert cnt.tolist() == want_cnt
    for b, row in enumerate(scores):
        assert sc[b, : want_cnt[b]].tolist() == row
        assert bool((sc[b, want_cnt[b] :] == float("-inf")).all())


def test_reference_ranking_ties_and_repeats():
    rp, col, table = _hand_ckg()
    users = torch.tensor([0, 1, 2, 0])
    got = recommend_ref(table, users, torch.arange(5), 3)
    _check(got, [[4, 0, 2], [1, 2, 3], [2, 4, 0], [4, 0, 2]], [[2, 1, 1], [1, 1, .5], [2, 2, 1], [2, 1, 1]])
    # the tie order is the position in `items`, not the id
    got = recommend_ref(table, torch.tensor([2]), torch.tensor([4, 3, 2, 1, 0]), 3)
    _check(got, [[4, 2, 3]], [[2, 2, 1]])


def test_reference_filter_groups():
    rp, col, _ = _hand_ckg()
    items = torch.arange(5)
    f = lambda groups: filter_ref(rp, col, items, groups, USER_NUM).tolist()  # noqa: E731
    assert f([[5], [7, 8]]) == [0, 1]  # AND across groups, OR within: tag 5 and a rating (problem 3 has none)
    assert f([[9]]) == [0, 4]
    assert f([[6, 9]]) == [0, 2, 4]
    assert f([[7], [8]]) == []
    assert f([]) == [0, 1, 2, 3, 4]
    assert filter_ref(rp, col, torch.tensor([4, 2, 0]), [[6]], USER_NUM).tolist() == [0, 1]  # positions, input order


def test_reference_exclusion_filter_and_padding():
    rp, col, table = _hand_ckg()
    ptr, ex = _exclude([[0], [], [4, 2]])
    users = torch.tensor([0, 1, 2])
    got = recommend_ref(table, users, torch.arange(5), 3, ptr, ex)
    _check(got, [[4, 2, 3], [1, 2, 3], [0, 1, 3]], [[2, 1, .5], [1, 1, .5], [1, 1, 1]])
    got = recommend_ref(table, users, torch.arange(5), 3, ptr, ex, groups=[[5], [7, 8]], row_ptr=rp, col_idx=col, user_num=USER_NUM)
    _check(got, [[1, -1, -1], [1, 0, -1], [0, 1, -1]], [[0], [1, 0], [1, 1]])
    got = recommend_ref(table, users, torch.arange(5), 3, groups=[[7], [8]], row_ptr=rp, col_idx=col, user_num=USER_NUM)
    _check(got, [[-1] * 3] * 3, [[], [], []])


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


def _codeforces_sm():
    from kgat_b200 import synthetic
    from kgat_b200.trainer import build_model

    g = synthetic.make_ckg("codeforces-sm", with_dicts=False)
    return g, build_model(g, "cuda").eval()


def _cf_entities(g):
    """First entity id of each Codeforces block (synthetic._codeforces_triples): contests, divisions, tags, ratings."""
    c0 = g.item_num
    d0 = c0 + 1_913
    t0 = d0 + 5
    return c0, d0, t0, t0 + 37


def _random_exclusion(user_num, item_num, seed, per_user=6):
    from kgat_b200.metrics import InteractionCSR

    rng = np.random.default_rng(seed)
    pairs = np.stack([np.repeat(np.arange(user_num), per_user), rng.integers(0, item_num, user_num * per_user)], 1)
    return InteractionCSR(pairs, user_num, item_num, "cuda")


def _materialised(m, users, cand, k, exclude):
    """recommend_topk over the same candidates, with the exclusion turned into column positions; + eligible counts."""
    pos_of = {int(c): j for j, c in enumerate(cand.tolist())}
    ptr, flat, n_elig = [0], [], []
    for u in users.tolist():
        cols = sorted(pos_of[i] for i in exclude.items[exclude.ptr_host[u] : exclude.ptr_host[u + 1]].tolist() if i in pos_of)
        flat += cols
        ptr.append(len(flat))
        n_elig.append(cand.numel() - len(cols))
    idx, val = m.recommend_topk(users.cuda(), cand.cuda(), k, torch.tensor(ptr, dtype=torch.int32, device="cuda"),
                                torch.tensor(flat, dtype=torch.int32, device="cuda"), want_values=True)
    return cand.cuda()[idx.long()], val, torch.tensor(n_elig, device="cuda")


def _assert_matches_materialised(m, users, cand, k, exclude, rec):
    items, vals, n_elig = _materialised(m, users, cand, k, exclude)
    assert torch.equal(rec.count.long(), n_elig.clamp(max=k))
    full = n_elig >= k
    assert int(full.sum()) > 0
    assert torch.equal(rec.items[full], items[full])
    assert torch.equal(rec.scores[full].view(torch.int32), vals[full].view(torch.int32))
    r = torch.arange(k, device="cuda")[None, :] < rec.count[:, None]  # short users: the eligible part agrees too
    assert torch.equal(rec.items[r & ~full[:, None]], items[r & ~full[:, None]])


@pytest.mark.gpu
def test_matches_recommend_topk_on_golden_models(kb, golden_model):
    g = golden_model
    m = _model_from_golden(g)
    users, items, ent = int(g["user_num"]), int(g["item_num"]), int(g["entity_num"])
    ex = _random_exclusion(users, items, seed=1)
    u = torch.cat([torch.arange(users), torch.tensor([0, users - 1, 0])])  # repeats
    k = min(20, items - 7)
    rec = m.recommend(u, items, k=k, exclude=ex)
    _assert_matches_materialised(m, u, torch.arange(items), k, ex, rec)
    # with a filter: two groups over the non-item entities, chosen so that some items pass
    from kgat_b200 import ops

    graph = m._graph()
    kg = [e for e in range(items, ent)]
    require = [kg[: len(kg) // 2], kg[len(kg) // 4 :]]
    cand = torch.arange(items)[filter_ref(graph.row_ptr.cpu(), graph.col_idx.cpu(), torch.arange(items), require, users)]
    assert cand.numel() > 0
    k = min(k, cand.numel())
    rec = m.recommend(u, items, k=k, exclude=ex, require=require)
    _, fc, fn = ops.recommend_filter(graph, torch.arange(items), require, users)
    assert torch.equal(fc[: int(fn)].long().cpu(), cand)
    assert cand.numel() >= k + 6  # so every user keeps k eligible candidates after its 6 exclusions
    assert bool((rec.count == k).all())
    _assert_matches_materialised(m, u, cand, k, ex, rec)


@pytest.mark.gpu
@pytest.mark.parametrize("filtered", [False, True])
def test_matches_recommend_topk_on_codeforces_sm(kb, filtered):
    g, m = _codeforces_sm()
    c0, d0, t0, r0 = _cf_entities(g)
    from kgat_b200.metrics import InteractionCSR

    ex = InteractionCSR(g.train_interactions, g.user_num, g.item_num, "cuda")
    users = torch.arange(g.user_num)
    require = [list(range(r0 + 8, r0 + 14)), [t0, t0 + 1, t0 + 2]] if filtered else None
    cand = torch.arange(g.item_num)
    if filtered:
        graph = m._graph()
        cand = cand[filter_ref(graph.row_ptr.cpu(), graph.col_idx.cpu(), cand, require, g.user_num)]
        assert 20 < cand.numel() < g.item_num
    rec = m.recommend(users, g.item_num, k=20, exclude=ex, require=require)
    _assert_matches_materialised(m, users, cand, 20, ex, rec)
    # the reference agrees on indices away from near-ties
    table = torch.cat(m._tables(), 1)
    r_items, r_scores, r_count = recommend_ref(table, users, torch.arange(g.item_num), 21, ex.ptr_dev, ex.items, groups=require,
                                               row_ptr=m._graph().row_ptr, col_idx=m._graph().col_idx, user_num=g.user_num)
    assert torch.equal(r_count.clamp(max=20), rec.count)
    tol = 1e-5 * float(r_scores[torch.isfinite(r_scores)].abs().max())
    apart = (r_scores[:, :-1] - r_scores[:, 1:]) > tol  # rank j is clear of rank j + 1
    safe = apart & torch.cat([torch.ones_like(apart[:, :1]), apart[:, :-1]], 1)
    agree = rec.items == r_items[:, :20]
    assert bool((agree | ~safe).all()) and float(agree.float().mean()) > 0.95


@pytest.mark.gpu
def test_filter_kernel_equals_reference(kb):
    from kgat_b200 import ops

    g, m = _codeforces_sm()
    c0, d0, t0, r0 = _cf_entities(g)
    graph = m._graph()
    rp, col = graph.row_ptr.cpu(), graph.col_idx.cpu()
    perm = torch.from_numpy(np.random.default_rng(3).permutation(g.item_num))
    used = set(np.unique(g.tails).tolist())
    unused_contest = next(c for c in range(c0, d0) if g.user_num + c not in used)
    cases = [
        [[t0, t0 + 3, t0 + 7]],                        # a group of tags
        [list(range(r0 + 5, r0 + 12))],                # a contiguous rating range
        [[c0 + 17]],                                   # one contest
        [[d0]],                                        # a division: linked to contests, never to a problem
        [[unused_contest]],                            # an entity with no edges at all
        [[t0, t0 + 1], list(range(r0, r0 + 28))],      # tags AND any rating
        [[t0 + 2], [r0 + 10, r0 + 11], list(range(c0, c0 + 1000))],
    ]
    empty = {3, 4}
    for items in (torch.arange(g.item_num), perm, perm[:1000].cuda().int()):
        for groups in cases:
            pos, cand, n = ops.recommend_filter(graph, items, groups, g.user_num)
            want = filter_ref(rp, col, items.cpu(), groups, g.user_num)
            n = int(n)
            assert n == want.numel()
            assert torch.equal(pos[:n].long().cpu(), want)
            assert torch.equal(cand[:n].long().cpu(), items.cpu().long()[want])
            if items.numel() == g.item_num:
                assert (n == 0) == (cases.index(groups) in empty)


@pytest.mark.gpu
def test_result_does_not_depend_on_the_split(kb):
    from kgat_b200 import ops

    g, m = _codeforces_sm()
    ex = _random_exclusion(g.user_num, g.item_num, seed=2, per_user=40)
    tables = m._tables()
    users = torch.arange(130).repeat(2)
    cand = torch.from_numpy(np.random.default_rng(4).permutation(g.item_num))
    for k in (1, 20, 128):
        outs = [ops.recommend_topk_fused(tables, users, cand, k, ex.ptr_dev, ex.items, slices=s) for s in (1, 2, 7, 64, None, None)]
        for o in outs[1:]:
            assert torch.equal(o[0], outs[0][0]) and torch.equal(o[2], outs[0][2])
            assert torch.equal(o[1].view(torch.int32), outs[0][1].view(torch.int32))
        assert torch.equal(outs[0][0][:130], outs[0][0][130:])


@pytest.mark.gpu
def test_count_and_padding(kb, golden_small):
    from kgat_b200.metrics import InteractionCSR

    g = golden_small
    m = _model_from_golden(g)
    users, items = int(g["user_num"]), int(g["item_num"])
    cand = torch.arange(40, 80)
    lists = {0: list(range(40, 80)), 1: list(range(40, 75)), 2: [41, 43]}  # nothing left, 5 left, 38 left
    pairs = np.array([(u, i) for u, x in lists.items() for i in x])
    ex = InteractionCSR(pairs, users, items, "cuda")
    u = torch.tensor([0, 1, 2, 3])
    for k in (1, 5, 20, 128):
        rec = m.recommend(u, cand, k=k, exclude=ex)
        want = torch.tensor([0, min(k, 5), min(k, 38), min(k, 40)], dtype=torch.int32, device="cuda")
        assert torch.equal(rec.count, want)
        r = torch.arange(k, device="cuda")[None, :]
        pad = r >= want[:, None].long()
        assert bool((rec.items[pad] == -1).all()) and bool((rec.scores[pad] == float("-inf")).all())
        assert bool((rec.items[~pad] >= 40).all() & (rec.items[~pad] < 80).all())
        assert set(rec.items[1, : int(want[1])].tolist()) <= set(range(75, 80))
        assert not (set(rec.items[2, : int(want[2])].tolist()) & {41, 43})
        s = rec.scores[~pad].view(-1)
        assert bool(torch.isfinite(s).all())
    rec = m.recommend(torch.tensor([3]), 0, k=5)  # no candidates at all
    assert rec.count.tolist() == [0] and rec.items.tolist() == [[-1] * 5]
    rec = m.recommend(torch.zeros(0, dtype=torch.int64), items, k=5)
    assert rec.items.shape == (0, 5) and rec.scores.shape == (0, 5) and rec.count.shape == (0,)


@pytest.mark.gpu
def test_argument_errors(kb, golden_tiny):
    from kgat_b200 import ops
    from kgat_b200.metrics import InteractionCSR

    g = golden_tiny
    m = _model_from_golden(g)
    users, ent, items = int(g["user_num"]), int(g["entity_num"]), int(g["item_num"])
    u = torch.arange(3)
    bad = [
        dict(user_ids=u, items=items, k=0),
        dict(user_ids=u, items=items, k=129),
        dict(user_ids=torch.tensor([users]), items=items),
        dict(user_ids=torch.tensor([-1]), items=items),
        dict(user_ids=u, items=torch.tensor([0, ent])),
        dict(user_ids=u, items=torch.tensor([-1, 2])),
        dict(user_ids=u, items=ent + 1),
        dict(user_ids=u, items=torch.tensor([3, 1, 3])),
        dict(user_ids=u, items=items, require=[[items], []]),
        dict(user_ids=u, items=items, require=[[ent]]),
        dict(user_ids=u, items=items, exclude=InteractionCSR(np.array([[0, 1]]), users + 1, items, "cuda")),
        dict(user_ids=u[None, :], items=items),
        dict(user_ids=u, items=torch.arange(items)[None, :]),
        dict(user_ids=u.float(), items=items),
    ]
    for kw in bad:
        with pytest.raises(ValueError):
            m.recommend(**kw)
    tables = m._tables()
    n = tables[0].shape[0]
    for args, kw in (((u, torch.tensor([n]), 5), {}), ((torch.tensor([n]), torch.arange(4), 3), {}),
                     ((u, torch.arange(4), 3), dict(slices=65)), ((u, torch.arange(4), 3), dict(slices=0))):
        with pytest.raises(ValueError):
            ops.recommend_topk_fused(tables, *args, **kw)
    with pytest.raises(ValueError):
        ops.recommend_filter(m._graph(), torch.tensor([ent]), [[0]], users)


@pytest.mark.gpu
def test_yelp2018_shape_all_users_in_one_call(kb):
    """C4: every user x every item, k = 20, training positives excluded, in one call; equals the 256-user recommend_topk loop
    (the scheme of test_yelp2018_shape_full_graph_top20) index for index and recommends no training positive."""
    from kgat_b200 import synthetic
    from kgat_b200.metrics import InteractionCSR
    from kgat_b200.trainer import build_model

    g = synthetic.make_ckg("yelp2018", with_dicts=False)
    m = build_model(g, "cuda").eval()
    train = InteractionCSR(g.train_interactions, g.user_num, g.item_num, "cuda")
    k = 20
    rec = m.recommend(torch.arange(g.user_num), g.item_num, k=k, exclude=train)
    items = torch.arange(g.item_num, device="cuda")
    out = torch.empty(g.user_num, k, dtype=torch.int64, device="cuda")
    val = torch.empty(g.user_num, k, dtype=torch.float32, device="cuda")
    for s in range(0, g.user_num, 256):
        e = min(s + 256, g.user_num)
        ptr, flat = train.batch(s, e)
        idx, v = m.recommend_topk(torch.arange(s, e), items, k, ptr, flat, want_values=True)
        out[s:e], val[s:e] = idx.long(), v
    assert bool((rec.count == k).all())
    assert torch.equal(rec.items, out)
    assert torch.equal(rec.scores.view(torch.int32), val.view(torch.int32))
    users = torch.arange(g.user_num, device="cuda")[:, None].expand(-1, k)
    assert not bool(train.contains(users, rec.items).any())

"""Top-k recommendations with per-group caps (``kgat_recommend_group_masks`` / ``kgat_recommend_capped_round``,
``ops.recommend_capped``, ``KGAT.recommend_capped``) against the torch reference ``oracle/recommend_capped_ref.py`` fed the
bit-exact ``PREDICT`` scores, against ``KGAT.recommend`` when no cap binds, and across forced splits and round sizes."""

from __future__ import annotations

import numpy as np
import pytest
import torch

from oracle.recommend_capped_ref import recommend_capped_ref
from test_recommend import USER_NUM, _cf_entities, _codeforces_sm, _exclude, _hand_ckg, _model_from_golden

# ---------------------------------------------------------------------------------------------
# CPU: the reference on test_recommend's hand-built CKG
# ---------------------------------------------------------------------------------------------
# problem 0: tag 5, rating 7, contest 9      problem 1: tag 5, rating 8      problem 2: tag 6, rating 7
# problem 3: tag 5 (no rating)               problem 4: tag 6, rating 8, contest 9
# recommend's order:  user 0: p4 (2), p0 (1), p2 (1), p3 (.5), p1 (0)
#                     user 1: p1 (1), p2 (1), p3 (.5), p0 (0), p4 (0)
#                     user 2: p2 (2), p4 (2), p0 (1), p1 (1), p3 (1)
TAG5, TAG6, R7, R8 = 5, 6, 7, 8


def _ref(users, k, caps, items=None, **kw):
    rp, col, table = _hand_ckg()
    users = torch.tensor(users)
    scores = table[users] @ table[:5].T
    return recommend_capped_ref(scores, users, torch.arange(5) if items is None else torch.tensor(items), k, caps, rp, col, USER_NUM, **kw)


def _check(got, items, scores):
    it, sc, cnt = got
    want_cnt = [sum(1 for x in row if x >= 0) for row in items]
    assert it.tolist() == items
    assert cnt.tolist() == want_cnt
    for b, row in enumerate(scores):
        assert sc[b, : want_cnt[b]].tolist() == row
        assert bool((sc[b, want_cnt[b] :] == float("-inf")).all())


def test_reference_tag_cap_reorders():
    # user 2 without caps: p2, p4, p0; p4 shares tag 6 with p2
    _check(_ref([2], 3, [([TAG5], 1), ([TAG6], 1)]), [[2, 0, -1]], [[2, 1]])
    _check(_ref([2], 3, [([TAG6], 1)]), [[2, 0, 1]], [[2, 1, 1]])
    _check(_ref([2], 3, [([TAG6], 3)]), [[2, 4, 0]], [[2, 2, 1]])  # a cap >= k does not bind


def test_reference_cap_zero_excludes_the_group():
    _check(_ref([0, 1], 3, [([TAG6], 0)]), [[0, 3, 1], [1, 3, 0]], [[1, .5, 0], [1, .5, 0]])
    _check(_ref([0], 5, [([TAG5, TAG6], 0)]), [[-1] * 5], [[]])  # one group of two tags


def test_reference_problem_without_rating_ignores_rating_caps():
    # every rating capped at 0: only problem 3, which has no rating, is left; k is unreachable
    _check(_ref([0, 1, 2], 3, [([R7], 0), ([R8], 0)]), [[3, -1, -1]] * 3, [[.5], [.5], [1]])


def test_reference_problem_in_two_groups_counts_against_both():
    # user 0: p4 (tag 6, r8) accepted; p0 (tag 5, r7) accepted and fills both caps; p2 (r7) and p3, p1 (tag 5) are rejected
    _check(_ref([0], 4, [([TAG5], 1), ([R7], 1)]), [[4, 0, -1, -1]], [[2, 1]])
    # capping tag 5 alone lets p2 in
    _check(_ref([0], 4, [([TAG5], 1)]), [[4, 0, 2, -1]], [[2, 1, 1]])


def test_reference_ties_by_position_in_items():
    caps = [([TAG5], 1)]
    _check(_ref([2], 3, caps), [[2, 4, 0]], [[2, 2, 1]])
    # p2 and p4 tie at 2, p0 / p1 / p3 at 1: the earlier position in items goes first, so p3 takes tag 5's place
    _check(_ref([2], 3, caps, items=[4, 3, 2, 1, 0]), [[4, 2, 3]], [[2, 2, 1]])


def test_reference_exclude_and_require():
    ptr, ex = _exclude([[0], [], [4, 2]])
    kw = dict(exclude_ptr=ptr, exclude_items=ex, require=[[R7, R8]])  # problems with a rating: 0, 1, 2, 4
    _check(_ref([0, 1, 2], 3, [([TAG6], 1)], **kw), [[4, 1, -1], [1, 2, 0], [0, 1, -1]], [[2, 0], [1, 1, 0], [1, 1]])


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


@pytest.fixture(scope="module")
def cf_sm(kb):
    return _codeforces_sm()


def _predict(m, users, n):
    from kgat_b200.model import KGATMode

    return m(users.cuda(), torch.arange(n).cuda(), mode=KGATMode.PREDICT)


def _assert_equal_to_ref(m, users, n_items, k, caps, exclude=None, require=None, items=None):
    """KGAT.recommend_capped against the reference fed the PREDICT scores: items, score bits and counts equal."""
    got = m.recommend_capped(users, n_items if items is None else items, k, caps, exclude=exclude, require=require)
    graph = m._graph()
    scores = _predict(m, users, n_items).cpu()
    ex = dict(exclude_ptr=exclude.ptr_dev.cpu(), exclude_items=exclude.items.cpu()) if exclude is not None else {}
    want = recommend_capped_ref(scores, users.cpu(), torch.arange(n_items) if items is None else items.cpu(), k, caps, graph.row_ptr.cpu(),
                                graph.col_idx.cpu(), m._user_num, require=require, **ex)
    assert torch.equal(got.count.cpu(), want[2])
    assert torch.equal(got.items.cpu(), want[0])
    assert torch.equal(got.scores.cpu().view(torch.int32), want[1].view(torch.int32))
    return got


def _cf_caps(g, tag_cap=None, rating_cap=None, zero_tags=()):
    c0, d0, t0, r0 = _cf_entities(g)
    caps = []
    if tag_cap is not None:
        caps += [([t], tag_cap) for t in range(t0, t0 + 37)]
    if rating_cap is not None:
        caps += [([r], rating_cap) for r in range(r0, r0 + 28)]
    caps += [([t], 0) for t in zero_tags]
    return caps


@pytest.mark.gpu
def test_matches_reference_on_golden_models(kb, golden_model):
    g = golden_model
    m = _model_from_golden(g)
    users, items, ent = int(g["user_num"]), int(g["item_num"]), int(g["entity_num"])
    kg = list(range(items, ent))
    u = torch.cat([torch.arange(users), torch.tensor([0, users - 1])])
    k = min(20, items - 1)
    caps = [([e], 1 + j % 3) for j, e in enumerate(kg[:40])] + [(kg[40:60], 0)] if len(kg) > 60 else [([e], 1) for e in kg]
    _assert_equal_to_ref(m, u, items, k, caps)
    perm = torch.from_numpy(np.random.default_rng(5).permutation(items))
    _assert_equal_to_ref(m, u, items, k, caps, items=perm)


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["a", "b", "c", "d", "e"])
def test_matches_reference_on_codeforces_sm(kb, cf_sm, case):
    from kgat_b200.metrics import InteractionCSR

    g, m = cf_sm
    c0, d0, t0, r0 = _cf_entities(g)
    users = torch.arange(g.user_num)
    if case == "a":
        got = _assert_equal_to_ref(m, users, g.item_num, 20, _cf_caps(g, tag_cap=2))
    elif case == "b":
        ex = InteractionCSR(g.train_interactions, g.user_num, g.item_num, "cuda")
        got = _assert_equal_to_ref(m, users, g.item_num, 20, _cf_caps(g, tag_cap=3, rating_cap=4), exclude=ex,
                                   require=[list(range(r0 + 4, r0 + 20))])
    elif case == "c":
        got = _assert_equal_to_ref(m, users, g.item_num, 64, _cf_caps(g, rating_cap=1))
    elif case == "d":
        got = _assert_equal_to_ref(m, users, g.item_num, 64, _cf_caps(g, rating_cap=1), require=[list(range(r0, r0 + 28))])
        assert bool((got.count == 28).all())  # one problem per rating, then candidates run out
    else:
        caps = _cf_caps(g, zero_tags=(t0, t0 + 1, t0 + 5))
        got = _assert_equal_to_ref(m, users, g.item_num, 20, caps)
        rec = m.recommend(users, g.item_num, k=20)
        assert not torch.equal(rec.items, got.items)  # the zeroed tags were in some plain lists
    assert bool((got.count > 0).all())


@pytest.mark.gpu
def test_caps_that_never_bind_give_recommend(kb, cf_sm):
    from kgat_b200.metrics import InteractionCSR

    g, m = cf_sm
    c0, d0, t0, r0 = _cf_entities(g)
    ex = InteractionCSR(g.train_interactions, g.user_num, g.item_num, "cuda")
    users = torch.arange(g.user_num)
    for k in (1, 20, 128):
        caps = _cf_caps(g, tag_cap=k, rating_cap=k + 3)
        for require in (None, [[t0, t0 + 1, t0 + 2]]):
            got = m.recommend_capped(users, g.item_num, k, caps, exclude=ex, require=require)
            rec = m.recommend(users, g.item_num, k=k, exclude=ex, require=require)
            assert torch.equal(got.items, rec.items) and torch.equal(got.count, rec.count)
            assert torch.equal(got.scores.view(torch.int32), rec.scores.view(torch.int32))


@pytest.mark.gpu
def test_result_does_not_depend_on_split_or_round_size(kb, cf_sm):
    from kgat_b200 import ops
    from kgat_b200.metrics import InteractionCSR

    g, m = cf_sm
    c0, d0, t0, r0 = _cf_entities(g)
    tables, graph = m._tables(), m._graph()
    ex = InteractionCSR(g.train_interactions, g.user_num, g.item_num, "cuda")
    users = torch.arange(200).repeat(2)
    cand = torch.from_numpy(np.random.default_rng(4).permutation(g.item_num))
    cases = [(20, _cf_caps(g, tag_cap=1)), (20, _cf_caps(g, tag_cap=3, rating_cap=4)), (64, _cf_caps(g, rating_cap=1)),
             (5, _cf_caps(g, tag_cap=1, zero_tags=(t0 + 2,)))]
    most = 0
    for k, caps in cases:
        ref = None
        for M in sorted({k, 64, 128}):
            for s in (1, 2, 7, 64, None):
                it, sc, cnt, rounds = ops.recommend_capped(tables, graph, users, cand, k, caps, g.user_num, ex.ptr_dev, ex.items, m=M, slices=s)
                assert rounds <= len(caps) + 1
                most = max(most, rounds)
                if ref is None:
                    ref = (it, sc, cnt)
                    assert torch.equal(it[:200], it[200:])
                    continue
                assert torch.equal(it, ref[0]) and torch.equal(cnt, ref[2])
                assert torch.equal(sc.view(torch.int32), ref[1].view(torch.int32))
    assert most >= 3


@pytest.mark.gpu
def test_argument_errors_and_state(kb, golden_tiny):
    from kgat_b200 import ops
    from kgat_b200.metrics import InteractionCSR

    g = golden_tiny
    m = _model_from_golden(g)
    users, ent, items = int(g["user_num"]), int(g["entity_num"]), int(g["item_num"])
    u = torch.arange(3)
    good = [([items], 1)]
    bad = [
        dict(user_ids=u, items=items, k=0, caps=good),
        dict(user_ids=u, items=items, k=129, caps=good),
        dict(user_ids=torch.tensor([users]), items=items, k=3, caps=good),
        dict(user_ids=u, items=torch.tensor([0, ent]), k=3, caps=good),
        dict(user_ids=u, items=torch.tensor([3, 1, 3]), k=3, caps=good),
        dict(user_ids=u, items=items, k=3, caps=good, require=[[items], []]),
        dict(user_ids=u, items=items, k=3, caps=good, exclude=InteractionCSR(np.array([[0, 1]]), users + 1, items, "cuda")),
        dict(user_ids=u.float(), items=items, k=3, caps=good),
        dict(user_ids=u, items=items, k=3, caps=[([], 1)]),
        dict(user_ids=u, items=items, k=3, caps=[([ent], 1)]),
        dict(user_ids=u, items=items, k=3, caps=[([-1], 1)]),
        dict(user_ids=u, items=items, k=3, caps=[([items], -1)]),
        dict(user_ids=u, items=items, k=3, caps=[([items], 1.5)]),
        dict(user_ids=u, items=items, k=3, caps=[([items], True)]),
        dict(user_ids=u, items=items, k=3, caps=[([items], "2")]),
        dict(user_ids=u, items=items, k=3, caps=[([items], 1)] * 129),
        dict(user_ids=u, items=items, k=3, caps=[[items]]),
    ]
    for kw in bad:
        with pytest.raises(ValueError):
            m.recommend_capped(**kw)
    tables, graph = m._tables(), m._graph()
    for args, kw in (((u, torch.arange(4), 3, good, users), dict(m=2)), ((u, torch.arange(4), 3, good, users), dict(m=129)),
                     ((u, torch.arange(4), 3, good, users), dict(slices=65)), ((u, torch.tensor([ent]), 3, good, users), {}),
                     ((u, torch.arange(4), 3, good, graph.n), {})):
        with pytest.raises(ValueError):
            ops.recommend_capped(tables, graph, *args, **kw)
    assert len(m.recommend_capped(u, items, 3, [([items], 1)] * 128).count) == 3  # 128 groups are allowed

    # no RNG drawn; recommend and rank unchanged by a capped call
    from kgat_b200.metrics import InteractionCSR as CSR

    targets = CSR(np.array([[0, 1], [1, 2], [2, 3]]), users, items, "cuda")
    rec0, rank0 = m.recommend(u, items, k=5), m.rank(u, items, targets)
    cpu_rng, gpu_rng = torch.get_rng_state(), torch.cuda.get_rng_state()
    m.recommend_capped(u, items, 5, [([e], 1) for e in range(items, min(ent, items + 20))])
    assert torch.equal(torch.get_rng_state(), cpu_rng) and torch.equal(torch.cuda.get_rng_state(), gpu_rng)
    rec1, rank1 = m.recommend(u, items, k=5), m.rank(u, items, targets)
    assert torch.equal(rec0.items, rec1.items) and torch.equal(rec0.scores.view(torch.int32), rec1.scores.view(torch.int32))
    assert torch.equal(rank0.rank, rank1.rank)
    # no users / no candidates
    r = m.recommend_capped(torch.zeros(0, dtype=torch.int64), items, 5, good)
    assert r.items.shape == (0, 5) and r.count.shape == (0,)
    r = m.recommend_capped(u, 0, 5, good)
    assert r.count.tolist() == [0] * 3 and bool((r.items == -1).all()) and bool((r.scores == float("-inf")).all())


@pytest.mark.gpu
def test_codeforces_full_all_users_in_one_call(kb):
    """Every one of the 200,000 users, k = 20, cap 3 per tag and 4 per rating, training positives excluded, in one call; 256
    sampled rows equal the reference fed their PREDICT rows."""
    from kgat_b200 import synthetic
    from kgat_b200.metrics import InteractionCSR
    from kgat_b200.trainer import build_model

    g = synthetic.make_ckg("codeforces-full", with_dicts=False)
    m = build_model(g, "cuda").eval()
    ex = InteractionCSR(g.train_interactions, g.user_num, g.item_num, "cuda")
    caps = _cf_caps(g, tag_cap=3, rating_cap=4)
    got = m.recommend_capped(torch.arange(g.user_num), g.item_num, 20, caps, exclude=ex)
    assert got.items.shape == (g.user_num, 20)
    rows = torch.from_numpy(np.random.default_rng(6).choice(g.user_num, 256, replace=False))
    graph = m._graph()
    scores = _predict(m, rows, g.item_num).cpu()
    want = recommend_capped_ref(scores, rows, torch.arange(g.item_num), 20, caps, graph.row_ptr.cpu(), graph.col_idx.cpu(), g.user_num,
                                exclude_ptr=ex.ptr_dev.cpu(), exclude_items=ex.items.cpu())
    r = rows.cuda()
    assert torch.equal(got.count[r].cpu(), want[2])
    assert torch.equal(got.items[r].cpu(), want[0])
    assert torch.equal(got.scores[r].cpu().view(torch.int32), want[1].view(torch.int32))

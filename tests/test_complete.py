"""Knowledge-graph completion with the trained TransR half (``kgat_complete_topk`` / ``kgat_complete_rank``, ``KGAT.complete``,
``KGAT.kg_rank``, ``metrics.TripleSet``, ``metrics.link_metrics``) against the torch reference ``oracle/complete_ref.py`` fed the
kernel's bit-exact energies, and against the TransR loss kernel."""

from __future__ import annotations

import numpy as np
import pytest
import torch

from conftest import Golden
from oracle.complete_ref import complete_ref, energy_f64, kg_rank_ref, key32, link_metrics_ref

# ---------------------------------------------------------------------------------------------
# CPU: the reference on a hand-built case, TripleSet, and the metrics' reduction
# ---------------------------------------------------------------------------------------------
NAN, INF = float("nan"), float("inf")
N_NODES, N_REL = 7, 2
# energy against node x of the query rows used below
ENERGY = torch.tensor([[1.0, 1.0, 0.5, 0.0, 2.0, NAN, 3.0],   # q0: NaN first, then 0, .5, 1 (pos 0) before 1 (pos 1)
                       [4.0, 3.0, 2.0, 1.0, 0.0, 5.0, 6.0],   # q1
                       [1.0, 1.0, 1.0, 1.0, 1.0, 1.0, 1.0]])  # q2: all tied


def _keys(triples):
    return torch.tensor(sorted((h * N_REL + r) * N_NODES + t for h, r, t in triples), dtype=torch.int64)


def test_key_orders_low_energy_first_nan_first_and_signed_zero():
    k = key32(torch.tensor([NAN, 0.0, -0.0, 1.0, INF]))
    assert k[0] > k[1] and k[1] < k[2] and k[2] > k[3] > k[4]


def test_reference_topk_ties_nan_exclusions_and_repeats():
    heads, rels = torch.tensor([0, 1, 2, 0]), torch.tensor([0, 1, 0, 0])
    known = _keys([(0, 0, 3), (1, 1, 4), (2, 1, 0)])  # (2, 1, 0) is another relation than query 2's
    t, e, c = complete_ref(ENERGY[[0, 1, 2, 0]], heads, rels, torch.arange(6), 4, known, N_NODES, N_REL)
    assert t.tolist() == [[5, 2, 0, 1], [3, 2, 1, 0], [0, 1, 2, 3], [5, 2, 0, 1]]
    assert c.tolist() == [4, 4, 4, 4]
    assert torch.isnan(e[0, 0]) and e[0, 1:].tolist() == [0.5, 1.0, 1.0]
    # k past the eligible candidates pads with -1 / +inf; a permuted subset breaks ties by its order
    t, e, c = complete_ref(ENERGY[2:3], heads[2:3], rels[2:3], torch.tensor([4, 1, 0]), 5, known, N_NODES, N_REL)
    assert t.tolist() == [[4, 1, 0, -1, -1]] and c.tolist() == [3] and e[0, 3:].tolist() == [INF, INF]


def test_reference_rank_target_stays_eligible_and_missing_target():
    heads, rels = torch.tensor([0, 0, 1, 1, 2]), torch.tensor([0, 0, 1, 1, 0])
    tails = torch.tensor([3, 1, 4, 6, 2])
    known = _keys([(0, 0, 3), (0, 0, 2), (1, 1, 4), (1, 1, 3)])
    energy, rank, elig = kg_rank_ref(ENERGY[[0, 0, 1, 1, 2]], heads, rels, tails, torch.arange(6), known, N_NODES, N_REL)
    # q0: target 3 is known but stays eligible; NaN beats it, 2 is excluded.  q1: target 1 beaten by NaN and 0 (3 is excluded,
    # 2 is excluded).  q2: target 4 known, stays; 3 excluded, so it is first.  q3: 6 is not a candidate.  q4: ties, position 2.
    assert rank.tolist() == [1, 2, 0, -1, 2]
    assert elig.tolist() == [5, 4, 5, 4, 6]
    assert energy.tolist() == [0.0, 1.0, 0.0, 6.0, 1.0]
    # rank < k  <=>  complete(exclude minus the target's triple) lists the target at that rank
    t, _, _ = complete_ref(ENERGY[:1], heads[:1], rels[:1], torch.arange(6), 3, _keys([(0, 0, 2)]), N_NODES, N_REL)
    assert t[0, 1] == 3


def test_triple_set_keys_decode_and_overflow():
    from kgat_b200.metrics import TripleSet

    ts = TripleSet([2, 0, 2, 0], [1, 0, 1, 1], [5, 3, 5, 6], N_NODES, N_REL, "cpu")
    assert ts.keys.tolist() == sorted({(2 * N_REL + 1) * N_NODES + 5, 3, (0 * N_REL + 1) * N_NODES + 6})
    h, r, t = ts.triples()
    assert list(zip(h.tolist(), r.tolist(), t.tolist())) == [(0, 0, 3), (0, 1, 6), (2, 1, 5)]
    with pytest.raises(ValueError):
        TripleSet([0], [0], [0], 2**32, 2**4, "cpu")
    with pytest.raises(ValueError):
        TripleSet([0], [2], [0], N_NODES, N_REL, "cpu")
    with pytest.raises(ValueError):
        TripleSet([0, 1], [0], [0], N_NODES, N_REL, "cpu")


def test_link_terms_reduce_to_numpy_metrics():
    from kgat_b200.metrics import link_terms

    rng = np.random.default_rng(3)
    ranks = rng.integers(-1, 40, 1000)
    hits = (1, 3, 10)
    s = link_terms(torch.from_numpy(ranks), hits).sum(0).tolist()
    want = link_metrics_ref(ranks, hits)
    n = s[0]
    assert n == want["n_ranked"] == int((ranks >= 0).sum())
    assert abs(s[1] / n - want["mrr"]) < 1e-14 and abs(s[2] / n - want["mean_rank"]) < 1e-12
    for j, k in enumerate(hits):
        assert s[3 + j] / n == want["hits"][k]


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


def _energies(m, heads, rels, n):
    """The kernel's exact energies of every (heads[q], rels[q]) against nodes 0 .. n-1, through kg_rank's target energies."""
    Q = heads.numel()
    r = m.kg_rank(heads.repeat_interleave(n), rels.repeat_interleave(n), torch.arange(n).repeat(Q), torch.tensor([0]))
    return r.energy.view(Q, n).cpu()


def _assert_complete_equals_reference(m, heads, rels, cand, k, known):
    got = m.complete(heads, rels, cand, k=k, exclude=known)
    E = _energies(m, heads, rels, m.node_num)
    c = torch.arange(cand) if isinstance(cand, int) else cand
    keys = None if known is None else known.keys.cpu()
    t, e, cnt = complete_ref(E, heads, rels, c, k, keys, m.node_num, m._relation_num)
    assert torch.equal(got.tails.cpu(), t) and torch.equal(got.count.cpu(), cnt)
    assert torch.equal(got.energy.cpu().view(torch.int32), e.view(torch.int32))
    return got, E


def _assert_rank_equals_reference(m, heads, rels, tails, cand, known, E=None):
    got = m.kg_rank(heads, rels, tails, cand, exclude=known)
    E = _energies(m, heads, rels, m.node_num) if E is None else E
    c = torch.arange(cand) if isinstance(cand, int) else cand
    keys = None if known is None else known.keys.cpu()
    e, r, el = kg_rank_ref(E, heads, rels, tails, c, keys, m.node_num, m._relation_num)
    assert torch.equal(got.energy.cpu().view(torch.int32), e.view(torch.int32))
    assert torch.equal(got.rank.cpu(), r) and torch.equal(got.eligible.cpu(), el)
    return got


def _random_known(m, rng, n=400):
    from kgat_b200.metrics import TripleSet

    N, R = m.node_num, m._relation_num
    return TripleSet(torch.from_numpy(rng.integers(0, N, n)), torch.from_numpy(rng.integers(0, R, n)), torch.from_numpy(rng.integers(0, N, n)),
                     N, R, "cuda")


@pytest.mark.gpu
def test_energies_are_the_transr_loss_terms(kb):
    """For every supported width: kg_rank's E(h, r, n) - E(h, r, p) equals transr_forward's per-sample margin bit for bit, and
    the energies are within 1e-5 relative of fp64."""
    from kgat_b200 import ops, synthetic
    from kgat_b200.model import KGAT, KGATArgs

    g = synthetic.make_ckg("tiny", seed=7)
    rng = np.random.default_rng(1)
    B = 300
    for d in (32, 64, 128):
        torch.manual_seed(d)
        m = KGAT(KGATArgs(user_num=g.user_num, entity_num=g.entity_num, relation_num=g.relation_num, cf_embedding_dim=d, kg_embedding_dim=d,
                          layer_size=[d, d // 2])).cuda().eval()
        with torch.no_grad():  # spread the parameters out of xavier's narrow range
            m._relation_embedding.weight.mul_(3.0)
        N, R = m.node_num, m._relation_num
        h, r, p, n = (torch.from_numpy(rng.integers(0, hi, B)).cuda() for hi in (N, R, N, N))
        scratch = torch.empty(2 * B, device="cuda")
        loss = torch.empty(1, device="cuda")
        emb, rel, w = m._transr_params()
        ops.transr_forward(emb, rel, w, h, r, p, n, 1e-5, loss, scratch)
        ep = m.kg_rank(h, r, p, N).energy
        en = m.kg_rank(h, r, n, N).energy
        assert torch.equal((en - ep).view(torch.int32), scratch[:B].view(torch.int32)), d
        ref = energy_f64(emb, rel, w, h, r, p)
        assert float(((ep.double() - ref).abs() / ref.abs().clamp(min=1e-30)).max()) < 1e-5, d


@pytest.mark.gpu
def test_golden_models_equal_reference(kb, golden_model):
    g = golden_model
    m = _model_from_golden(g)
    N, R = m.node_num, m._relation_num
    rng = np.random.default_rng(5)
    Q = 40
    heads = torch.from_numpy(rng.integers(0, N, Q))
    rels = torch.from_numpy(rng.integers(0, R, Q))
    heads[-3:] = heads[0]  # repeated queries
    rels[-3:] = rels[0]
    known = _random_known(m, rng)
    # plant known triples of the queries themselves, so the filter has something to remove
    from kgat_b200.metrics import TripleSet

    extra = torch.from_numpy(rng.integers(0, N, Q))
    known = TripleSet(torch.cat([known.triples()[0].cpu(), heads]), torch.cat([known.triples()[1].cpu(), rels]),
                      torch.cat([known.triples()[2].cpu(), extra]), N, R, "cuda")
    subset = torch.from_numpy(rng.permutation(N)[: 2 * N // 3])
    E = None
    for cand in (N, subset):
        for ex in (None, known):
            for k in (1, 10, 128):
                _, E = _assert_complete_equals_reference(m, heads, rels, cand, k, ex)
            tails = torch.cat([torch.from_numpy(rng.integers(0, N, Q - 5)), extra[:5]])
            _assert_rank_equals_reference(m, heads, rels, tails, cand, ex, E)


def _rating_relation(g):
    """The relation from a problem node to its rating node: tails are the 28 rating entities, heads problem nodes."""
    for r in np.unique(g.relations):
        sel = g.relations == r
        hs, ts = g.heads[sel], g.tails[sel]
        if np.unique(ts).size == 28 and hs.min() >= g.user_num and hs.max() < g.user_num + g.item_num:
            return int(r), np.unique(ts)
    raise AssertionError("no rating relation")


@pytest.mark.gpu
def test_codeforces_rating_prediction_equals_reference(kb):
    from kgat_b200.metrics import TripleSet

    g, m = _codeforces_sm()
    r, ratings = _rating_relation(g)
    known = TripleSet.from_ckg(g)
    rated = np.unique(g.heads[g.relations == r])
    unrated = np.setdiff1d(np.arange(g.user_num, g.user_num + g.item_num), rated)
    assert unrated.size > 0
    heads = torch.from_numpy(np.concatenate([unrated[:50], rated[:30]]))
    rels = torch.full_like(heads, r)
    cand = torch.from_numpy(np.random.default_rng(2).permutation(ratings))
    got, E = _assert_complete_equals_reference(m, heads, rels, cand, 5, known)
    assert bool((got.count[:50] == 5).all()) and bool((got.count[50:] == 5).all())
    assert bool(torch.isin(got.tails.cpu(), cand).all())
    _assert_complete_equals_reference(m, heads, rels, m.node_num, 20, None)
    # held-in ratings ranked among the 28 (the target stays eligible), and the consistency with complete
    tails = torch.from_numpy(np.array([g.tails[(g.relations == r) & (g.heads == h)][0] for h in rated[:30]]))
    rk = _assert_rank_equals_reference(m, heads[50:], rels[50:], tails, cand, known, E[50:])
    assert bool((rk.eligible == 28).all())  # a rated problem's one known rating is its target, which stays eligible
    rk = _assert_rank_equals_reference(m, heads[50:], rels[50:], tails, cand, None, E[50:])
    top = m.complete(heads[50:], rels[50:], cand, k=28)
    for q in range(30):
        rq = int(rk.rank[q])
        assert int(top.tails[q, rq]) == int(tails[q])
        assert all(int(x) != int(tails[q]) for x in top.tails[q, :rq].tolist())


@pytest.mark.gpu
def test_rank_below_k_iff_complete_lists_target(kb):
    from kgat_b200.metrics import TripleSet

    g, m = _codeforces_sm()
    rng = np.random.default_rng(9)
    sel = rng.choice(g.nnz, 200, replace=False)
    h, r, t = (torch.from_numpy(np.asarray(x[sel]).astype(np.int64)) for x in (g.heads, g.relations, g.tails))
    known = TripleSet.from_ckg(g)
    rk = m.kg_rank(h, r, t, m.node_num, exclude=known)
    kh, kr, kt = (x.cpu() for x in known.triples())
    k = 64
    for q in range(0, 200, 10):
        keep = ~((kh == h[q]) & (kr == r[q]) & (kt == t[q]))
        ex = TripleSet(kh[keep], kr[keep], kt[keep], m.node_num, m._relation_num, "cuda")
        top = m.complete(h[q : q + 1], r[q : q + 1], m.node_num, k=k, exclude=ex)
        rq = int(rk.rank[q])
        assert (rq < k) == bool((top.tails[0] == t[q]).any())
        if rq < k:
            assert int(top.tails[0, rq]) == int(t[q])


@pytest.mark.gpu
def test_forced_splits_and_repeats_give_identical_bytes(kb):
    from kgat_b200 import ops
    from kgat_b200.metrics import TripleSet

    g, m = _codeforces_sm()
    emb, rel, w = m._transr_params()
    rng = np.random.default_rng(4)
    Q = 300
    h = torch.from_numpy(rng.integers(0, m.node_num, Q))
    r = torch.from_numpy(rng.integers(0, m._relation_num, Q))
    t = torch.from_numpy(rng.integers(0, m.node_num, Q))
    known = TripleSet.from_ckg(g).keys
    outs = []
    for s in (None, 1, 2, 7, 64, None):
        a = ops.complete_topk(emb, rel, w, h, r, m.node_num, 32, known, slices=s)
        b = ops.kg_rank(emb, rel, w, h, r, t, m.node_num, known, slices=s)
        outs.append([x.cpu() for x in (*a, *b)])
    for o in outs[1:]:
        for x, y in zip(outs[0], o):
            assert torch.equal(x.view(torch.uint8) if x.is_floating_point() else x, y.view(torch.uint8) if y.is_floating_point() else y)


@pytest.mark.gpu
def test_complete_does_not_disturb_training(kb):
    """CF steps, then KG steps with ``complete`` / ``kg_rank`` calls inside the deferred KG phase: parameters, both Adam moments,
    losses and torch's RNG state are bitwise those of the same run without the calls."""
    from kgat_b200 import synthetic
    from kgat_b200.model import KGATMode
    from kgat_b200.trainer import EpochData, build_model

    g = synthetic.make_ckg("small", seed=11)
    data = EpochData.sample(g, seed=3, n_cf=4, n_kg=12).tensors(device="cuda")
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
                m.complete(torch.arange(5), torch.zeros(5, dtype=torch.int64), m.node_num, k=7)
                m.kg_rank(torch.arange(5), torch.ones(5, dtype=torch.int64), torch.arange(5) + 1, 100)
        rng = torch.get_rng_state().clone(), torch.cuda.get_rng_state().clone()
        sd = {k: v.clone() for k, v in m.state_dict().items() if not v.is_sparse}
        mom = []
        for opt in (m._cf_optimizer, m._kg_optimizer):
            for grp in opt.param_groups:
                for p in grp["params"]:
                    st = opt.state.get(p, {})
                    mom += [st[n].clone() for n in ("exp_avg", "exp_avg_sq") if n in st]
        out[call] = (torch.stack(losses), sd, rng, mom)
    a, b = out[False], out[True]
    assert torch.equal(a[0], b[0])
    for k in a[1]:
        assert torch.equal(a[1][k], b[1][k]), k
    assert torch.equal(a[2][0], b[2][0]) and torch.equal(a[2][1], b[2][1])
    assert len(a[3]) == len(b[3]) > 0 and all(torch.equal(x, y) for x, y in zip(a[3], b[3]))


@pytest.mark.gpu
def test_argument_errors(kb):
    from kgat_b200.metrics import TripleSet

    g, m = _codeforces_sm()
    N, R = m.node_num, m._relation_num
    h, r, t = torch.tensor([0, 1]), torch.tensor([0, 1]), torch.tensor([2, 3])
    bad = [
        lambda: m.complete(h, r, N, k=0),
        lambda: m.complete(h, r, N, k=129),
        lambda: m.complete(torch.tensor([N]), r[:1], N),
        lambda: m.complete(torch.tensor([-1]), r[:1], N),
        lambda: m.complete(h, torch.tensor([0, R]), N),
        lambda: m.complete(h, r[:1], N),
        lambda: m.complete(h, r, N + 1),
        lambda: m.complete(h, r, -1),
        lambda: m.complete(h, r, torch.tensor([3, 4, 3])),
        lambda: m.complete(h, r, torch.tensor([N])),
        lambda: m.complete(h, r, torch.tensor([[1, 2]])),
        lambda: m.complete(h, r, 2.5),
        lambda: m.complete(h.float(), r, N),
        lambda: m.complete(h, r, N, exclude=TripleSet([0], [0], [0], N + 1, R, "cuda")),
        lambda: m.kg_rank(h, r, t[:1], N),
        lambda: m.kg_rank(h, r, torch.tensor([0, N]), N),
        lambda: m.kg_rank(h, r, t, torch.tensor([1, 1])),
        lambda: m.kg_rank(h, r, t, N, exclude=TripleSet([0], [0], [0], N, R + 1, "cuda")),
    ]
    for i, f in enumerate(bad):
        with pytest.raises(ValueError):
            f()
            pytest.fail(f"case {i} did not raise")


@pytest.mark.gpu
def test_link_metrics_equal_reference_ranks(kb):
    from kgat_b200.metrics import TripleSet, link_metrics

    g, m = _codeforces_sm()
    known = TripleSet.from_ckg(g)
    rng = np.random.default_rng(8)
    sel = rng.choice(g.nnz, 500, replace=False)
    h, r, t = (torch.from_numpy(np.asarray(x[sel]).astype(np.int64)) for x in (g.heads, g.relations, g.tails))
    for cand in ("relation", "all"):
        got = link_metrics(m, (h, r, t), known, hits=(1, 3, 10), candidates=cand)
        kh, kr, kt = known.triples()
        ranks = []
        for rel in sorted(set(r.tolist())):
            s = r == rel
            c = m.node_num if cand == "all" else torch.unique(kt[kr == rel])
            ranks.append(m.kg_rank(h[s], r[s], t[s], c, exclude=known).rank.cpu())
            want_r = link_metrics_ref(ranks[-1].numpy())
            assert got["per_relation"][rel]["n_ranked"] == want_r["n_ranked"]
            assert abs(got["per_relation"][rel]["mrr"] - want_r["mrr"]) < 1e-12
        want = link_metrics_ref(torch.cat(ranks).numpy())
        assert got["n_ranked"] == want["n_ranked"] == 500 and got["n_skipped"] == 0
        assert abs(got["mrr"] - want["mrr"]) < 1e-12 and abs(got["mean_rank"] - want["mean_rank"]) < 1e-9
        assert all(abs(got["hits"][k] - want["hits"][k]) < 1e-12 for k in (1, 3, 10))


@pytest.mark.gpu
def test_amazon_book_shape_one_call(kb):
    """10,000 triples ranked against all 159,251 nodes of the Amazon-book shape (80 relations, d = k = 64) in one call, and
    top-10 completion of 2,000 queries; a sample agrees with the reference."""
    from kgat_b200 import ops

    N, R, d = 159_251, 80, 64
    gen = torch.Generator(device="cuda").manual_seed(0)
    emb = torch.randn(N, d, device="cuda", generator=gen) * 0.1
    rel = torch.randn(R, d, device="cuda", generator=gen) * 0.1
    w = torch.randn(R, d, d, device="cuda", generator=gen) * 0.1
    rng = np.random.default_rng(0)
    Q = 10_000
    h, r, t = (torch.from_numpy(rng.integers(0, hi, Q)) for hi in (N, R, N))
    energy, rank, eligible = ops.kg_rank(emb, rel, w, h, r, t, N)
    assert bool((eligible == N).all()) and bool((rank >= 0).all())
    tails, en, count = ops.complete_topk(emb, rel, w, h[:2000], r[:2000], N, 10)
    assert bool((count == 10).all())
    sample = torch.from_numpy(rng.choice(2000, 6, replace=False))
    hs, rs = h[sample], r[sample]
    e_all = ops.kg_rank(emb, rel, w, hs.repeat_interleave(N), rs.repeat_interleave(N), torch.arange(N).repeat(6), torch.tensor([0]))[0]
    E = e_all.view(6, N).cpu()
    tr, er, _ = complete_ref(E, hs, rs, torch.arange(N), 10)
    assert torch.equal(tails[sample.cuda()].cpu(), tr) and torch.equal(en[sample.cuda()].cpu().view(torch.int32), er.view(torch.int32))
    _, rr, _ = kg_rank_ref(E, hs, rs, t[sample], torch.arange(N))
    assert torch.equal(rank[sample.cuda()].cpu(), rr)
    assert torch.equal(energy[sample.cuda()].cpu().view(torch.int32), E[torch.arange(6), t[sample]].view(torch.int32))

"""Pins the CPU oracle (oracle/kgat_oracle.py) to the golden vectors produced by running the
unmodified reference (oracle/make_golden.py).  CPU only.

Tolerance: the oracle and the reference are both fp32 PyTorch-CPU programs following the same
arithmetic, so floating-point outputs are compared at 1e-6 normwise-relative
(max|a-b| / max|b|); integer / index outputs must be bit-exact.
"""

from __future__ import annotations

import numpy as np
import torch

from conftest import rel_err
from oracle import kgat_oracle as O

TOL = 1e-6


def _masks(g, widths):
    out = []
    for l, w in enumerate(widths):
        keep = torch.from_numpy(g.unpack_mask(f"msg_mask{l}", w))
        out.append(keep.float() / (1 - 0.1))
    return out


def test_state_dict_key_set(golden_model):
    keys = set(golden_model["state_dict_keys"].tolist())
    mine = set(O.init_params(10, 4).keys()) | {"attentive_matrix"}
    assert keys == mine


def test_propagation_eval(golden_model):
    g = golden_model
    table = g.cut("all_embeddings_eval", O.all_embeddings(g.params(), g.att_coo()))
    assert table.shape == g["all_embeddings_eval"].shape
    assert rel_err(table, g["all_embeddings_eval"]) < TOL


def test_cf_loss_and_grads_eval(golden_model):
    g = golden_model
    p = g.params()
    for v in p.values():
        v.requires_grad_(True)
    loss = O.cf_loss(p, g.att_coo(), *(torch.from_numpy(g[k]) for k in ("cf_users", "cf_pos", "cf_neg")))
    loss.backward()
    assert rel_err(loss.detach(), g["cf_loss_eval"]) < TOL
    for k in g.keys():
        if k.startswith("cf_eval_grad::"):
            assert rel_err(g.cut(k, p[k[len("cf_eval_grad::") :]].grad), g[k]) < 1e-5, k


def test_cf_loss_train_mode_with_injected_masks(golden_model):
    g = golden_model
    p = g.params()
    for v in p.values():
        v.requires_grad_(True)
    loss = O.cf_loss(
        p,
        g.att_coo(),
        *(torch.from_numpy(g[k]) for k in ("cf_users", "cf_pos", "cf_neg")),
        drop_masks=_masks(g, [64, 32, 16]),
    )
    loss.backward()
    assert rel_err(loss.detach(), g["cf_loss_train"]) < TOL
    k = "cf_train_grad::_user_entity_embedding.weight"
    assert rel_err(g.cut(k, p["_user_entity_embedding.weight"].grad), g[k]) < 1e-5


def test_kg_loss_and_grads(golden_model):
    g = golden_model
    p = g.params()
    for v in p.values():
        v.requires_grad_(True)
    loss = O.kg_loss(p, *(torch.from_numpy(g[k]) for k in ("kg_heads", "kg_rels", "kg_pos", "kg_neg")))
    loss.backward()
    assert rel_err(loss.detach(), g["kg_loss"]) < TOL
    for name in ("_user_entity_embedding.weight", "_relation_embedding.weight", "_trans_matrix"):
        assert rel_err(g.cut("kg_grad::" + name, p[name].grad), g["kg_grad::" + name]) < 1e-5, name


def test_attention_refresh_eval(golden_model):
    g = golden_model
    with torch.no_grad():
        r, c, v = O.attention_refresh(g.params(), g["heads"], g["relations"], g["tails"], g["adjacency_relations"], g.node_num)
    assert bool(g["att_eval_is_coalesced"])
    np.testing.assert_array_equal(torch.stack([r, c]).numpy(), g["att_eval_indices"])  # bit-exact structure
    assert rel_err(v, g["att_eval_values"]) < 1e-5
    # the refreshed structure is the coalesced (row, col)-sorted initial structure
    np.testing.assert_array_equal(g["att_eval_indices"], np.vstack([g["att_rows"], g["att_cols"]]))


def test_attention_refresh_train_mode_with_injected_head_masks(golden_model):
    g = golden_model
    masks = {}
    for r in g["adjacency_relations"].tolist():
        keep = torch.from_numpy(g.unpack_mask(f"head_mask_r{r}", 8))
        masks[r] = keep.float() / (1 - 0.1)
    with torch.no_grad():
        _, _, v = O.attention_refresh(
            g.params(), g["heads"], g["relations"], g["tails"], g["adjacency_relations"], g.node_num, head_masks=masks
        )
    assert rel_err(v, g["att_train_values"]) < 1e-5


def test_numpy_segment_softmax_matches_torch_sparse_softmax(golden_model):
    g = golden_model
    p = g.params()
    rows, cols, vals = [], [], []
    heads = torch.from_numpy(g["heads"]).long()
    tails = torch.from_numpy(g["tails"]).long()
    rels = torch.from_numpy(g["relations"]).long()
    with torch.no_grad():
        for r in g["adjacency_relations"].tolist():
            sel = torch.where(rels == r)[0]
            rows.append(heads[sel])
            cols.append(tails[sel])
            vals.append(O.attention_by_relation(p, heads[sel], tails[sel], r, g.node_num))
    r_, c_, v_ = O.segment_softmax_coalesced(torch.cat(rows).numpy(), torch.cat(cols).numpy(), torch.cat(vals).numpy(), g.node_num)
    np.testing.assert_array_equal(np.vstack([r_, c_]), g["att_eval_indices"])
    assert rel_err(v_, g["att_eval_values"]) < 1e-5


def _refreshed_att(g):
    idx = torch.from_numpy(g["att_eval_indices"])
    return torch.sparse_coo_tensor(idx, torch.from_numpy(g["att_eval_values"].copy()), size=(g.node_num, g.node_num))


def test_predict_and_ranking(golden_model):
    g = golden_model
    users = torch.from_numpy(g["pred_users"])
    items = torch.arange(int(g["item_num"]))
    with torch.no_grad():
        scores = O.predict_scores(g.params(), _refreshed_att(g), users, items)
    assert rel_err(scores, g["pred_scores"]) < 1e-5
    train_dict, test_dict = g.ragged("train_dict"), g.ragged("test_dict")
    # ranking on the reference's own scores must be index-exact wherever the score is finite; the
    # order inside the masked -inf tail is implementation-defined in the reference's unstable
    # torch.sort (it never reaches the metrics: train and test items are disjoint) -> compare as sets
    idx = O.rank_items(torch.from_numpy(g["pred_scores"].copy()), train_dict, g["pred_users"]).numpy()
    for i, u in enumerate(g["pred_users"].tolist()):
        n_fin = int(g["item_num"]) - len(set(train_dict[u]))
        np.testing.assert_array_equal(idx[i, :n_fin], g["rank_indices"][i, :n_fin])
        assert set(idx[i, n_fin:].tolist()) == set(g["rank_indices"][i, n_fin:].tolist()) == set(train_dict[u])
    m = O.metrics_at_k(torch.from_numpy(g["pred_scores"].copy()), train_dict, test_dict, g["pred_users"], int(g["item_num"]), [20, 40])
    for k in (20, 40):
        for name in ("precision", "recall", "ndcg"):
            np.testing.assert_allclose(m[k][name], g[f"metric_{name}@{k}"], rtol=1e-6, atol=0, equal_nan=True)


def test_optimiser_trajectory(golden_model):
    """CF, CF, KG, KG, refresh, CF with two independent Adam states (model.py:393-419)."""
    g = golden_model
    p = g.params()
    n = g.node_num
    att = g.att_coo()
    cf_b = [torch.from_numpy(g[k]) for k in ("cf_users", "cf_pos", "cf_neg")]
    kg_b = [torch.from_numpy(g[k]) for k in ("kg_heads", "kg_rels", "kg_pos", "kg_neg")]
    state = {"cf": {}, "kg": {}}
    steps = {"cf": 0, "kg": 0}
    lr = {"cf": 1e-3, "kg": 1e-4}
    losses = []

    def train(kind, loss_fn):
        leaves = {k: v.clone().requires_grad_(True) for k, v in p.items()}
        loss = loss_fn(leaves)
        loss.backward()
        steps[kind] += 1
        for k, leaf in leaves.items():
            if leaf.grad is None:
                continue
            m, v = state[kind].setdefault(k, (torch.zeros_like(leaf), torch.zeros_like(leaf)))
            O.adam_step(p[k], leaf.grad, m, v, steps[kind], lr[kind])
        losses.append(float(loss))

    for what in ("cf", "cf", "kg", "kg", "att", "cf"):
        if what == "cf":
            train("cf", lambda q: O.cf_loss(q, att, *cf_b))
        elif what == "kg":
            train("kg", lambda q: O.kg_loss(q, *kg_b))
        else:
            with torch.no_grad():
                r, c, v = O.attention_refresh(p, g["heads"], g["relations"], g["tails"], g["adjacency_relations"], n)
            att = torch.sparse_coo_tensor(torch.stack([r, c]), v, size=(n, n))
    np.testing.assert_allclose(losses, g["traj_losses"], rtol=2e-6)
    for k in g.keys():
        if k.startswith("traj_param::"):
            assert rel_err(g.cut(k, p[k[len("traj_param::") :]]), g[k]) < 1e-5, k
    assert rel_err(att._values(), g["traj_att_values"]) < 1e-5


# ---------------------------------------------------------------------------------------------
# graph construction + samplers against the real Preprocess.run
# ---------------------------------------------------------------------------------------------


def test_ckg_construction_bit_exact(golden_pre):
    g = golden_pre
    out = O.build_ckg(int(g["user_num"]), int(g["entity_num"]), int(g["kg_relation_num"]), g["interactions"], g["triples"])
    assert out["adjacency_relations"] == g["adjacency_relations"].tolist() == [0, 5, 1, 6, 2, 7, 3, 8, 4, 9]
    np.testing.assert_array_equal(out["heads"], g["all_heads"])
    np.testing.assert_array_equal(out["relations"], g["all_relations"])
    np.testing.assert_array_equal(out["tails"], g["all_tails"])
    np.testing.assert_array_equal(out["values"].view(np.uint32), g["all_values"].view(np.uint32))
    np.testing.assert_array_equal(np.vstack([out["att_rows"], out["att_cols"]]), g["att_indices"])
    np.testing.assert_array_equal(out["att_vals"].view(np.uint32), g["att_values"].view(np.uint32))
    assert str(g["heads_tensor_dtype"]) == "torch.int32"


def _kg_dict(g):
    heads, ptr, rt = g["kg_dict_heads"], g["kg_dict_ptr"], g["kg_dict_rt"]
    return {int(h): [tuple(x) for x in rt[ptr[i] : ptr[i + 1]].tolist()] for i, h in enumerate(heads)}


def test_samplers_replay_reference_rng_stream(golden_pre):
    g = golden_pre
    train = g.ragged("train_dict")
    rng = np.random.default_rng(2024)
    for i in range(3):
        u, p, n = O.sample_cf_batch(rng, train, int(g["item_num"]), 8)
        np.testing.assert_array_equal(np.stack([u, p, n]), g[f"cf_batch{i}"])
    rng = np.random.default_rng(2025)
    kd = _kg_dict(g)
    n_nodes = int(g["user_num"]) + int(g["entity_num"])
    for i in range(3):
        b = O.sample_kg_batch(rng, kd, n_nodes, 16)
        np.testing.assert_array_equal(np.stack(b), g[f"kg_batch{i}"])


def test_canonical_kgat_attention_oracle_on_a_hand_case():
    """oracle.attention_refresh_kgat restates the paper's pi(h, r, t) = (W_r e_t)^T tanh(W_r e_h + e_r): check it against the formula
    written out by hand on a 3-node graph, incl. a duplicate (h, t) under two relations (summed before the softmax)."""
    torch.manual_seed(0)
    n, d, r = 3, 4, 2
    p = {"_user_entity_embedding.weight": torch.randn(n, d), "_relation_embedding.weight": torch.randn(r, d), "_trans_matrix": torch.randn(r, d, d)}
    heads, rels, tails = [0, 0, 0, 1], [0, 1, 0, 1], [1, 1, 2, 2]
    rows, cols, vals = O.attention_refresh_kgat(p, heads, rels, tails, [0, 1], n)

    def pi(h, rr, t):
        e, w, er = p["_user_entity_embedding.weight"], p["_trans_matrix"][rr], p["_relation_embedding.weight"][rr]
        return float(((e[t] @ w) * torch.tanh(e[h] @ w + er)).sum())

    s01, s02 = pi(0, 0, 1) + pi(0, 1, 1), pi(0, 0, 2)
    m = max(s01, s02)
    z = np.exp(s01 - m) + np.exp(s02 - m)
    assert rows.tolist() == [0, 0, 1] and cols.tolist() == [1, 2, 2]
    np.testing.assert_allclose(vals.numpy(), [np.exp(s01 - m) / z, np.exp(s02 - m) / z, 1.0], rtol=1e-5)

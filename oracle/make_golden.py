"""Generate the golden vectors under tests/golden/ by running the UNMODIFIED reference.

    python oracle/make_golden.py <checkout of the reference repository>

It imports ``src.model.KGAT.{model,preprocess}`` and ``src.utils.metrics_calculator`` from
that checkout (read-only; bytecode writing disabled), drives them with seeded inputs and
stores inputs + outputs as ``.npz`` files (``oracle/golden_io.py``: files above 1 MB are stored compacted).  The reference publishes no golden vectors of its own
(SURVEY.md section 8c), so these files are what pins the oracle and the CUDA path to the reference.

TEST INFRASTRUCTURE - not product code.
"""

from __future__ import annotations

import importlib
import os
import sys
import tempfile
from argparse import Namespace
from pathlib import Path

import numpy as np

sys.dont_write_bytecode = True
REPO = Path(__file__).resolve().parents[1]
if len(sys.argv) != 2:
    raise SystemExit("usage: python oracle/make_golden.py <checkout of the reference repository>")
REF = Path(sys.argv[1]).resolve()
sys.path.insert(0, str(REF))
sys.path.insert(0, str(REPO))

import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

pkg = importlib.import_module("problem-recommender-system-using-kgat-in-codeforces_b200.synthetic")
from oracle import golden_io  # noqa: E402

from src.model.KGAT import preprocess as ref_pre  # noqa: E402
from src.model.KGAT.model import KGAT, KGATArgs, KGATMode  # noqa: E402
from src.type import (  # noqa: E402
    Contest,
    Dataset,
    Problem,
    Rating,
    Relation,
    RelationType,
    Submission,
    SubmissionHistory,
    Tag,
    User,
)
from src.utils.metrics_calculator import Metrics, metrics_at_k  # noqa: E402

SEED = 2024
OUT = REPO / "tests" / "golden"


def sd_to_np(sd):
    out = {}
    for k, v in sd.items():
        if v.is_sparse:
            continue
        out["param::" + k] = v.detach().cpu().numpy().copy()
    return out


# ----------------------------------------------------------------------------------------------
# 1. a tiny Codeforces-like Dataset through the real Preprocess.run (rows P1-P5)
# ----------------------------------------------------------------------------------------------


def tiny_dataset(rng):
    n_users, n_problems, n_contests, n_tags, n_ratings = 12, 30, 7, 6, 4
    users = [User(id=i, handle=f"u{i}", rating=1500, max_rating=1600) for i in range(n_users)]
    contests = [
        Contest(id=100 + c, name=f"c{c}", type="CF", division_id=(None if c == 3 else int(rng.integers(0, 5))))
        for c in range(n_contests)
    ]
    problems = []
    for p in range(n_problems):
        tags = [Tag(id=int(t), name=f"t{t}") for t in sorted(set(rng.integers(0, n_tags, size=int(rng.integers(0, 4))).tolist()))]
        rating = None if p % 7 == 0 else Rating(id=int(rng.integers(0, n_ratings)), value=800)
        problems.append(
            Problem(
                id=p,
                contest_id=100 + int(rng.integers(0, n_contests)),
                index="A",
                name=f"p{p}",
                type="PROGRAMMING",
                tags=tags,
                rating=rating,
            )
        )
    histories = []
    sid = 0
    for u in users:
        n_sub = int(rng.integers(10, 22))
        chosen = rng.choice(n_problems, size=n_sub, replace=False)
        subs = []
        for j, p in enumerate(chosen.tolist()):
            subs.append(Submission(id=sid, problem=problems[p], created_at=f"2024-01-{(j % 28) + 1:02d}T00:00:{sid % 60:02d}", result="OK"))
            sid += 1
        histories.append(SubmissionHistory(user=u, submissions=subs))
    relations = [Relation(id=r.value, name=r.name) for r in RelationType]
    return Dataset(users=users, all_submission_history=histories, contests=contests, problems=problems, relations=relations)


def golden_preprocess():
    rng = np.random.default_rng(SEED)
    ds = tiny_dataset(rng)
    cwd = os.getcwd()
    with tempfile.TemporaryDirectory() as tmp:
        # json_writer writes to cwd/../../../dataset (kg_triplets_generator.py:188-195)
        (Path(tmp) / "dataset").mkdir()
        work = Path(tmp) / "a" / "b" / "c"
        work.mkdir(parents=True)
        os.chdir(work)
        try:
            pre = ref_pre.Preprocess(args=Namespace(sm=True), dataset=ds, cf_batch_size=8, kg_batch_size=16, device=torch.device("cpu"))
            pre.run(dataset_name="training")
        finally:
            os.chdir(cwd)
    triples = np.array([[t.head, t.relation, t.tail] for t in pre.triplets], np.int64)
    att = pre.attentive_matrix
    out = {
        "user_num": pre.user_num,
        "entity_num": pre.entity_num,
        "item_num": pre.item_num,
        "kg_relation_num": len(RelationType),
        "interactions": np.asarray(pre.interaction_matrix, np.int64),
        "triples": triples,
        "adjacency_relations": np.array(pre.adjacency_relations, np.int64),
        "all_heads": np.array(pre.all_heads, np.int64),
        "all_relations": np.array(pre.all_relation_indices, np.int64),
        "all_tails": np.array(pre.all_tails, np.int64),
        "all_values": np.array(pre.all_values, np.float32),
        "att_indices": att._indices().numpy(),
        "att_values": att._values().numpy(),
        "att_is_coalesced": np.array(att.is_coalesced()),
    }
    # dtype facts the boundary must accept (SURVEY.md section 8)
    out["heads_tensor_dtype"] = np.array(str(torch.tensor(pre.all_heads).dtype))
    # interaction dict (train) as ragged arrays, in the reference's own list order
    users = sorted(pre.train_interaction_dict.keys())
    out["train_dict_ptr"] = np.cumsum([0] + [len(pre.train_interaction_dict[u]) for u in users])
    out["train_dict_items"] = np.concatenate([np.array(pre.train_interaction_dict[u], np.int64) for u in users])
    # kg_dict in the reference's list order (head order = dict insertion order)
    kd_heads = list(pre._kg_dict.keys())
    out["kg_dict_heads"] = np.array(kd_heads, np.int64)
    out["kg_dict_ptr"] = np.cumsum([0] + [len(pre._kg_dict[h]) for h in kd_heads])
    out["kg_dict_rt"] = np.concatenate([np.array(pre._kg_dict[h], np.int64).reshape(-1, 2) for h in kd_heads])
    # samplers under an injected seeded Generator (quirk Q5)
    ref_pre.rng = np.random.default_rng(SEED)
    for i in range(3):
        u, p, n = pre.generate_cf_batch()
        out[f"cf_batch{i}"] = np.stack([u.numpy(), p.numpy(), n.numpy()])
    ref_pre.rng = np.random.default_rng(SEED + 1)
    for i in range(3):
        h, r, pt, nt = pre.generate_kg_batch()
        out[f"kg_batch{i}"] = np.stack([np.array(x, np.int64) for x in (h, r, pt, nt)])
    np.savez_compressed(OUT / "preprocess_tiny.npz", **out)
    print("preprocess_tiny:", {k: (v.shape if hasattr(v, "shape") else v) for k, v in out.items() if k.startswith("all_") or k == "adjacency_relations"})


# ----------------------------------------------------------------------------------------------
# 2. model goldens on synthetic CKGs (rows A1-A10, M1)
# ----------------------------------------------------------------------------------------------


def coo_from_graph(g):
    idx = torch.from_numpy(np.vstack([g.att_rows, g.att_cols])).long()
    return torch.sparse_coo_tensor(idx, torch.from_numpy(g.att_vals), size=(g.node_num, g.node_num))


def grads_of(model, names):
    sd = dict(model.named_parameters())
    return {"grad::" + n: sd[n].grad.detach().clone().numpy() for n in names if sd[n].grad is not None}


def golden_model(tag: str, shape: str, dup: int, cf_b: int, kg_b: int, n_pred_users: int, sample: dict | None = None):
    g = pkg.make_ckg(shape, seed=SEED, duplicate_pairs=dup)
    n = g.node_num
    torch.manual_seed(SEED)
    model = KGAT(KGATArgs(user_num=g.user_num, entity_num=g.entity_num, relation_num=g.relation_num, attentive_matrix=coo_from_graph(g)))
    # make LayerNorm affine non-trivial so the kernel's gamma/beta path is exercised
    with torch.no_grad():
        model._multi_head_attention._layer_norm.weight.add_(0.1 * torch.randn(64))
        model._multi_head_attention._layer_norm.bias.add_(0.1 * torch.randn(64))
    out = {
        "user_num": g.user_num,
        "entity_num": g.entity_num,
        "item_num": g.item_num,
        "relation_num": g.relation_num,
        "adjacency_relations": np.array(g.adjacency_relations, np.int64),
        "heads": g.heads,
        "relations": g.relations,
        "tails": g.tails,
        "att_rows": g.att_rows,
        "att_cols": g.att_cols,
        "att_vals": g.att_vals,
    }
    out.update(sd_to_np(model.state_dict()))
    out["state_dict_keys"] = np.array(list(model.state_dict().keys()))

    rng = np.random.default_rng(SEED + 7)
    users = torch.from_numpy(rng.integers(0, g.user_num, size=cf_b))
    pos = torch.from_numpy(rng.integers(0, g.item_num, size=cf_b))
    neg = torch.from_numpy(rng.integers(0, g.item_num, size=cf_b))
    kg_sel = rng.integers(0, g.nnz, size=kg_b)
    kg_h = torch.from_numpy(g.heads[kg_sel].astype(np.int64))
    kg_r = torch.from_numpy(g.relations[kg_sel].astype(np.int64))
    kg_pt = torch.from_numpy(g.tails[kg_sel].astype(np.int64))
    kg_nt = torch.from_numpy(rng.integers(0, n, size=kg_b))
    out.update(cf_users=users.numpy(), cf_pos=pos.numpy(), cf_neg=neg.numpy())
    out.update(kg_heads=kg_h.numpy(), kg_rels=kg_r.numpy(), kg_pos=kg_pt.numpy(), kg_neg=kg_nt.numpy())

    cf_names = ["_user_entity_embedding.weight"] + [f"_aggregator_layers.{l}.linear{k}.{w}" for l in range(3) for k in (1, 2) for w in ("weight", "bias")]
    kg_names = ["_user_entity_embedding.weight", "_relation_embedding.weight", "_trans_matrix"]

    # (b) eval-mode propagation
    model.eval()
    with torch.no_grad():
        out["all_embeddings_eval"] = model._build_cf_embeddings().numpy()
    # (c) CF loss + grads, eval mode (no dropout)
    model.zero_grad()
    loss = model(users, pos, neg, mode=KGATMode.TRAIN_CF)
    loss.backward()
    out["cf_loss_eval"] = loss.detach().numpy()
    out.update({"cf_eval_" + k: v for k, v in grads_of(model, cf_names).items()})
    # (d) CF loss + grads, train mode, masks re-derivable by F.dropout(ones) under the same seed
    model.train()
    model.zero_grad()
    torch.manual_seed(SEED + 11)
    loss = model(users, pos, neg, mode=KGATMode.TRAIN_CF)
    loss.backward()
    out["cf_loss_train"] = loss.detach().numpy()
    out.update({"cf_train_" + k: v for k, v in grads_of(model, ["_user_entity_embedding.weight", "_aggregator_layers.0.linear1.weight", "_aggregator_layers.2.linear2.bias"]).items()})
    torch.manual_seed(SEED + 11)
    for l, d_out in enumerate([64, 32, 16]):
        m = F.dropout(torch.ones(n, d_out), p=0.1, training=True)
        out[f"msg_mask{l}"] = np.packbits((m != 0).numpy(), axis=1)
    # (e) KG loss + grads
    model.eval()
    model.zero_grad()
    loss = model(kg_h, kg_r, kg_pt, kg_nt, mode=KGATMode.TRAIN_KG)
    loss.backward()
    out["kg_loss"] = loss.detach().numpy()
    out.update({"kg_" + k: v for k, v in grads_of(model, kg_names).items()})
    model.zero_grad()

    # (f) attention refresh: eval mode, then train mode with a known seed
    heads_t = torch.tensor(list(g.heads))  # int32, exactly like main.py:351-353
    rels_t = torch.tensor(g.relations.tolist())
    tails_t = torch.tensor(list(g.tails))
    rel_idx = torch.tensor(g.adjacency_relations)
    att0 = model.attentive_matrix.data
    model.eval()
    with torch.no_grad():
        model(heads_t, rels_t, tails_t, rel_idx, mode=KGATMode.UPDATE_ATTENTION)
    a = model.attentive_matrix.data
    out["att_eval_indices"] = a._indices().numpy()
    out["att_eval_values"] = a._values().numpy()
    out["att_eval_is_coalesced"] = np.array(a.is_coalesced())
    # predict + ranking after the eval refresh
    pred_users = torch.from_numpy(rng.choice(g.user_num, size=n_pred_users, replace=False))
    items = torch.arange(g.item_num)
    with torch.no_grad():
        scores = model(pred_users, items, mode=KGATMode.PREDICT)
    out["pred_users"] = pred_users.numpy()
    out["pred_scores"] = scores.numpy()
    train_dict = {u: g.train_dict[u] for u in range(g.user_num)}
    test_dict = {u: g.test_dict[u] for u in range(g.user_num)}
    sc = scores.clone()
    md = metrics_at_k(sc, train_dict, test_dict, pred_users.numpy(), items.numpy(), [20, 40])
    for k in (20, 40):
        for m in Metrics:
            out[f"metric_{m.value}@{k}"] = md[k][m]
    _, rank = torch.sort(sc, descending=True)  # sc was masked in place by metrics_at_k
    out["rank_indices"] = rank.numpy().astype(np.int32)
    out["train_dict_ptr"] = np.cumsum([0] + [len(train_dict[u]) for u in range(g.user_num)])
    out["train_dict_items"] = np.concatenate([np.array(train_dict[u], np.int64) for u in range(g.user_num)])
    out["test_dict_ptr"] = np.cumsum([0] + [len(test_dict[u]) for u in range(g.user_num)])
    out["test_dict_items"] = np.concatenate([np.array(test_dict[u], np.int64) for u in range(g.user_num)] + [np.zeros(0, np.int64)])

    # train-mode refresh (quirk Q2): per relation F.dropout(ones(n_r, 8, 1, 1)) in loop order
    model.attentive_matrix.data = att0
    model.train()
    torch.manual_seed(SEED + 13)
    with torch.no_grad():
        model(heads_t, rels_t, tails_t, rel_idx, mode=KGATMode.UPDATE_ATTENTION)
    a = model.attentive_matrix.data
    out["att_train_values"] = a._values().numpy()
    torch.manual_seed(SEED + 13)
    for r in g.adjacency_relations:
        n_r = int((g.relations == r).sum())
        m = F.dropout(torch.ones(n_r, 8, 1, 1), p=0.1, training=True)
        out[f"head_mask_r{r}"] = np.packbits((m.view(n_r, 8) != 0).numpy(), axis=1)

    # (h) optimiser trajectory in eval mode (deterministic): CF, CF, KG, KG, refresh, CF
    model.attentive_matrix.data = att0
    model.eval()
    model.build_optimizer(cf_lr=1e-3, kg_lr=1e-4)
    losses = []
    for step in ("cf", "cf", "kg", "kg", "att", "cf"):
        if step == "cf":
            l = model(users, pos, neg, mode=KGATMode.TRAIN_CF)
            l.backward()
            model.update_cf_weights()
            losses.append(l.item())
        elif step == "kg":
            l = model(kg_h, kg_r, kg_pt, kg_nt, mode=KGATMode.TRAIN_KG)
            l.backward()
            model.update_kg_weights()
            losses.append(l.item())
        else:
            with torch.no_grad():
                model(heads_t, rels_t, tails_t, rel_idx, mode=KGATMode.UPDATE_ATTENTION)
    out["traj_losses"] = np.array(losses, np.float64)
    out.update({"traj_" + k: v for k, v in sd_to_np(model.state_dict()).items() if "multi_head" not in k})
    out["traj_att_values"] = model.attentive_matrix.data._values().numpy()
    if sample:  # keeps the file under 1 MB: inputs as digests + recipe, the largest outputs as a seeded row sample
        out = golden_io.compact(out, (shape, SEED, dup), sample)
    np.savez_compressed(OUT / f"model_{tag}.npz", **out)
    size = (OUT / f"model_{tag}.npz").stat().st_size
    print(f"model_{tag}: N={n} nnz={g.nnz} att_nnz={g.att_rows.size} R={g.relation_num} file={size / 1e6:.2f} MB losses={losses}")


# ----------------------------------------------------------------------------------------------
# 3. end-to-end training tier (SURVEY.md section 4): the unmodified reference trained for a few epochs in train() mode
#    (message dropout and attention dropout live), several seeds -> the band the drop-in's metrics must fall into
# ----------------------------------------------------------------------------------------------


def golden_training(tag: str = "train_small", shape: str = "small", epochs: int = 3, seeds=(0, 1, 2, 3, 4, 5, 6, 7)):
    trainer = importlib.import_module("problem-recommender-system-using-kgat-in-codeforces_b200.trainer")
    g = pkg.make_ckg(shape, seed=SEED)
    users = np.array(sorted(u for u, v in g.test_dict.items() if len(v) > 0), np.int64)
    items = np.arange(g.item_num)
    recs, ndcgs, cf_losses, kg_losses = [], [], [], []
    for seed in seeds:
        torch.manual_seed(1000 + seed)  # parameter init + every dropout draw of the run
        model = KGAT(KGATArgs(user_num=g.user_num, entity_num=g.entity_num, relation_num=g.relation_num, attentive_matrix=coo_from_graph(g)))
        model.build_optimizer(cf_lr=1e-3, kg_lr=1e-4)
        heads = torch.tensor(list(g.heads))  # int32, like main.py:351-353
        rels = torch.tensor(g.relations.tolist())
        tails = torch.tensor(list(g.tails))
        rel_idx = torch.tensor(g.adjacency_relations)
        cf_l, kg_l = [], []
        for ep in range(epochs):
            data = trainer.EpochData.sample(g, seed=7000 + 100 * seed + ep)  # the batches the drop-in test regenerates
            model.train()
            tot = 0.0
            for i in range(data.n_cf):
                b = [torch.from_numpy(a[i]) for a in data.cf]
                loss = model(*b, mode=KGATMode.TRAIN_CF)
                loss.backward()
                model.update_cf_weights()
                tot += loss.item()
            cf_l.append(tot / data.n_cf)
            tot = 0.0
            for i in range(data.n_kg):
                b = [torch.from_numpy(a[i]) for a in data.kg]
                loss = model(*b, mode=KGATMode.TRAIN_KG)
                loss.backward()
                model.update_kg_weights()
                tot += loss.item()
            kg_l.append(tot / data.n_kg)
            model(heads, rels, tails, rel_idx, mode=KGATMode.UPDATE_ATTENTION)  # still in train(): attention dropout live (Q2)
        model.eval()
        with torch.no_grad():
            scores = model(torch.from_numpy(users), torch.from_numpy(items), mode=KGATMode.PREDICT)
        md = metrics_at_k(scores.clone(), g.train_dict, g.test_dict, users, items, [20])
        recs.append(float(np.nanmean(md[20][Metrics.RECALL])))
        ndcgs.append(float(np.nanmean(md[20][Metrics.NDCG])))
        cf_losses.append(cf_l)
        kg_losses.append(kg_l)
        print(f"train[{tag}] seed {seed}: recall@20 {recs[-1]:.4f} ndcg@20 {ndcgs[-1]:.4f} cf {cf_l} kg {kg_l}")
    np.savez_compressed(OUT / f"{tag}.npz", shape=np.array(shape), epochs=np.array(epochs), seeds=np.array(seeds), recall20=np.array(recs),
                        ndcg20=np.array(ndcgs), cf_loss=np.array(cf_losses), kg_loss=np.array(kg_losses))


if __name__ == "__main__":
    OUT.mkdir(parents=True, exist_ok=True)
    torch.set_num_threads(4)
    golden_preprocess()
    golden_model("tiny", "tiny", dup=0, cf_b=16, kg_b=32, n_pred_users=8)
    golden_model("tiny_dup", "tiny", dup=40, cf_b=16, kg_b=32, n_pred_users=8)
    E = "_user_entity_embedding.weight"
    golden_model("small", "small", dup=0, cf_b=64, kg_b=128, n_pred_users=16,
                 sample={"all_embeddings_eval": 256, **{f"{p}::{E}": 256 for p in ("cf_eval_grad", "cf_train_grad", "kg_grad", "traj_param")},
                         "kg_grad::_trans_matrix": 6, "traj_param::_trans_matrix": 6})
    golden_training()

"""The deterministic gradient sums of the fused TransR step (transr_reduce_kernel) and the BPR backward on the batch patterns
a real epoch produces and the uniform fixtures elsewhere do not: every sample in one relation, one hot relation plus a long
tail, one node in many slots (more than 32 for BPR), batches of 1, 37 and 512, and batches large enough that the id slots are
staged in more than one chunk.  Each case is checked against an fp64 autograd reference, and two calls must give the same bytes.
"""

from __future__ import annotations

import pytest
import torch

from conftest import rel_err
from oracle import kgat_oracle as O

pytestmark = pytest.mark.gpu

GTOL = 5e-5


@pytest.fixture(scope="module")
def ops():
    if not torch.cuda.is_available():
        pytest.skip("needs CUDA")
    import kgat_b200
    from kgat_b200 import ops

    kgat_b200._lib.load()
    return ops


def _relations(kind: str, B: int, R: int, g: torch.Generator) -> torch.Tensor:
    if kind == "one":
        return torch.full((B,), R - 1, dtype=torch.int64)
    r = torch.randint(1, R, (B,), generator=g)
    if kind == "hot":  # ~42 % of the batch in relation 0, as in the Amazon-book KG batches
        hot = torch.rand(B, generator=g) < 0.42
        r[hot] = 0
    return r


def _nodes(kind: str, n: int, B: int, g: torch.Generator) -> torch.Tensor:
    ids = torch.randint(0, n, (3, B), generator=g)
    if kind == "repeat":  # one node in many slots of every role, a few more in several
        hub = torch.rand(3, B, generator=g) < 0.3
        ids[hub] = 7
        few = torch.rand(3, B, generator=g) < 0.1
        ids[few] = torch.randint(0, 5, (int(few.sum()),), generator=g)
    return ids


def _transr_step(ops, emb, rel, W, h, r, pt, nt, reg):
    n, d = emb.shape
    B = h.numel()
    dev = emb.device
    loss, loss_sum = torch.zeros(1, device=dev), torch.zeros(1, device=dev)
    scratch = torch.full((ops.transr_scratch_numel(B, rel.shape[1]),), float("nan"), device=dev)
    slot = torch.full((n,), -1, dtype=torch.int32, device=dev)
    rows = torch.full((3 * B, d), 3.0, device=dev)
    g_rel, g_W = torch.full_like(rel, 5.0), torch.full_like(W, 5.0)
    ops.transr_step(emb, rel, W, h, r, pt, nt, reg, loss, loss_sum, scratch, slot, rows, g_rel, g_W)
    claimed = slot >= 0
    dense = torch.zeros_like(emb)
    dense[claimed] = rows[slot[claimed].long()]
    return loss, loss_sum, dense, g_rel, g_W


CASES = [  # (relations, nodes, B, d)
    ("one", "distinct", 512, 64),
    ("hot", "distinct", 512, 64),
    ("hot", "repeat", 512, 64),
    ("uniform", "repeat", 1, 64),
    ("hot", "repeat", 37, 64),
    ("hot", "repeat", 2048, 64),  # 6144 id slots: more than one staged chunk
    ("one", "repeat", 300, 32),
    ("hot", "repeat", 300, 128),
]


@pytest.mark.parametrize("rels_kind,nodes_kind,B,d", CASES)
def test_transr_step_gradients(ops, rels_kind, nodes_kind, B, d):
    g = torch.Generator().manual_seed(B * 131 + d)
    n, R, reg = 3000, 12, 1e-3
    emb = torch.randn(n, d, generator=g) * 0.1
    rel = torch.randn(R, d, generator=g) * 0.1
    W = torch.randn(R, d, d, generator=g) * 0.1
    r = _relations(rels_kind, B, R, g)
    ids = _nodes(nodes_kind, n, B, g)
    if nodes_kind == "distinct":
        ids = torch.randperm(n, generator=g)[: 3 * B].view(3, B)
    h, pt, nt = (x.contiguous() for x in ids)

    leaves = {"_user_entity_embedding.weight": emb.double().requires_grad_(True), "_relation_embedding.weight": rel.double().requires_grad_(True),
              "_trans_matrix": W.double().requires_grad_(True)}
    ref = O.kg_loss(leaves, h, r, pt, nt, reg=reg)
    ref.backward()

    args = [x.cuda() for x in (emb, rel, W, h, r, pt, nt)]
    loss, loss_sum, g_emb, g_rel, g_W = _transr_step(ops, *args, reg)
    assert rel_err(loss, ref.detach()) < 1e-5 and torch.equal(loss, loss_sum)
    for got, k in ((g_emb, "_user_entity_embedding.weight"), (g_rel, "_relation_embedding.weight"), (g_W, "_trans_matrix")):
        assert rel_err(got, leaves[k].grad) < GTOL, k
    again = _transr_step(ops, *args, reg)
    for a, b in zip((loss, loss_sum, g_emb, g_rel, g_W), again):
        assert torch.equal(a.view(torch.int32), b.view(torch.int32))


@pytest.mark.parametrize("nodes_kind,B", [("repeat", 1), ("repeat", 37), ("distinct", 256), ("repeat", 256), ("repeat", 2048)])
def test_bpr_backward_gradients(ops, nodes_kind, B):
    g = torch.Generator().manual_seed(B * 17 + len(nodes_kind))
    n, reg = 1200, 1e-2
    tabs = [torch.randn(n, w, generator=g) * 0.2 for w in (64, 32, 16)]
    ids = _nodes(nodes_kind, n, B, g)
    if nodes_kind == "repeat" and B >= 256:
        assert int((ids == 7).sum()) > 32  # the rescanning path of a node held by more than 32 slots
    u, p, q = (x.contiguous() for x in ids)
    leaves = [t.double().requires_grad_(True) for t in tabs]
    ref = O.bpr_loss_from_table(torch.cat(leaves, dim=1), u, p, q, reg=reg)
    ref.backward()

    ct = [t.cuda() for t in tabs]
    uc, pc, qc = u.cuda(), p.cuda(), q.cuda()
    loss, scratch = torch.zeros(1, device="cuda"), torch.empty(2 * B, device="cuda")
    ops.bpr_forward(ct, uc, pc, qc, reg, loss, scratch)
    assert rel_err(loss, ref.detach()) < 1e-5

    def backward():
        grads = [torch.zeros_like(t) for t in ct]
        ops.bpr_backward(ct, grads, uc, pc, qc, reg, scratch, torch.ones(1, device="cuda"))
        return grads

    first = backward()
    for got, leaf in zip(first, leaves):
        assert rel_err(got, leaf.grad) < GTOL
    for a, b in zip(first, backward()):
        assert torch.equal(a.view(torch.int32), b.view(torch.int32))

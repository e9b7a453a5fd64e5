"""The attention-refresh kernels (csrc/attention.cu) against float64 references, at d = 32, 64 and 128 (the three template
instances of every kernel).

* ``UPDATE_ATTENTION`` in eval mode, in train mode with injected per-head masks (p = 0.1 and 0.5, some edges with every head
  dropped) and with ``score_mode = "kgat"``, against ``oracle.kgat_oracle.attention_refresh`` / ``attention_refresh_kgat`` run on
  float64 parameters.  The synthetic graph has a hub row with more than 2,000 slots, rows of 33-100 slots, single-slot and empty
  rows, (h, t) pairs repeated under two or three relations, and more unique (tail, relation) pairs and edges than one pass of the
  pair and edge kernels' grids covers, so their grid-stride loops run.  Structure is compared bit-exactly; the weights normwise
  and per element with a relative floor of 1e-6 max|ref| (a 1e-3 weight of the hub row that is 1 % off fails).
* The stand-alone ``MultiHeadAttention.forward`` (``mha_forward_kernel``) with 1, 2, 4 and 8 heads, eval and with injected
  masks, against a float64 restatement here (which itself matches ``oracle.mha_forward`` at 8 heads).
* The in-kernel RNG of the head masks: each output row of a train-mode call is matched against all 256 float64 candidates; the
  match must be unique, every head must keep at the binomial rate and the heads must be pairwise independent (the two 16-bit
  halves of a Philox word go to different heads).  ``edge_scores_dropout_kernel`` draws its masks with the same code.

Measured maxima on a B200 (1,000 W), per element / normwise: refresh weights 2.6e-6 / 2.4e-7 (score_mode "kgat": 1.1e-5 /
3.0e-6), stand-alone MHA 2.1e-4 / 5.9e-7 (per element with the usual floor of 1e-3 max|ref|: LayerNorm outputs near zero); the
RNG match: best candidate <= 2.0e-6 (max abs difference), second best >= 0.18.  The bounds sit about 10x above the errors.
"""

from __future__ import annotations

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import elem_err, rel_err
from oracle import kgat_oracle as O

pytestmark = pytest.mark.gpu

DIMS = [32, 64, 128]
LAYERS = {32: [32, 16], 64: [64, 32, 16], 128: [128, 64]}
USERS, ENTITIES, RELATIONS = 50, 3000, 6
NODES = USERS + ENTITIES
HUB = 7
VAL_TOL = (3e-5, 3e-6)  # attention weights: per element (floor 1e-6 max|ref|), normwise
KGAT_TOL = (1.1e-4, 3e-5)  # score_mode "kgat": larger scores, so larger relative errors of the smaller weights
MHA_TOL = (2e-3, 6e-6)  # stand-alone MHA output: per element (floor 1e-3 max|ref|), normwise
MATCH_TOL = 2e-5  # max |y - candidate| of the matching head mask


@pytest.fixture(scope="module")
def kb():
    if not torch.cuda.is_available():
        pytest.skip("needs CUDA")
    import kgat_b200

    kgat_b200._lib.load()
    return kgat_b200


def make_edges(seed: int = 0):
    """(heads, relations, tails) in shuffled input order; see the module docstring for what the graph contains."""
    rng = np.random.default_rng(seed)
    h, t = [np.full(2100, HUB)], [rng.choice(NODES, 2100, replace=False)]
    for head in range(100, 180):
        k = int(rng.integers(33, 101))
        h.append(np.full(k, head))
        t.append(rng.choice(NODES, k, replace=False))
    h.append(np.arange(200, 240))
    t.append(rng.integers(0, NODES, 40))
    h, t = np.concatenate(h), np.concatenate(t)
    r = rng.integers(0, RELATIONS, h.size)
    dh, dt, dr = [h], [t], [r]
    for i in rng.choice(np.flatnonzero(h != HUB), 400, replace=False).tolist() + rng.choice(np.flatnonzero(h == HUB), 100, replace=False).tolist():
        others = rng.choice([x for x in range(RELATIONS) if x != r[i]], int(rng.integers(1, 3)), replace=False)
        dh.append(np.full(others.size, h[i]))
        dt.append(np.full(others.size, t[i]))
        dr.append(others)
    h, t, r = np.concatenate(dh), np.concatenate(dt), np.concatenate(dr)
    perm = rng.permutation(h.size)
    return h[perm].astype(np.int64), r[perm].astype(np.int64), t[perm].astype(np.int64)


@pytest.fixture(scope="module")
def edges(kb):
    h, r, t = make_edges()
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    n_pairs = np.unique(t * RELATIONS + r).size
    # one pass of the widest grids: pair_scores_kernel sms * 4 CTAs x 4 warps, edge_scores_dropout_kernel sms * 8 CTAs x 4 warps
    assert n_pairs > 16 * sms and h.size > 32 * sms, (n_pairs, h.size, sms)
    slots = np.unique(h * NODES + t) // NODES
    per_row = np.bincount(slots, minlength=NODES)
    assert per_row[HUB] >= 2000 and ((per_row >= 33) & (per_row <= 100)).sum() >= 50
    assert (per_row == 1).sum() >= 20 and (per_row == 0).sum() > 0
    assert np.unique(h * NODES + t).size < h.size  # duplicate (h, t) pairs
    return h, r, t


def make_model(kb, d: int):
    from kgat_b200.model import KGAT, KGATArgs

    torch.manual_seed(d)
    m = KGAT(KGATArgs(user_num=USERS, entity_num=ENTITIES, relation_num=RELATIONS, cf_embedding_dim=d, kg_embedding_dim=d,
                      layer_size=LAYERS[d]))
    with torch.no_grad():  # every parameter the score reads is away from its trivial init
        m._user_entity_embedding.weight.normal_()
        m._relation_embedding.weight.normal_()
        m._trans_matrix.normal_(0.0, d**-0.5)
        mha = m._multi_head_attention
        mha._layer_norm.weight.uniform_(0.5, 1.5)
        mha._layer_norm.bias.uniform_(-0.2, 0.2)
    return m.cuda()


def params64(m) -> dict:
    return {k: v.detach().cpu().double() for k, v in m.state_dict().items() if not v.is_sparse}


def refresh(m, h, r, t):
    from kgat_b200.model import KGATMode

    m(torch.from_numpy(h.astype(np.int32)).cuda(), torch.from_numpy(r).cuda(), torch.from_numpy(t.astype(np.int32)).cuda(),
      torch.arange(RELATIONS).cuda(), mode=KGATMode.UPDATE_ATTENTION)
    return m.attentive_matrix.data


def oracle64(fn, *args, **kw):
    """Run an oracle function with float64 as the default dtype (its degree weights are computed from integer counts)."""
    old = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)
    try:
        return fn(*args, **kw)
    finally:
        torch.set_default_dtype(old)


def check_matrix(a, rows, cols, vals, what: str, tol=None) -> None:
    tol = tol or VAL_TOL
    assert a.is_coalesced()
    assert torch.equal(a._indices().cpu(), torch.stack([rows, cols])), f"{what}: structure"
    got = a._values()
    e, n = elem_err(got, vals, floor_frac=1e-6), rel_err(got, vals)
    assert e < tol[0] and n < tol[1], f"{what}: per-element {e:.3g}, normwise {n:.3g}"
    assert float(vals[rows == HUB].median()) < 1e-3  # the hub row's weights are small: the per-element check is what sees them


def head_bits(n: int, p: float, seed: int) -> np.ndarray:
    """Per-edge keep bits (bit h keeps head h) at drop rate p; every 20th edge drops all heads, every 31st keeps all."""
    rng = np.random.default_rng(seed)
    keep = rng.random((n, 8)) >= p
    bits = np.packbits(keep, axis=1, bitorder="little")[:, 0]
    bits[::20] = 0
    bits[5::31] = 0xFF
    return bits


def unpack(bits: np.ndarray, heads: int = 8) -> torch.Tensor:
    return torch.from_numpy(np.unpackbits(bits[:, None], axis=1, bitorder="little")[:, :heads].astype(np.float64))


@pytest.mark.parametrize("d", DIMS)
def test_refresh_eval(kb, edges, d):
    h, r, t = edges
    m = make_model(kb, d).eval()
    a = refresh(m, h, r, t)
    ref = oracle64(O.attention_refresh, params64(m), h, r, t, list(range(RELATIONS)), NODES)
    check_matrix(a, *ref, f"eval d={d}")


@pytest.mark.parametrize("p", [0.1, 0.5])
@pytest.mark.parametrize("d", DIMS)
def test_refresh_train_injected_head_masks(kb, edges, d, p):
    h, r, t = edges
    m = make_model(kb, d).train()
    m._multi_head_attention._dropout.p = p
    bits = head_bits(h.size, p, seed=d)
    m._injected_head_bits = torch.from_numpy(bits)
    a = refresh(m, h, r, t)
    masks = {rel: unpack(bits[r == rel]) / (1 - p) for rel in range(RELATIONS)}
    ref = oracle64(O.attention_refresh, params64(m), h, r, t, list(range(RELATIONS)), NODES, head_masks=masks)
    check_matrix(a, *ref, f"train d={d} p={p}")


@pytest.mark.parametrize("d", DIMS)
def test_refresh_kgat_score_mode(kb, edges, d):
    h, r, t = edges
    m = make_model(kb, d).train()
    m.score_mode = "kgat"
    a = refresh(m, h, r, t)
    ref = oracle64(O.attention_refresh_kgat, params64(m), h, r, t, list(range(RELATIONS)), NODES)
    check_matrix(a, *ref, f"kgat d={d}", KGAT_TOL)


# ---------------------------------------------------------------------------------------------
# stand-alone MultiHeadAttention.forward
# ---------------------------------------------------------------------------------------------


def make_mha(d: int, heads: int, p: float = 0.1):
    from kgat_b200.multi_head_attention import MultiHeadAttention

    torch.manual_seed(100 * d + heads)
    mha = MultiHeadAttention(d, d, head_num=heads, dropout=p)
    with torch.no_grad():
        for lin in (mha._value_weight, mha._output):
            lin.bias.uniform_(-0.3, 0.3)
        mha._layer_norm.weight.uniform_(0.5, 1.5)
        mha._layer_norm.bias.uniform_(-0.2, 0.2)
    return mha.cuda()


def mha64(mha, x: torch.Tensor, keep: torch.Tensor | None = None) -> torch.Tensor:
    """float64 LayerNorm(Wo drop(Wv x + bv) + bo); ``keep``: (n, heads) 0/1 head mask, kept heads scaled by 1 / (1 - p)."""
    P = {k: v.double() for k, v in mha.kernel_params().items()}
    v = x.double() @ P["Wv"].T + P["bv"]
    if keep is not None:
        d = v.shape[1]
        v = v * keep.to(v).repeat_interleave(d // mha.head_num, dim=1) / (1 - mha.dropout_p)
    o = v @ P["Wo"].T + P["bo"]
    return F.layer_norm(o, (o.shape[1],), P["gamma"], P["beta"], mha.ln_eps)


def call_mha(mha, x: torch.Tensor) -> torch.Tensor:
    n, d = x.shape
    head = torch.randn(n, d, device="cuda")
    rel = torch.randn(d, device="cuda")
    y = mha(head, rel, x)
    assert y.shape == (n, 1, d)
    return y.squeeze(1)


def check_mha(got, ref, what: str) -> None:
    e, n = elem_err(got, ref), rel_err(got, ref)
    assert e < MHA_TOL[0] and n < MHA_TOL[1], f"{what}: per-element {e:.3g}, normwise {n:.3g}"


@pytest.mark.parametrize("heads", [1, 2, 4, 8])
@pytest.mark.parametrize("d", DIMS)
def test_mha_forward(kb, d, heads):
    """Eval and train mode with injected head masks (p = 0.1 and 0.5), n = 3000 rows (past one pass of the grid)."""
    n = 3000
    x = torch.randn(n, d, device="cuda")
    mha = make_mha(d, heads).eval()
    check_mha(call_mha(mha, x), mha64(mha, x), f"eval d={d} heads={heads}")
    if heads == 8:  # the restatement is the oracle's multi-head attention
        pre = {f"_multi_head_attention.{k}": v.detach().cpu().double() for k, v in mha.state_dict().items()}
        xd = x.cpu().double()
        ref = O.mha_forward(pre, torch.randn(n, d).double(), torch.randn(d).double(), xd).squeeze(1)
        assert rel_err(mha64(mha, x).cpu(), ref) < 1e-12
        keep = unpack(head_bits(n, 0.1, seed=3))
        ref = O.mha_forward(pre, torch.randn(n, d).double(), torch.randn(d).double(), xd, head_mask=keep / (1 - O.MHA_DROPOUT)).squeeze(1)
        assert rel_err(mha64(mha.train(), x, keep).cpu(), ref) < 1e-12
    for p in (0.1, 0.5):
        mha = make_mha(d, heads, p).train()
        bits = head_bits(n, p, seed=d + heads)
        mha._injected_head_bits = torch.from_numpy(bits).cuda()
        check_mha(call_mha(mha, x), mha64(mha, x, unpack(bits, heads)), f"train d={d} heads={heads} p={p}")


def test_mha_in_kernel_head_masks(kb):
    """Train mode with the kernel's own RNG at p = 0.5, 60,000 rows: recover each row's head mask as the unique float64
    candidate (of 256) within MATCH_TOL of the output, then check the per-head keep rate and the pairwise joint keep rate of
    the heads against binomial 6-sigma bounds."""
    d, heads, p, n = 64, 8, 0.5, 60000
    mha = make_mha(d, heads, p).train()
    x = torch.randn(n, d, device="cuda")
    y = call_mha(mha, x).double()
    P = {k: v.double() for k, v in mha.kernel_params().items()}
    depth = d // heads
    v = x.double() @ P["Wv"].T + P["bv"]
    cand = torch.tensor([[(m >> hd) & 1 for hd in range(heads)] for m in range(256)], dtype=torch.float64, device="cuda")
    masks = torch.empty(n, dtype=torch.long, device="cuda")
    for s in range(0, n, 2048):
        vs = v[s : s + 2048]
        # contribution of each head to Wo v: (rows, heads, d)
        contrib = torch.stack([vs[:, hd * depth : (hd + 1) * depth] @ P["Wo"][:, hd * depth : (hd + 1) * depth].T for hd in range(heads)], 1)
        o = P["bo"] + torch.einsum("mh,nhd->nmd", cand, contrib) / (1 - p)
        yc = F.layer_norm(o, (d,), P["gamma"], P["beta"], mha.ln_eps)
        err = (yc - y[s : s + 2048, None, :]).abs().amax(-1)
        two = err.topk(2, dim=1, largest=False)
        assert bool((two.values[:, 0] < MATCH_TOL).all()), f"rows without a matching head mask (best {float(two.values[:, 0].max()):.3g})"
        assert bool((two.values[:, 1] >= MATCH_TOL).all()), "rows with more than one matching head mask"
        masks[s : s + 2048] = two.indices[:, 0]
    keep = ((masks[:, None] >> torch.arange(heads, device="cuda")) & 1).double()
    q = 1 - p
    rate = keep.mean(0)
    assert float((rate - q).abs().max()) < 6 * (q * (1 - q) / n) ** 0.5, rate.tolist()
    joint = keep.T @ keep / n
    off = ~torch.eye(heads, dtype=torch.bool, device="cuda")
    assert float((joint - q * q)[off].abs().max()) < 6 * (q * q * (1 - q * q) / n) ** 0.5, joint.tolist()
    # heads 2k and 2k + 1 take the two 16-bit halves of Philox word k: they differ on about half of the rows
    for k in range(heads // 2):
        assert float((keep[:, 2 * k] != keep[:, 2 * k + 1]).double().mean()) > 0.45

"""Storage format of the model goldens (``tests/golden/model_*.npz``, written by ``oracle/make_golden.py``).

A golden file holds what the unmodified reference was given and what it returned.  A file that would exceed 1 MB
is stored compacted:

* the inputs are regenerated instead of stored: the file keeps the recipe (``recipe::shape``, ``recipe::seed``,
  ``recipe::duplicate_pairs``) and, for every input array, the SHA-256 of the array the reference was run on
  (``sha256::<key>``).  ``load`` rebuilds the synthetic CKG (``synthetic.make_ckg``) and the initial parameters
  (the KGAT constructor under ``torch.manual_seed`` plus the LayerNorm perturbation of ``make_golden.py``) and
  fails unless every rebuilt array matches its digest byte for byte;
* a large output keeps a fixed, seeded sample of its leading-dimension rows: ``rows::<key>`` lists the rows
  stored under ``<key>`` and ``shape::<key>`` the full shape.  ``cut`` restricts a computed output to them.

The rebuild ties a compacted golden to the project's own ``synthetic.make_ckg`` RNG stream and to the order in which the
KGAT constructor registers and initialises its parameters: a change to either makes ``load`` fail on the digest check
(by design -- the inputs would no longer be the reference's).  Regenerating the file then needs a checkout of the reference
(``python oracle/make_golden.py <checkout>``).

TEST INFRASTRUCTURE - not product code.
"""

from __future__ import annotations

import hashlib

import numpy as np
import torch

GRAPH_KEYS = ("heads", "relations", "tails", "att_rows", "att_cols", "att_vals")


def digest(a: np.ndarray) -> str:
    a = np.ascontiguousarray(a)
    return hashlib.sha256(f"{a.dtype.str}{a.shape}".encode() + a.tobytes()).hexdigest()


def rebuild_inputs(shape: str, seed: int, duplicate_pairs: int) -> dict[str, np.ndarray]:
    """The graph and the initial parameters ``make_golden.golden_model`` hands the reference."""
    from kgat_b200 import synthetic
    from kgat_b200.model import KGAT, KGATArgs

    g = synthetic.make_ckg(shape, seed=seed, duplicate_pairs=duplicate_pairs, with_dicts=False)
    out = {k: getattr(g, k) for k in GRAPH_KEYS}
    torch.manual_seed(seed)
    model = KGAT(KGATArgs(user_num=g.user_num, entity_num=g.entity_num, relation_num=g.relation_num))
    with torch.no_grad():
        model._multi_head_attention._layer_norm.weight.add_(0.1 * torch.randn(64))
        model._multi_head_attention._layer_norm.bias.add_(0.1 * torch.randn(64))
    out.update({"param::" + k: v.detach().numpy().copy() for k, v in model.state_dict().items() if not v.is_sparse})
    return out


def compact(out: dict, recipe: tuple[str, int, int], sample: dict[str, int], seed: int = 0) -> dict:
    """``out`` as make_golden.golden_model built it -> the compacted form.  ``sample`` maps an output key to the number of
    its leading-dimension rows to keep (drawn without replacement from ``numpy.random.default_rng(seed)``, sorted)."""
    shape, rseed, dup = recipe
    inputs = rebuild_inputs(shape, rseed, dup)
    res = {k: v for k, v in out.items() if k not in inputs}
    for k, v in inputs.items():
        if digest(out[k]) != digest(v):
            raise ValueError(f"{k}: the recipe does not rebuild the array the reference was run on")
        res["sha256::" + k] = np.array(digest(v))
    res.update({"recipe::shape": np.array(shape), "recipe::seed": np.array(rseed), "recipe::duplicate_pairs": np.array(dup)})
    rng = np.random.default_rng(seed)
    for k, n in sample.items():
        v = np.asarray(out[k])
        rows = np.sort(rng.choice(v.shape[0], size=n, replace=False)).astype(np.int64)
        res[k], res["rows::" + k], res["shape::" + k] = v[rows], rows, np.array(v.shape, np.int64)
    return res


def load(path) -> dict[str, np.ndarray]:
    """All arrays of a golden file, the regenerated inputs of a compacted one included (checked against their digests)."""
    with np.load(path, allow_pickle=False) as z:
        d = {k: z[k] for k in z.files}
    if "recipe::shape" not in d:
        return d
    inputs = rebuild_inputs(str(d.pop("recipe::shape")), int(d.pop("recipe::seed")), int(d.pop("recipe::duplicate_pairs")))
    for k, v in inputs.items():
        want = str(d.pop("sha256::" + k))
        if digest(v) != want:
            raise AssertionError(f"{path}: regenerated input {k} differs from the one the reference was run on")
    missing = [k for k in d if k.startswith("sha256::")]
    if missing:
        raise AssertionError(f"{path}: inputs not regenerated: {missing}")
    d.update(inputs)
    return d


def cut(d: dict, key: str, full):
    """``full`` -- the whole of output ``key`` as computed (numpy array or tensor) -- restricted to the rows the golden stores."""
    rows = d.get("rows::" + key)
    if rows is None:
        return full
    assert tuple(full.shape) == tuple(d["shape::" + key].tolist()), (key, tuple(full.shape), d["shape::" + key])
    if isinstance(full, torch.Tensor):
        return full[torch.from_numpy(rows).to(full.device)]
    return np.asarray(full)[rows]

"""Shared test plumbing.

* registers the ``gpu`` marker (tests that need a B200 are ``@pytest.mark.gpu``),
* puts the repo root on ``sys.path`` so ``kgat_b200`` (alias of the hyphen-named package
  directory) and ``oracle`` import,
* loads the golden vectors produced by ``oracle/make_golden.py`` from the unmodified reference
  (stored as ``oracle/golden_io.py`` describes).
"""

from __future__ import annotations

import sys
from collections import OrderedDict
from pathlib import Path

import numpy as np
import pytest
import torch

ROOT = Path(__file__).resolve().parents[1]
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

from oracle import golden_io  # noqa: E402

GOLDEN = ROOT / "tests" / "golden"


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


class Golden:
    """A golden ``.npz`` with helpers to rebuild reference-shaped objects."""

    def __init__(self, name: str):
        self.z = golden_io.load(GOLDEN / name)

    def __getitem__(self, k):
        return self.z[k]

    def __contains__(self, k):
        return k in self.z

    def keys(self):
        return list(self.z)

    def cut(self, k, full):
        """A computed output restricted to the rows the golden stores of ``k`` (all of them unless ``k`` is a row sample)."""
        return golden_io.cut(self.z, k, full)

    def params(self, prefix: str = "param::", device="cpu") -> "OrderedDict[str, torch.Tensor]":
        out = OrderedDict()
        for k in self.z:
            if k.startswith(prefix):
                out[k[len(prefix) :]] = torch.from_numpy(self.z[k].copy()).to(device)
        return out

    def att_coo(self, device="cpu") -> torch.Tensor:
        n = int(self.z["user_num"]) + int(self.z["entity_num"])
        idx = torch.from_numpy(np.vstack([self.z["att_rows"], self.z["att_cols"]])).long()
        return torch.sparse_coo_tensor(idx, torch.from_numpy(self.z["att_vals"].copy()), size=(n, n)).to(device)

    @property
    def node_num(self) -> int:
        return int(self.z["user_num"]) + int(self.z["entity_num"])

    def ragged(self, stem: str) -> dict[int, list[int]]:
        ptr, items = self.z[stem + "_ptr"], self.z[stem + "_items"]
        return {u: items[ptr[u] : ptr[u + 1]].tolist() for u in range(len(ptr) - 1)}

    def unpack_mask(self, key: str, width: int) -> np.ndarray:
        return np.unpackbits(self.z[key], axis=1)[:, :width].astype(bool)


@pytest.fixture(scope="session", params=["model_tiny.npz", "model_tiny_dup.npz", "model_small.npz"])
def golden_model(request):
    return Golden(request.param)


@pytest.fixture(scope="session")
def golden_small():
    return Golden("model_small.npz")


@pytest.fixture(scope="session")
def golden_tiny():
    return Golden("model_tiny.npz")


@pytest.fixture(scope="session")
def golden_pre():
    return Golden("preprocess_tiny.npz")


def elem_err(a, b, floor_frac: float = 1e-3) -> float:
    """Per-element relative error with an absolute floor: max |a - b| / (|b| + floor_frac * max|b|).  Unlike ``rel_err`` (normwise) a
    small entry that is wrong by a large factor shows; the floor keeps entries that are pure cancellation noise from dominating."""
    a = torch.as_tensor(a, dtype=torch.float64).flatten().cpu()
    b = torch.as_tensor(b, dtype=torch.float64).flatten().cpu()
    floor = floor_frac * max(float(b.abs().max()), 1e-30)
    return float(((a - b).abs() / (b.abs() + floor)).max())


def rel_err(a, b) -> float:
    a = torch.as_tensor(a, dtype=torch.float64).flatten().cpu()
    b = torch.as_tensor(b, dtype=torch.float64).flatten().cpu()
    denom = max(float(b.abs().max()), 1e-30)
    return float((a - b).abs().max()) / denom


# ---------------------------------------------------------------------------------------------
# KGAT_POISON=1: every CUDA buffer handed out by torch.empty / torch.empty_like is filled with NaN (0xFF for bytes)
# -- inside captured graphs on every replay -- so a kernel that reads memory nobody wrote (a row outside the
# needed-row frontier, a partial a CTA skipped, ...) poisons the result instead of silently reusing stale bytes.
# (compute-sanitizer's initcheck is closed on the GPU pool; this is the stand-in.)
# ---------------------------------------------------------------------------------------------
import os  # noqa: E402

if os.environ.get("KGAT_POISON") == "1":
    _empty, _empty_like = torch.empty, torch.empty_like

    def _poison(t):
        if t.is_cuda and t.numel():
            if t.dtype == torch.float32:
                t.fill_(float("nan"))
            elif t.dtype == torch.uint8:
                t.fill_(255)
        return t

    def _p_empty(*a, **k):
        return _poison(_empty(*a, **k))

    def _p_empty_like(*a, **k):
        return _poison(_empty_like(*a, **k))

    torch.empty, torch.empty_like = _p_empty, _p_empty_like

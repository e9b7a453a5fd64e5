"""Recipe for ``oracle/_ref``: the UNMODIFIED reference modules of the hot path, staged for the GPU box.

    python oracle/build_ref.py <checkout of the reference repository>

The reference is pure Python (no compile step), so "building" it means staging, byte for byte, the
handful of modules the KGAT hot path consists of -- ``src/model/KGAT/{model, aggregator,
multi_head_attention, preprocess}.py``, ``src/utils/metrics_calculator.py`` and the small modules
they import (``src/type.py``, ``src/constants.py``, ``src/utils/{kg_triplets_generator,
json_writer}.py``) plus the package ``__init__`` files -- from where they lie in a checkout of the
reference into ``oracle/_ref/`` (git-ignored).  Nothing is edited; ``MANIFEST.json`` records the sha256 of every staged file
so the bench line can say exactly which bytes were timed.

Users: ``bench.py --impl reference`` / the ``cpu_baseline`` and ``gpu_incumbent`` legs (the reference's
own ``KGAT`` driven through its own public API), falling back to the oracle port when ``_ref`` is
missing.  TEST / MEASUREMENT INFRASTRUCTURE -- the product package never imports it.
"""

from __future__ import annotations

import hashlib
import json
import shutil
import sys
from pathlib import Path

OUT = Path(__file__).resolve().parent / "_ref"

FILES = [
    "src/__init__.py",
    "src/constants.py",
    "src/type.py",
    "src/model/__init__.py",
    "src/model/KGAT/__init__.py",
    "src/model/KGAT/model.py",
    "src/model/KGAT/aggregator.py",
    "src/model/KGAT/multi_head_attention.py",
    "src/model/KGAT/preprocess.py",
    "src/utils/__init__.py",
    "src/utils/metrics_calculator.py",
    "src/utils/kg_triplets_generator.py",
    "src/utils/json_writer.py",
]


def build(ref: Path, quiet: bool = False) -> bool:
    manifest = {}
    for rel in FILES:
        src, dst = ref / rel, OUT / rel
        if not src.exists():
            if rel.endswith("__init__.py"):  # namespace-style package in the reference: an empty marker is equivalent
                dst.parent.mkdir(parents=True, exist_ok=True)
                dst.write_bytes(b"")
                manifest[rel] = "absent in the reference (empty package marker written)"
                continue
            raise FileNotFoundError(src)
        dst.parent.mkdir(parents=True, exist_ok=True)
        shutil.copyfile(src, dst)
        manifest[rel] = hashlib.sha256(dst.read_bytes()).hexdigest()
    (OUT / "MANIFEST.json").write_text(json.dumps({"source": str(ref), "files": manifest}, indent=1) + "\n")
    if not quiet:
        print(f"oracle/_ref: staged {len(manifest)} unmodified reference files")
    return True


def load():
    """Import the staged reference: returns (model module, metrics module) or None when ``_ref`` is absent."""
    if not (OUT / "src" / "model" / "KGAT" / "model.py").exists():
        return None
    sys.dont_write_bytecode = True
    stale = [k for k in sys.modules if k == "src" or k.startswith("src.")]
    for k in stale:  # another `src` package (the reference tree itself in the build container) must not shadow the staged one
        del sys.modules[k]
    sys.path.insert(0, str(OUT))
    try:
        import importlib

        model = importlib.import_module("src.model.KGAT.model")
        metrics = importlib.import_module("src.utils.metrics_calculator")
    finally:
        sys.path.remove(str(OUT))
    return model, metrics


if __name__ == "__main__":
    if len(sys.argv) != 2:
        raise SystemExit("usage: python oracle/build_ref.py <checkout of the reference repository>")
    build(Path(sys.argv[1]).resolve())

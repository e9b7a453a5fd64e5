"""The fused bi-interaction aggregator (csrc/biagg.cu, biagg_mma.cu, biagg_tc5.cu) against a float64 restatement, for each of
its three implementations.

    out = normalize(dropout(lrelu((E+S) W1^T + b1) + lrelu((E*S) W2^T + b2))),  eps = 1e-12

``KGAT_BIAGG_IMPL`` is read once per process, so every implementation runs in a child process of its own (this file, run as a
script) that writes its outputs to a temporary directory; the test process rebuilds the same seeded inputs and compares them with
the float64 reference on the GPU: ``out``, ``inv_norm`` (sign included), ``flags``, ``g_E``, ``g_S`` and the four parameter
gradients, per element (``conftest.elem_err``) and normwise.

* ffma: the CUDA-core forward and backward of biagg.cu;
* mma:  the 3xTF32 ``mma.sync`` forward and backward of biagg_mma.cu;
* tc5:  the tcgen05 forward of biagg_tc5.cu for the six shapes it takes (mma.sync for 128->128 and 128->64), mma.sync backward.
The row-list entry points run the mma.sync kernels under ffma too (and the tcgen05 forward under tc5).

Every shape at n = 1, 127, 128, 129 (one 128-row tile and its edges) and 2 * 128 * SMs + 77 (every persistent tcgen05 CTA runs at
least two tiles, so both TMEM accumulator sets and the mbarrier parity flip are used).  The Philox dropout layouts of the three
implementations differ by design: the reference of an in-kernel dropout run takes the mask the kernel reports in ``flags & 4``,
and the statistics check that mask's per-column keep rate and that no two columns of a row share a random draw.

Measured maxima on a B200 (1,000 W), per element (elem_err, floor 1e-3 max|ref|) / normwise, over every case but the Philox ones:
  ffma  out 1.6e-4 / 4.7e-7, gradients 1.9e-4 / 4.2e-7;
  mma   out 5.9e-4 / 1.9e-6, gradients 5.7e-4 / 1.7e-6 (the row-list kernels under every implementation: 3.5e-4 / 1.3e-6);
  tc5   out 5.9e-4 / 1.9e-6, gradients 5.7e-4 / 1.7e-6.
Philox dropout at p = 0.5 drops half of a row, and rows whose kept columns nearly cancel amplify the 3xTF32 truncation of the
tensor-core paths (worst at 64 -> 16):
  ffma  out 2.7e-4 / 1.7e-6, gradients 2.0e-4 / 1.5e-6;
  mma   out 3.8e-4 / 1.0e-5, gradients 2.7e-3 / 1.6e-5;
  tc5   out 4.6e-4 / 7.8e-6, gradients 1.3e-3 / 3.3e-5.
The bounds sit about 10x above these maxima.
"""

from __future__ import annotations

import os
import subprocess
import sys
import zlib
from pathlib import Path

import numpy as np
import pytest
import torch

ROOT = Path(__file__).resolve().parents[1]

pytestmark = pytest.mark.gpu

DIMS = [(64, 64), (64, 32), (32, 16), (16, 16), (32, 32), (64, 16), (128, 128), (128, 64)]
IMPLS = ["ffma", "mma", "tc5"]
NORM_EPS = 1e-12
DEV = "cuda"  # where the float64 reference runs
SLOPE = 0.01
PHILOX_P = [0.1, 0.5]
PHILOX_N = 20000
OFFSETS = [1 << 40, 2 << 40]  # layers 0 and 1 (functions.py: offset = (l + 1) << 40)
# per-element / normwise bounds of the forward output (and inv_norm) and of the gradients, per implementation
TOL = {
    "ffma": {"out": (2e-3, 5e-6), "grad": (2e-3, 5e-6)},
    "mma": {"out": (6e-3, 2e-5), "grad": (6e-3, 2e-5)},
    "tc5": {"out": (6e-3, 2e-5), "grad": (6e-3, 2e-5)},
}
# the same with in-kernel Philox dropout (p up to 0.5)
DROPOUT_TOL = {
    "ffma": {"out": (3e-3, 2e-5), "grad": (2e-3, 1.5e-5)},
    "mma": {"out": (4e-3, 1e-4), "grad": (3e-2, 2e-4)},
    "tc5": {"out": (5e-3, 8e-5), "grad": (1.5e-2, 3.5e-4)},
}


def sizes(sms: int) -> list[int]:
    return [1, 127, 128, 129, 2 * 128 * sms + 77]


def _gen(*key) -> torch.Generator:
    return torch.Generator().manual_seed(zlib.crc32(repr(key).encode()))


def make_inputs(din: int, dout: int, n: int, *key, zero_bias: bool = False) -> dict:
    """Seeded CPU inputs of one case (the child and the test process build the same ones)."""
    g = _gen(din, dout, n, *key)
    inp = {
        "E": torch.randn(n, din, generator=g),
        "S": 0.5 * torch.randn(n, din, generator=g),
        "W1": torch.randn(dout, din, generator=g) / din**0.5,
        "W2": torch.randn(dout, din, generator=g) / din**0.5,
        "b1": 0.1 * torch.randn(dout, generator=g),
        "b2": 0.1 * torch.randn(dout, generator=g),
        "g_out": torch.randn(n, dout, generator=g),
    }
    if zero_bias:
        inp["b1"].zero_()
        inp["b2"].zero_()
    return inp


def clamp_rows(n: int) -> tuple[np.ndarray, np.ndarray]:
    """Rows of the eps-clamp case: exactly zero, and scaled so that ||x|| < 1e-12 with every product a normal fp32."""
    return np.arange(0, n, 7), np.arange(3, n, 7)


def make_clamp_inputs(din: int, dout: int, n: int = 300) -> dict:
    inp = make_inputs(din, dout, n, "clamp", zero_bias=True)
    zero, tiny = clamp_rows(n)
    for k in ("E", "S"):
        inp[k][zero] = 0.0
        inp[k][tiny] *= 1e-13 / dout**0.5
    return inp


def rows_case(din: int, dout: int):
    """Row list of the row-list entry points: 3000 of 4000 nodes in shuffled order, capacity 3500."""
    n_nodes, n_list, max_rows = 4000, 3000, 3500
    g = _gen(din, dout, "rows")
    rows = torch.randperm(n_nodes, generator=g)[:n_list].to(torch.int32)
    return make_inputs(din, dout, n_nodes, "rows"), rows, max_rows


def keep_bits_case(din: int, dout: int, n: int = 1000, p: float = 0.1):
    inp = make_inputs(din, dout, n, "bits")
    keep = torch.rand(n, dout, generator=_gen(din, dout, "keep")) >= p
    return inp, keep


def pack_keep_bits(keep: torch.Tensor) -> torch.Tensor:
    """bool [N, d] -> int32 [N, ceil(d / 32)], bit j of word w = column 32 w + j."""
    n, d = keep.shape
    words = (d + 31) // 32
    padded = np.zeros((n, words * 32), dtype=bool)
    padded[:, :d] = keep.numpy()
    return torch.from_numpy(np.packbits(padded, axis=1, bitorder="little").view(np.int32).reshape(n, words).copy())


# ---------------------------------------------------------------------------------------------
# child process: run every case under one KGAT_BIAGG_IMPL and save the outputs
# ---------------------------------------------------------------------------------------------


def _launch(kb, inp, p=0.0, seed=0, offset=0, seed_dev=None, keep=None, rows=None, max_rows=None, pad=0, acc=None):
    """Forward, backward and parameter-gradient reduce of one case.  Buffers start as NaN / 0xAA so that a value nobody wrote
    shows; ``pad`` > 0 makes ``out`` and ``g_out`` column slices of wider buffers (ld = d_out + 2 pad) and calls the C ABI
    directly; ``acc`` is added onto by the reduce (accumulate=True)."""
    from kgat_b200 import ops

    lib = kb._lib.load()
    c = {k: v.cuda().contiguous() for k, v in inp.items()}
    n, din = c["E"].shape
    dout = c["W1"].shape[0]
    nan = float("nan")
    if pad:
        wide = torch.full((n, dout + 2 * pad), nan, device="cuda")
        out = wide[:, pad : pad + dout]
        gwide = torch.full((n, dout + 2 * pad), nan, device="cuda")
        gwide[:, pad : pad + dout] = c["g_out"]
        g_out = gwide[:, pad : pad + dout]
    else:
        out = torch.full((n, dout), nan, device="cuda")
        g_out = c["g_out"]
    inv = torch.full((n,), nan, device="cuda")
    flags = torch.full((n, dout), 0xAA, dtype=torch.uint8, device="cuda")
    bits = pack_keep_bits(keep).cuda() if keep is not None else None
    sd = torch.tensor([seed_dev], dtype=torch.int64, device="cuda") if seed_dev is not None else None
    args = (c["E"], c["S"], c["W1"], c["b1"], c["W2"], c["b2"])
    if pad:
        ops.check(lib.kgat_biagg_forward(*(t.data_ptr() for t in args[:2]), n, din, dout, *(t.data_ptr() for t in args[2:]), float(p),
                                         int(seed), int(offset), None, bits.data_ptr() if bits is not None else None, out.data_ptr(),
                                         out.stride(0), inv.data_ptr(), flags.data_ptr(), None, 0, ops._stream()), "biagg_forward (strided)")
    elif rows is not None:
        r = rows.cuda()
        n_dev = torch.tensor([rows.numel()], dtype=torch.int32, device="cuda")
        ops.biagg_forward(*args, out, inv, flags, dropout_p=p, seed=seed, offset=offset, keep_bits=bits, seed_dev=sd, rows=r,
                          n_rows_dev=n_dev, max_rows=max_rows)
    else:
        ops.biagg_forward(*args, out, inv, flags, dropout_p=p, seed=seed, offset=offset, keep_bits=bits, seed_dev=sd)
    n_ctas = ops.biagg_backward_ctas(max_rows if rows is not None else n, din, dout, rows=rows is not None)
    partials = torch.full((n_ctas * (2 * din * dout + 2 * dout),), nan, device="cuda")
    g_s, g_e = torch.full((n, din), nan, device="cuda"), torch.full((n, din), nan, device="cuda")
    if pad:
        ops.check(lib.kgat_biagg_backward(g_out.data_ptr(), g_out.stride(0), out.data_ptr(), out.stride(0), inv.data_ptr(), flags.data_ptr(),
                                          c["E"].data_ptr(), c["S"].data_ptr(), n, din, dout, c["W1"].data_ptr(), c["W2"].data_ptr(), float(p),
                                          g_s.data_ptr(), g_e.data_ptr(), partials.data_ptr(), n_ctas, None, 0, ops._stream()),
                  "biagg_backward (strided)")
    elif rows is not None:
        ops.biagg_backward(g_out, out, inv, flags, c["E"], c["S"], c["W1"], c["W2"], p, g_s, g_e, partials, n_ctas, rows=r, n_rows_dev=n_dev,
                           max_rows=max_rows)
    else:
        ops.biagg_backward(g_out, out, inv, flags, c["E"], c["S"], c["W1"], c["W2"], p, g_s, g_e, partials, n_ctas)
    if acc is not None:
        gw1, gb1, gw2, gb2 = (acc[k].cuda().clone() for k in ("gW1", "gb1", "gW2", "gb2"))
    else:
        gw1, gb1, gw2, gb2 = (torch.full_like(c[k], nan) for k in ("W1", "b1", "W2", "b2"))
    ops.biagg_reduce_param_grads(partials, n_ctas, din, dout, gw1, gb1, gw2, gb2, accumulate=acc is not None)
    res = {"out": out, "inv": inv, "flags": flags, "gE": g_e, "gS": g_s, "gW1": gw1, "gb1": gb1, "gW2": gw2, "gb2": gb2}
    if pad:
        res["out_wide"] = wide
    return {k: v.cpu() for k, v in res.items()}


def accumulate_init(din: int, dout: int) -> dict:
    g = _gen(din, dout, "acc")
    return {"gW1": torch.randn(dout, din, generator=g), "gb1": torch.randn(dout, generator=g), "gW2": torch.randn(dout, din, generator=g),
            "gb2": torch.randn(dout, generator=g)}


def _child(out_dir: Path, sms: int) -> None:
    sys.path.insert(0, str(ROOT))
    import kgat_b200 as kb

    kb._lib.load()
    res = {}
    for din, dout in DIMS:
        for n in sizes(sms):
            res[("dense", din, dout, n)] = _launch(kb, make_inputs(din, dout, n, "dense"))
        inp, rows, max_rows = rows_case(din, dout)
        res[("rows", din, dout)] = _launch(kb, inp, rows=rows, max_rows=max_rows)
        res[("clamp", din, dout)] = _launch(kb, make_clamp_inputs(din, dout))
        res[("strided", din, dout)] = _launch(kb, make_inputs(din, dout, 1000, "strided"), pad=4, acc=accumulate_init(din, dout))
        inp, keep = keep_bits_case(din, dout)
        res[("bits", din, dout)] = _launch(kb, inp, p=0.1, keep=keep)
        for p in PHILOX_P:
            res[("philox", din, dout, p)] = _launch(kb, make_inputs(din, dout, PHILOX_N, "philox", p), p=p, seed=1234, offset=OFFSETS[0])
    # one input, four dropout streams: two layers (offsets) and two steps (device-side seed offsets)
    inp = make_inputs(64, 64, PHILOX_N, "philox", 0.5)
    for off in OFFSETS:
        for step in (1, 2):
            r = _launch(kb, inp, p=0.5, seed=1234, offset=off, seed_dev=step)
            res[("stream", off, step)] = {"flags": r["flags"]}
    torch.cuda.synchronize()
    torch.save(res, out_dir / "results.pt")


def _child_devices() -> None:
    """The tcgen05 forward (193 KB of shared memory), the d = 128 attention pair kernel (128 KB) and the frontier expand
    (200 KB) on cuda:0 and then on cuda:1: each needs its dynamic shared-memory limit raised on the device it runs on."""
    sys.path.insert(0, str(ROOT))
    import kgat_b200 as kb
    from kgat_b200 import ops
    from kgat_b200.frontier import Frontier
    from kgat_b200.graph import AttentiveGraph

    kb._lib.load()
    inp = make_inputs(64, 64, 1000, "devices")
    g = torch.Generator().manual_seed(5)
    n_att, d_att = 300, 128
    emb, W = torch.randn(n_att, d_att, generator=g), torch.randn(3, d_att, d_att, generator=g) / d_att**0.5
    mha = {k: torch.randn(d_att, d_att, generator=g) / d_att**0.5 for k in ("Wv", "Wo")}
    mha.update({k: 0.1 * torch.randn(d_att, generator=g) for k in ("bv", "bo", "beta")})
    mha["gamma"] = 1 + 0.1 * torch.randn(d_att, generator=g)
    pair_tail = torch.arange(n_att, dtype=torch.int32)
    pair_rel = (torch.arange(n_att) % 3).to(torch.int32)
    n_nodes = 5000
    rng = np.random.default_rng(3)
    rows, cols = rng.integers(0, n_nodes, 20000), rng.integers(0, n_nodes, 20000)
    ids = torch.from_numpy(rng.integers(0, n_nodes, 64))
    outs = []
    for dev in (0, 1):
        with torch.cuda.device(dev):
            r = {}
            c = {k: v.cuda() for k, v in inp.items()}
            out = torch.empty(1000, 64, device="cuda")
            ops.biagg_forward(c["E"], c["S"], c["W1"], c["b1"], c["W2"], c["b2"], out, None, None)
            r["biagg"] = out
            _, r["att"] = ops.att_pair_scores(emb.cuda(), W.cuda(), pair_tail.cuda(), pair_rel.cuda(), {k: v.cuda() for k, v in mha.items()},
                                              n_heads=8, eps=1e-5)
            ag = AttentiveGraph.from_coo(torch.from_numpy(rows).cuda(), torch.from_numpy(cols).cuda(), torch.ones(rows.size, device="cuda"),
                                         n_nodes)
            f = Frontier(ag, 2, 64).build([ids.cuda()])
            r["frontier"] = f.rows(1)[: int(f.count(1).item())].clone()
            torch.cuda.synchronize()
            outs.append({k: v.cpu() for k, v in r.items()})
    # dev 0 against float64, dev 1 bit-identical to dev 0
    ref = reference(inp, device="cpu")
    assert float((outs[0]["biagg"].double() - ref["out"]).abs().max()) < 1e-5, "biagg forward on cuda:0"
    level = set(ids.tolist())
    level |= set(cols[np.isin(rows, ids.numpy())].tolist())
    assert sorted(outs[0]["frontier"].tolist()) == sorted(level), "frontier expand on cuda:0"
    for k in outs[0]:
        assert torch.equal(outs[0][k], outs[1][k]), f"{k}: cuda:1 differs from cuda:0"


# ---------------------------------------------------------------------------------------------
# float64 reference
# ---------------------------------------------------------------------------------------------




def reference(inp: dict, keep=None, p: float = 0.0, flags=None, device=None) -> dict:
    """float64 autograd of the aggregator.  ``keep``: dropout keep decisions (bool [n, d_out], scaled by 1 / (1 - p)) or None;
    ``flags``: the kernel's flags, whose sign bits stand in for the reference's where |z| is within rounding of 0 (either
    choice is right there, and the kernel's is the one its backward used)."""
    device = device or DEV
    leaves = {k: inp[k].to(device, torch.float64).requires_grad_(k != "g_out") for k in inp}
    E, S, W1, b1, W2, b2 = (leaves[k] for k in ("E", "S", "W1", "b1", "W2", "b2"))
    z1 = (E + S) @ W1.T + b1
    z2 = (E * S) @ W2.T + b2
    pos = []
    for z, bit in ((z1, 1), (z2, 2)):
        zd = z.detach()
        p_ = zd > 0
        if flags is not None:
            amb = zd.abs() <= 1e-6 * zd.abs().amax(dim=1, keepdim=True)
            p_ = torch.where(amb, (flags.to(device) & bit) != 0, p_)
        pos.append(p_)
    x = z1 * torch.where(pos[0], 1.0, SLOPE) + z2 * torch.where(pos[1], 1.0, SLOPE)
    kept = torch.ones_like(pos[0]) if keep is None else keep.to(device)
    if keep is not None:
        x = x * kept.double() / (1 - p)
    norm = x.detach().norm(dim=1)
    out = torch.nn.functional.normalize(x, p=2.0, dim=1, eps=NORM_EPS)
    out.backward(leaves["g_out"])
    flags_ref = pos[0].to(torch.uint8) | (pos[1].to(torch.uint8) << 1) | (kept.to(torch.uint8) << 2)
    inv = torch.where(norm < NORM_EPS, -1.0 / NORM_EPS, 1.0 / norm.clamp_min(NORM_EPS))
    return {"out": out.detach(), "inv": inv, "flags": flags_ref, "norm": norm, "gE": E.grad, "gS": S.grad, "gW1": W1.grad, "gb1": b1.grad,
            "gW2": W2.grad, "gb2": b2.grad}


def _errs(got, ref, floor_frac: float = 1e-3) -> tuple[float, float]:
    a, b = got.to(DEV, torch.float64), ref.to(DEV, torch.float64)
    amax = max(float(b.abs().max()), 1e-300)
    return float(((a - b).abs() / (b.abs() + floor_frac * amax)).max()), float((a - b).abs().max()) / amax


def check(name: str, got, ref, tol: tuple[float, float]) -> None:
    """Per element (``conftest.elem_err``: |a - b| / (|b| + 1e-3 max|b|)) and normwise (max|a - b| / max|b|)."""
    e, r = _errs(got, ref)
    assert e < tol[0] and r < tol[1], f"{name}: per-element {e:.3g} (bound {tol[0]:g}), normwise {r:.3g} (bound {tol[1]:g})"


def compare(impl: str, got: dict, inp: dict, keep=None, p: float = 0.0, rows=None, what: str = "", ref=None, tol=None) -> dict:
    """Every output of a run against the float64 reference (only the listed ``rows`` when given: the row-list kernels are the
    mma.sync ones under ffma too)."""
    if rows is not None:
        idx = rows.long()
        inp = {k: v[idx] if k in ("E", "S", "g_out") else v for k, v in inp.items()}
        got = {k: v[idx] if k in ("out", "inv", "flags", "gE", "gS") else v for k, v in got.items()}
        keep = None if keep is None else keep[idx]
    flags = got["flags"].to(DEV)
    if ref is None:
        ref = reference(inp, keep, p, flags)
    tol = tol or TOL["mma" if rows is not None and impl == "ffma" else impl]
    check(f"{what} out", got["out"], ref["out"], tol["out"])
    inv = got["inv"].to(DEV).double()
    assert torch.equal(inv < 0, ref["inv"] < 0), f"{what} inv_norm: sign differs on {int(((inv < 0) != (ref['inv'] < 0)).sum())} rows"
    check(f"{what} inv_norm", inv.abs(), ref["inv"].abs(), tol["out"])
    bad = int((flags != ref["flags"]).sum())
    assert bad == 0, f"{what} flags: {bad} entries differ"
    for k in ("gE", "gS", "gW1", "gb1", "gW2", "gb2"):
        check(f"{what} {k}", got[k], ref[k], tol["grad"])
    return ref


# ---------------------------------------------------------------------------------------------
# tests
# ---------------------------------------------------------------------------------------------


@pytest.fixture(scope="module")
def sms():
    if not torch.cuda.is_available():
        pytest.skip("needs CUDA")
    return torch.cuda.get_device_properties(0).multi_processor_count


def _run_child(args: list[str], env: dict, timeout: float) -> None:
    r = subprocess.run([sys.executable, str(Path(__file__).resolve()), *args], env=env, cwd=str(ROOT), capture_output=True, text=True,
                       timeout=timeout)
    assert r.returncode == 0, f"child {args[0]} failed ({r.returncode}):\n{r.stdout[-2000:]}\n{r.stderr[-4000:]}"


@pytest.fixture(scope="module", params=IMPLS)
def run(request, sms, tmp_path_factory):
    """(implementation, {case: outputs}) of one child process under KGAT_BIAGG_IMPL."""
    impl = request.param
    out_dir = tmp_path_factory.mktemp(f"biagg_{impl}")
    _run_child(["child", str(out_dir), str(sms)], dict(os.environ, KGAT_BIAGG_IMPL=impl), timeout=600)
    return impl, torch.load(out_dir / "results.pt")


@pytest.mark.parametrize("din,dout", DIMS)
def test_dense_forward_backward(run, sms, din, dout):
    """Dense entry points at n = 1, 127, 128, 129 and 2 * 128 * SMs + 77, no dropout."""
    impl, res = run
    for n in sizes(sms):
        compare(impl, res[("dense", din, dout, n)], make_inputs(din, dout, n, "dense"), what=f"{impl} {din}->{dout} n={n}")


@pytest.mark.parametrize("din,dout", DIMS)
def test_row_list_forward_backward(run, din, dout):
    """Row-list entry points over a shuffled list shorter than its capacity: listed rows match the reference, the other rows of
    every node-indexed output are left alone."""
    impl, res = run
    inp, rows, _ = rows_case(din, dout)
    got = res[("rows", din, dout)]
    compare(impl, got, inp, rows=rows, what=f"{impl} rows {din}->{dout}")
    other = torch.ones(inp["E"].shape[0], dtype=torch.bool)
    other[rows.long()] = False
    for k in ("out", "inv", "gE", "gS"):
        assert bool(got[k][other].isnan().all()), f"{k} written outside the row list"
    assert bool((got["flags"][other] == 0xAA).all()), "flags written outside the row list"


@pytest.mark.parametrize("din,dout", DIMS)
def test_eps_clamp_rows(run, din, dout):
    """Zero biases, rows that are exactly zero and rows with ||x|| < 1e-12: the forward divides by eps and stores -1/eps in
    inv_norm, the backward drops the projection term for those rows.  Clamped and ordinary rows are compared separately (the
    clamped rows' gradients are ~1e12 times larger)."""
    impl, res = run
    inp = make_clamp_inputs(din, dout)
    got = res[("clamp", din, dout)]
    zero, tiny = clamp_rows(inp["E"].shape[0])
    full = reference(inp, flags=got["flags"].to(DEV))
    norm = full["norm"].cpu()
    assert float(norm[zero].max()) == 0.0
    assert float(norm[tiny].max()) < 0.5 * NORM_EPS and float(norm[tiny].min()) > 1e-3 * NORM_EPS
    clamped = torch.from_numpy(np.concatenate([zero, tiny]))
    normal = torch.from_numpy(np.setdiff1d(np.arange(inp["E"].shape[0]), clamped.numpy()))
    assert bool((got["inv"][clamped] == -1.0 / np.float32(NORM_EPS)).all()), "inv_norm of the clamped rows is not -1/eps"
    assert float(got["out"][zero].abs().max()) == 0.0 and float(got["gE"][zero].abs().max()) > 0
    for sel, name in ((torch.from_numpy(tiny), "tiny"), (normal, "normal")):
        sub = {k: v[sel] if k in ("E", "S", "g_out") else v for k, v in inp.items()}
        g = {k: v[sel] if k in ("out", "inv", "flags", "gE", "gS") else v for k, v in got.items()}
        ref = reference(sub, flags=g["flags"].to(DEV))
        for k in ("out", "gE", "gS"):
            check(f"{impl} clamp {din}->{dout} {name} {k}", g[k], ref[k], TOL[impl]["grad" if k != "out" else "out"])
        assert torch.equal(g["inv"].to(DEV).double() < 0, ref["inv"] < 0)
    # the zero rows contribute nothing to the parameter gradients; all rows together match
    for k in ("gW1", "gb1", "gW2", "gb2"):
        check(f"{impl} clamp {din}->{dout} {k}", got[k], full[k], TOL[impl]["grad"])


@pytest.mark.parametrize("din,dout", DIMS)
def test_strided_out_and_accumulated_param_grads(run, din, dout):
    """``out`` and ``g_out`` as column slices of wider buffers (ld = d_out + 8); the columns around them stay untouched.  The
    parameter-gradient reduce adds onto nonzero gradients (accumulate=True)."""
    impl, res = run
    got = res[("strided", din, dout)]
    inp = make_inputs(din, dout, 1000, "strided")
    ref = reference(inp, flags=got["flags"].to(DEV))
    acc = accumulate_init(din, dout)
    for k in ("gW1", "gb1", "gW2", "gb2"):
        ref[k] = ref[k] + acc[k].to(DEV).double()
    compare(impl, got, inp, ref=ref, what=f"{impl} strided {din}->{dout}")
    wide = got["out_wide"]
    assert bool(wide[:, :4].isnan().all()) and bool(wide[:, 4 + dout :].isnan().all()), "columns outside the out slice were written"


@pytest.mark.parametrize("din,dout", DIMS)
def test_injected_keep_bits(run, din, dout):
    """Dropout p = 0.1 with caller-provided keep bits: flags & 4 reproduces them and the result is the masked reference."""
    impl, res = run
    inp, keep = keep_bits_case(din, dout)
    compare(impl, res[("bits", din, dout)], inp, keep=keep, p=0.1, what=f"{impl} keep_bits {din}->{dout}")


@pytest.mark.parametrize("p", PHILOX_P)
@pytest.mark.parametrize("din,dout", DIMS)
def test_philox_dropout(run, din, dout, p):
    """In-kernel Philox dropout: the output and gradients equal the reference under the mask the kernel reports in flags & 4;
    each column keeps within 6 sigma of (1 - p) * n, and every pair of columns of a row is kept together within 6 sigma of
    (1 - p)^2 (two columns that share one random draw would be kept together at rate 1 - p)."""
    impl, res = run
    got = res[("philox", din, dout, p)]
    inp = make_inputs(din, dout, PHILOX_N, "philox", p)
    keep = (got["flags"] & 4) != 0
    compare(impl, got, inp, keep=keep, p=p, what=f"{impl} philox p={p} {din}->{dout}", tol=DROPOUT_TOL[impl])
    k = keep.to(DEV, torch.float64)
    n, q = k.shape[0], 1 - p
    rate = k.mean(0)
    sigma = (q * (1 - q) / n) ** 0.5
    assert float((rate - q).abs().max()) < 6 * sigma, f"per-column keep rate {rate.min().item():.4f}..{rate.max().item():.4f}, expected {q}"
    joint = (k.T @ k) / n
    off = ~torch.eye(dout, dtype=torch.bool, device=None)
    q2 = q * q
    sigma2 = (q2 * (1 - q2) / n) ** 0.5
    worst = float((joint - q2)[off].abs().max())
    assert worst < 6 * sigma2, f"joint keep rate of a column pair off by {worst:.4f} (6 sigma = {6 * sigma2:.4f})"


def test_philox_streams_per_layer_and_step(run):
    """Two layer offsets x two device-side step seeds: the four masks of one input are pairwise independent (they agree on
    p^2 + (1-p)^2 of the entries within 6 sigma), not copies or shifts of each other."""
    impl, res = run
    masks = {key[1:]: (v["flags"] & 4) != 0 for key, v in res.items() if key[0] == "stream"}
    assert len(masks) == 4
    keys = sorted(masks)
    m = masks[keys[0]].numel()
    expect = 0.5  # p = 0.5
    sigma = (expect * (1 - expect) / m) ** 0.5
    for i in range(4):
        assert abs(float(masks[keys[i]].float().mean()) - 0.5) < 6 * (0.25 / m) ** 0.5
        for j in range(i + 1, 4):
            agree = float((masks[keys[i]] == masks[keys[j]]).float().mean())
            assert abs(agree - expect) < 6 * sigma, f"{impl}: masks {keys[i]} and {keys[j]} agree on {agree:.4f} of the entries"


def test_launch_attributes_are_per_device():
    """Kernels that need more than 48 KB of dynamic shared memory, run on cuda:0 and then on cuda:1 in one process, give the
    same results on both: the shared-memory limit is raised for each device a kernel runs on."""
    if not torch.cuda.is_available() or torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    _run_child(["devices"], dict(os.environ, KGAT_BIAGG_IMPL="tc5"), timeout=300)


if __name__ == "__main__":
    if sys.argv[1] == "child":
        _child(Path(sys.argv[2]), int(sys.argv[3]))
    elif sys.argv[1] == "devices":
        _child_devices()

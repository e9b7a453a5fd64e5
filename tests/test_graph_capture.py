"""CUDA graph captures run with Python's cyclic garbage collector paused (``functions.capture_graph``): captured steps and
optimiser plans sit in reference cycles, and a collection during a capture would destroy an unreachable graph inside it."""

from __future__ import annotations

import gc

import pytest
import torch


@pytest.mark.gpu
def test_capture_pauses_the_collector_and_restores_it():
    if not torch.cuda.is_available():
        pytest.skip("needs CUDA")
    from kgat_b200.functions import capture_graph

    x = torch.arange(8, dtype=torch.float32, device="cuda")
    y = torch.empty_like(x)
    for enabled in (True, False):
        (gc.enable if enabled else gc.disable)()
        try:
            g = torch.cuda.CUDAGraph()
            seen = []
            with capture_graph(g):
                seen.append(gc.isenabled())
                torch.mul(x, 2.0, out=y)
            assert seen == [False]
            assert gc.isenabled() is enabled
            x.add_(1.0)
            g.replay()
            torch.cuda.synchronize()
            assert torch.equal(y, 2.0 * x)
            with pytest.raises(RuntimeError), capture_graph(torch.cuda.CUDAGraph()):
                raise RuntimeError("body failed")
            assert gc.isenabled() is enabled
        finally:
            gc.enable()

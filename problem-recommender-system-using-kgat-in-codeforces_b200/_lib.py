"""ctypes binding of ``libkgat_b200.so`` (the C ABI declared in ``include/kgat_b200.h``).

There is deliberately no fallback: if the shared library is missing, or a kernel is asked to run
without a CUDA device, the caller gets an exception (``KgatLibraryError``), never a silent
PyTorch/CPU substitute.
"""

from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

KGAT_MAX_LAYERS = 8
KGAT_MAX_TENSORS = 24
ABI_VERSION = 9

_PKG_DIR = Path(__file__).resolve().parent
LIB_PATH = Path(os.environ.get("KGAT_B200_LIB", _PKG_DIR / "lib" / "libkgat_b200.so"))


class KgatLibraryError(RuntimeError):
    pass


class TablesT(C.Structure):
    _fields_ = [
        ("n_tables", C.c_int32),
        ("dims", C.c_int32 * KGAT_MAX_LAYERS),
        ("tables", C.c_void_p * KGAT_MAX_LAYERS),
        ("lds", C.c_int64 * KGAT_MAX_LAYERS),
    ]


class MhaT(C.Structure):
    _fields_ = [
        ("Wv", C.c_void_p),
        ("bv", C.c_void_p),
        ("Wo", C.c_void_p),
        ("bo", C.c_void_p),
        ("ln_gamma", C.c_void_p),
        ("ln_beta", C.c_void_p),
        ("ln_eps", C.c_float),
        ("n_heads", C.c_int32),
    ]


class AdamTensorsT(C.Structure):
    _fields_ = [
        ("n_tensors", C.c_int32),
        ("param", C.c_void_p * KGAT_MAX_TENSORS),
        ("grad", C.c_void_p * KGAT_MAX_TENSORS),
        ("exp_avg", C.c_void_p * KGAT_MAX_TENSORS),
        ("exp_avg_sq", C.c_void_p * KGAT_MAX_TENSORS),
        ("numel", C.c_int64 * KGAT_MAX_TENSORS),
        ("peer_param0", C.c_void_p),
        ("n_peers", C.c_int32),
        ("row_slot0", C.c_void_p),
        ("row_dim0", C.c_int32),
    ]


class PublishT(C.Structure):
    _fields_ = [("serial_dev", C.c_void_p), ("ring_host_mapped", C.c_void_p), ("n_slots", C.c_int32)]


_P = C.c_void_p
_I64 = C.c_int64
_I32 = C.c_int32
_F = C.c_float
_D = C.c_double
_U64 = C.c_uint64

# name -> (restype, argtypes); mirrors include/kgat_b200.h one to one
SIGNATURES: dict[str, tuple] = {
    "kgat_abi_version": (_I32, []),
    "kgat_error_string": (C.c_char_p, [_I32]),
    "kgat_last_cuda_error": (C.c_char_p, []),
    "kgat_device_info": (_I32, [C.POINTER(_I32), C.POINTER(_I32), C.POINTER(_I32), C.POINTER(_I64)]),
    "kgat_group_by_key_workspace_bytes": (_I64, [_I64]),
    "kgat_group_by_key": (_I32, [_P, _I64, _I32, _P, _I64, _P, _P, _P, _P, C.POINTER(_I64), _P]),
    "kgat_decode_sorted_keys": (_I32, [_P, _I64, _I64, _I64, _P, _P, _P]),
    "kgat_segment_sum_f32": (_I32, [_P, _P, _P, _I64, _P, _P]),
    "kgat_gather_f32": (_I32, [_P, _P, _I64, _P, _P]),
    "kgat_ids64_to_i32": (_I32, [_P, _I64, _I64, _P, _P, _P]),
    "kgat_spmm_csr": (_I32, [_P, _I64, _P, _I64, _P, _P, _P, _I64, _I64, _P, _I64, _P, _I64, _I32, _P, _P]),
    "kgat_spmm_csr_masked": (_I32, [_P, _I64, _P, _I64, _P, _P, _P, _I64, _I64, _P, _I64, _P, _I64, _I32, _P, _P, _P, _P]),
    "kgat_spmm_csr_rows": (_I32, [_P, _I64, _I64, _P, _P, _I64, _P, _P, _P, _I64, _I64, _P, _I64, _P, _I64, _I32, _P, _P, _P, _P, _P, _I64, _P]),
    "kgat_spmm_scatter_rows": (_I32, [_P, _I64, _P, _P, _P, _I64, _P, _P, _P, _P, _I64, _P, _I64, _P, _I64, _I32, _P]),
    "kgat_frontier_mark_ids": (_I32, [_P, _I64, _I64, _P, _P, _P]),
    "kgat_frontier_expand": (_I32, [_P, _I64, _P, _P, _P, _P, _I64, _P, _P, _I64, _P]),
    "kgat_frontier_scratch_ints": (_I64, [_I64]),
    "kgat_frontier_list": (_I32, [_P, _P, _I64, _P, _P, _P, _P]),
    "kgat_frontier_segment": (_I32, [_P, _P, _P, _I64, _I64, _I64, _P, _P, _P, _P]),
    "kgat_frontier_zero_rows": (_I32, [_P, _I64, _I32, _P, _P, _I64, _P]),
    "kgat_biagg_forward_rows": (_I32, [_P, _P, _P, _P, _I64, _I32, _I32, _P, _P, _P, _P, _F, _U64, _U64, _P, _P, _P, _I64, _P, _P, _P]),
    "kgat_biagg_backward_rows_ctas": (_I32, [_I64, _I32, _I32]),
    "kgat_biagg_backward_rows": (_I32, [_P, _I64, _P, _I64, _P, _P, _P, _P, _P, _P, _I64, _I32, _I32, _P, _P, _F, _P, _P, _P, _I32, _P]),
    "kgat_biagg_forward": (_I32, [_P, _P, _I64, _I32, _I32, _P, _P, _P, _P, _F, _U64, _U64, _P, _P, _P, _I64, _P, _P, _P, _I32, _P]),
    "kgat_biagg_backward_ctas": (_I32, [_I64, _I32, _I32]),
    "kgat_biagg_backward": (_I32, [_P, _I64, _P, _I64, _P, _P, _P, _P, _I64, _I32, _I32, _P, _P, _F, _P, _P, _P, _I32, _P, _I32, _P]),
    "kgat_biagg_reduce_param_grads": (_I32, [_P, _I32, _I32, _I32, _P, _P, _P, _P, _I32, _P]),
    "kgat_zero_rows_i64": (_I32, [_P, _I64, _I64, _I32, _P, _I64, _P]),
    "kgat_transr_rows_to_dense": (_I32, [_P, _P, _P, _P, _P, _I32, _I32, _P, _I64, _P, _P, _P, _P]),
    "kgat_transr_release_rows": (_I32, [_P, _I64, _I64, _I32, _P, _I64, _P, _P]),
    "kgat_bpr_forward": (_I32, [C.POINTER(TablesT), _P, _P, _P, _I32, _F, _P, _P, _P, C.POINTER(PublishT), _P]),
    "kgat_bpr_backward": (_I32, [C.POINTER(TablesT), C.POINTER(TablesT), _P, _P, _P, _I32, _F, _P, _P, _P]),
    "kgat_transr_forward": (_I32, [_P, _P, _P, _I32, _I32, _P, _P, _P, _P, _I32, _F, _P, _P, _P]),
    "kgat_transr_backward": (_I32, [_P, _P, _P, _I32, _I32, _P, _P, _P, _P, _I32, _F, _P, _P, _P, _P, _P, _P, _P]),
    "kgat_transr_claim_rows": (_I32, [_P, _P, _P, _I32, _I32, _P, _P, _P]),
    "kgat_transr_step": (_I32, [_P, _P, _P, _I32, _I32, _I32, _P, _P, _P, _P, _I32, _F, _P, _P, _P, _P, _P, _P, _P, C.POINTER(PublishT), _P]),
    "kgat_mha_forward": (_I32, [_P, _I64, _I32, C.POINTER(MhaT), _F, _P, _U64, _U64, _P, _P]),
    "kgat_att_pair_project": (_I32, [_P, _P, _I32, _P, _P, _I64, _P, _P]),
    "kgat_att_edge_scores_kgat": (_I32, [_P, _P, _P, _P, _P, _P, _I64, _I32, _P, _P]),
    "kgat_att_pair_scores": (_I32, [_P, _P, _I32, _P, _P, _I64, C.POINTER(MhaT), _P, _P, _P]),
    "kgat_att_edge_scores_dropout": (_I32, [_P, _P, _I64, _I32, C.POINTER(MhaT), _F, _P, _U64, _U64, _P, _P, _P]),
    "kgat_att_row_softmax": (_I32, [_P, _I64, _P, _P, _P, _P, _P, _P, _P]),
    "kgat_att_edge_weights": (_I32, [_P, _P, _P, _I64, _P, _P]),
    "kgat_gather_concat": (_I32, [C.POINTER(TablesT), _P, _I64, _P, _I64, _P]),
    "kgat_sgemm_nt": (_I32, [_P, _I64, _P, _I64, _P, _I64, _I32, _I32, _I32, _P]),
    "kgat_mask_scores": (_I32, [_P, _I64, _I32, _I32, _P, _P, _P]),
    "kgat_topk_rows": (_I32, [_P, _I64, _I32, _I32, _I32, _P, _P, _P]),
    "kgat_adam_advance": (_I32, [_P, _D, _D, _D, _D, _P, _P]),
    "kgat_adam_set_hyper": (_I32, [_I64, _D, _D, _D, _D, _P, _P]),
    "kgat_adam_apply": (_I32, [C.POINTER(AdamTensorsT), _P, _P]),
    "kgat_adam_hyper_table": (_I32, [_P, _I32, _D, _D, _D, _P, _P]),
    "kgat_adam_lazy_catchup": (_I32, [_P, _P, _P, _P, _P, _I32, _I32, _P, _P, _P, _P, _P]),
    "kgat_adam_sparse_rows": (_I32, [_P, _P, _P, _P, _P, _P, _I32, _I32, _P, _P, _P, _P]),
    "kgat_adam_lazy_flush": (_I32, [_P, _P, _P, _P, _I64, _I32, _P, _P, _P, _P, _P]),
    "kgat_adam_rolling_prepare": (_I32, [_P, _P, _P, _I32, _I32, _P, _P, _P, _I64, _P, _I64, _P, _P, _P, _P, _P, _I32, _P, _P, _P, _P, _P, _P, _P,
                                         _I64, _P]),
    "kgat_step_begin_i64": (_I32, [_P, _I64, _I64, _P, _P, _D, _D, _D, _D, _P, _P]),
    "kgat_transr_step_claimed": (_I32, [_P, _P, _P, _I32, _I32, _P, _P, _P, _P, _I32, _F, _P, _P, _P, _P, _P, _P, _P, C.POINTER(PublishT), _P]),
    "kgat_adam_rolling_apply": (_I32, [_P, _P, _P, _I32, _I32, _P, _P, _P, _P, _P, _P, _I64, _I32, C.POINTER(AdamTensorsT), _I32, _P, _P, _P, _P, _P]),
    "kgat_selftest_adam_arith": (_I32, [_P, _P, _I64, _F, _F, _P, _P]),
    "kgat_fill_f32": (_I32, [_P, _I64, _F, _P]),
    "kgat_select_batch_i64": (_I32, [_P, _I64, _I64, _P, _P, _P]),
    "kgat_sample_cf_batch": (_I32, [_P, _P, _P, _I32, _I32, _I32, _U64, _P, _P, _P]),
    "kgat_sample_kg_batch": (_I32, [_P, _P, _P, _P, _I32, _I32, _I32, _U64, _P, _P, _P]),
    "kgat_publish_loss": (_I32, [_P, _P, _P, _I32, _P]),
    "kgat_graph_launch": (_I32, [_P, _P]),
    "kgat_step_submit": (_I32, [_P, _P, _I64, _P, _P]),
    "kgat_peer_alloc": (_I32, [_I64, _P]),
    "kgat_peer_free": (_I32, [_P]),
    "kgat_peer_export": (_I32, [_P, _P]),
    "kgat_peer_import": (_I32, [_P, _P]),
    "kgat_peer_close": (_I32, [_P]),
    "kgat_peer_push": (_I32, [_P, _P, _I32, _I64, _I32, _P]),
    "kgat_peer_push_rows": (_I32, [_P, _P, _I32, _P, _P, _I64, _I32, _I64, _P]),
    "kgat_peer_copy": (_I32, [_P, _P, _I64, _P]),
    "kgat_peer_signal_wait": (_I32, [_P, _P, _I32, _P, _P, _I64, _P]),
}

_lib = None

# kernels launched per entry-point call (our own kernels only; feeds bench.py's "gpu_launches")
KERNELS_PER_CALL = {
    "kgat_group_by_key": 6, "kgat_decode_sorted_keys": 1, "kgat_segment_sum_f32": 1, "kgat_gather_f32": 1,
    "kgat_ids64_to_i32": 1, "kgat_spmm_csr": 1, "kgat_spmm_csr_masked": 1, "kgat_spmm_csr_rows": 1, "kgat_spmm_scatter_rows": 1, "kgat_frontier_mark_ids": 1, "kgat_frontier_expand": 1,
    "kgat_frontier_list": 2, "kgat_frontier_zero_rows": 1, "kgat_frontier_segment": 1, "kgat_biagg_forward_rows": 1, "kgat_biagg_backward_rows": 1, "kgat_biagg_forward": 1, "kgat_biagg_backward": 1,
    "kgat_biagg_reduce_param_grads": 1, "kgat_bpr_forward": 2, "kgat_bpr_backward": 1, "kgat_transr_forward": 2,
    "kgat_transr_backward": 1, "kgat_att_pair_scores": 1, "kgat_mha_forward": 1, "kgat_att_pair_project": 1, "kgat_att_edge_scores_kgat": 1, "kgat_att_edge_scores_dropout": 1, "kgat_att_row_softmax": 1,
    "kgat_att_edge_weights": 1, "kgat_gather_concat": 1, "kgat_sgemm_nt": 1, "kgat_mask_scores": 1, "kgat_topk_rows": 1,
    "kgat_adam_advance": 1, "kgat_adam_set_hyper": 1, "kgat_adam_apply": 1, "kgat_adam_hyper_table": 1, "kgat_adam_lazy_catchup": 1, "kgat_adam_sparse_rows": 1,
    "kgat_adam_lazy_flush": 1, "kgat_fill_f32": 1, "kgat_select_batch_i64": 1, "kgat_sample_cf_batch": 1, "kgat_sample_kg_batch": 1,
    "kgat_peer_push": 1, "kgat_peer_push_rows": 1, "kgat_publish_loss": 1, "kgat_zero_rows_i64": 1, "kgat_transr_rows_to_dense": 1, "kgat_transr_release_rows": 1, "kgat_peer_signal_wait": 1, "kgat_transr_claim_rows": 1, "kgat_transr_step": 4,
    "kgat_adam_rolling_prepare": 1, "kgat_transr_step_claimed": 3, "kgat_adam_rolling_apply": 1, "kgat_selftest_adam_arith": 1, "kgat_step_begin_i64": 1,
}


class LaunchCounter:
    """Counts kernel launches issued through the C ABI (reset / read by bench.py)."""

    count = 0


def _counted(fn, name: str):
    k = KERNELS_PER_CALL.get(name, 0)
    if k == 0:
        return fn
    def call(*args):
        LaunchCounter.count += k
        return fn(*args)

    return call


def load() -> C.CDLL:
    """Load the shared library once and attach the signatures.  Raises if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise KgatLibraryError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            f"(or `make -C {_PKG_DIR / 'csrc'}`).  There is no CPU / PyTorch fallback."
        )
    lib = C.CDLL(str(LIB_PATH))
    for name, (res, args) in SIGNATURES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError as e:  # pragma: no cover - build/header mismatch
            raise KgatLibraryError(f"{LIB_PATH} does not export {name}") from e
        fn.restype = res
        fn.argtypes = args
        setattr(lib, name, _counted(fn, name))
    if lib.kgat_abi_version() != ABI_VERSION:
        raise KgatLibraryError(f"ABI mismatch: library {lib.kgat_abi_version()} != binding {ABI_VERSION}")
    _lib = lib
    return lib


def check(rc: int, what: str = "") -> None:
    if rc == 0:
        return
    lib = load()
    msg = lib.kgat_error_string(rc).decode()
    if rc == -2:
        msg += ": " + lib.kgat_last_cuda_error().decode()
    raise KgatLibraryError(f"{what or 'kgat call'} failed ({rc}): {msg}")

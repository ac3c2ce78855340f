"""ctypes binding of libngcf_b200.so (the C ABI declared in include/ngcf_b200.h).

There is no CPU fallback and no pure-PyTorch path: if the shared library is missing or a call fails,
a RuntimeError is raised.
"""
from __future__ import annotations

import ctypes as C
import os

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("NGCF_B200_LIB") or os.path.join(_PKG, "libngcf_b200.so")   # env override: A/B builds

_vp, _i64, _i32, _f32, _u64, _sz = C.c_void_p, C.c_int64, C.c_int32, C.c_float, C.c_uint64, C.c_size_t



class NgcfCsr(C.Structure):
    """Mirror of ``ngcf_csr`` (include/ngcf_b200.h): a host struct of device pointers."""
    _fields_ = [("n_rows", _i64), ("rowptr", _vp), ("ent", _vp), ("tiles", _vp),
                ("hub_of_row", _vp), ("hub_chunk_ptr", _vp), ("chunk_ptr", _vp), ("hub_ent", _vp),
                ("chunk_row", _vp), ("chunk_tiles", _vp), ("hub_rows", _vp), ("hub_done", _vp), ("key_l", _vp), ("key_t", _vp), ("key_row_offset", _i64),
                ("n_tiles", _i32), ("n_hub", _i32), ("n_chunks", _i32),
                ("n_chunk_tiles", _i32), ("rowptr_nnz", _i32), ("tile_hubmask", _vp)]


_csr_p = C.POINTER(NgcfCsr)

# name -> argtypes (restype is int unless noted); mirrors include/ngcf_b200.h one to one
SIGNATURES = {
    "ngcf_abi_version": [],
    "ngcf_last_error": [],
    "ngcf_launch_count": [],
    "ngcf_coo_to_csr_workspace": [_i64, _i64, C.POINTER(_sz)],
    "ngcf_coo_to_csr": [_vp, _vp, _i64, _i64, _i64, C.c_int, _vp, _vp, _vp, _vp, _sz, _vp],
    "ngcf_edge_entries": [_vp, _vp, _vp, _vp, _vp, _i64, _vp],
    "ngcf_spmm_tile_rows": [],
    "ngcf_spmm_tile_entries": [],
    "ngcf_feature_mix": [_vp, _i64, C.c_int, C.POINTER(_vp), C.POINTER(C.c_int), C.POINTER(_vp), _vp, _i64, _f32,
                         _vp, _vp],
    "ngcf_spmm_split_threshold": [],
    "ngcf_spmm": [_csr_p, _vp, _i64, C.c_int, _vp, _i64, _vp, _vp, _i64, _vp, _f32, _u64, _vp, C.c_int, C.c_int, _i64,
                  _vp, _vp, _vp, _vp, _i64, _vp],
    "ngcf_entry_keys": [_csr_p, _i64, _vp, _vp, _vp],
    "ngcf_node_dropout_compact": [_csr_p, _f32, _u64, _vp, C.c_int, _i64, C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp),
                                  C.POINTER(_vp), _vp],
    "ngcf_node_dropout_bits": [_csr_p, _f32, _u64, _vp, C.c_int, _i64, _vp, _vp, _vp],
    "ngcf_pack_weights": [_vp, _vp, _vp, _vp, C.c_int, C.c_int, _vp, _vp, _vp],
    "ngcf_pack_weights_all": [C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp), C.POINTER(C.c_int),
                              C.POINTER(C.c_int), C.c_int, C.POINTER(_vp), C.POINTER(_vp), _vp],
    "ngcf_dense_fwd": [_vp, _vp, _i64, C.c_int, C.c_int, _vp, _vp, _f32, _vp, _vp, _f32, _u64, _vp, C.c_int, _i64, _vp,
                       _vp],
    "ngcf_mess_dropout_bits": [_i64, C.c_int, _f32, _u64, _vp, C.c_int, _i64, _vp, _vp],
    "ngcf_gather_concat": [C.POINTER(_vp), C.POINTER(C.c_int), C.c_int, _vp, _i64, _i64, _vp, _i64, _vp],
    "ngcf_gather_concat_sets": [C.POINTER(_vp), C.POINTER(C.c_int), C.c_int, C.POINTER(_vp), C.POINTER(_i64), C.POINTER(_i64),
                                C.POINTER(_vp), C.c_int, _i64, _vp],
    "ngcf_bpr_fwd_bwd": [_vp, _vp, _vp, _i64, C.c_int, _f32, _f32, _f32, _f32, _f32, _vp, _vp, _vp, _vp, _vp],
    "ngcf_rowgrad_scatter": [C.POINTER(_vp), C.POINTER(_i64), C.POINTER(_vp), C.POINTER(_i64), C.c_int, C.c_int, _vp,
                             _vp, _vp],
    "ngcf_rowgrad_reset": [C.POINTER(_vp), C.POINTER(_i64), C.POINTER(_i64), C.c_int, _vp, _vp],
    "ngcf_dense_bwd": [_vp, _vp, _vp, _i64, C.c_int, _vp, _vp, _vp, _i64, C.c_int, C.c_int, _vp, _vp, _f32, _vp, _vp, _f32,
                       _u64, _vp, C.c_int, _i64, C.c_int, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp],
    "ngcf_set_wgrad_stream": [_vp],
    "ngcf_wgrad_stream_forked": [],
    "ngcf_rowgrad_normalize": [C.POINTER(_vp), C.POINTER(_i64), C.POINTER(_i64), C.c_int, C.POINTER(_vp),
                               C.POINTER(C.c_int), C.c_int, _vp, _vp, C.c_int, _vp],
    "ngcf_adam_step": [C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_i64), C.c_int,
                       C.c_double, C.c_double, C.c_double, C.c_double, C.c_double, _i64, _vp, C.c_int, _vp],
    "ngcf_debug_bwd_timeline": [C.c_int, _vp],
    "ngcf_debug_spmm_timeline": [_vp],
    "ngcf_debug_compact_timeline": [_vp],
    "ngcf_score_topk_workspace": [_i64, _i64, C.c_int, C.c_int, C.POINTER(_sz)],
    "ngcf_eval_groups": [_vp, _vp, _vp, _vp, _vp, _i64, C.c_int, C.c_int, C.c_int, C.c_int, _f32, _f32, _vp, _vp, _vp, _vp, _vp,
                         _vp, _vp],
    "ngcf_sample_negatives": [_vp, _vp, _vp, _i64, _vp, C.c_int, C.c_int, _u64, _vp, _vp, _vp],
    "ngcf_laplacian_entries": [_vp, _vp, _vp, _i64, _i64, _i64, _vp, _vp, _vp, _vp, _vp],
    "ngcf_plgraph_entries": [_i64, _i64, _i64, C.c_double, _u64, _i64, _i64, _vp, _vp, _i64, _vp],
    "ngcf_build_tiles": [_vp, _i64, C.c_int, C.c_int, _vp, _vp, _i64, _vp, _vp],
    "ngcf_exchange_flag_words": [],
    "ngcf_push_rows": [C.POINTER(_vp), C.POINTER(_vp), _vp, C.c_int, C.c_int, _i64, _i64, C.c_int, _vp, _vp],
    "ngcf_push_selected_rows": [C.POINTER(_vp), C.POINTER(_vp), _vp, C.c_int, C.c_int, _i64, _i64, C.c_int, C.POINTER(_vp),
                                C.POINTER(_i64), C.POINTER(_i64), C.c_int, _vp, _vp],
    "ngcf_score_topk": [_vp, _i64, _vp, _i64, C.c_int, C.c_int, _vp, _vp, _vp, _sz, _vp],
    "ngcf_score_topk_excluding": [_vp, _i64, _vp, _i64, C.c_int, C.c_int, _vp, _vp, _vp, _vp, _vp, _sz, _vp],
    "ngcf_rank_metrics": [_vp, _i64, C.c_int, _vp, _vp, C.POINTER(C.c_int), C.c_int, _vp, _vp, _vp],
}

_lib = None


def load() -> C.CDLL:
    """Loads the in-tree shared library; raises (never falls back) if it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: the NGCF B200 hot path has no CPU/PyTorch fallback. "
            "Build it with `python -m seoul_tourism_recommendation_ngcf_b200.build` (needs nvcc, targets sm_100a).")
    lib = C.CDLL(LIB_PATH)
    for name, argtypes in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.argtypes = argtypes
        fn.restype = {"ngcf_last_error": C.c_char_p, "ngcf_launch_count": C.c_uint64}.get(name, C.c_int)
    _lib = lib
    return lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = load().ngcf_last_error()
        raise RuntimeError(f"ngcf_b200 {what} failed (status {rc}): {msg.decode() if msg else '?'}")


def ptr(t) -> int | None:
    """Device pointer of a tensor (None -> NULL)."""
    return None if t is None else t.data_ptr()


def ptr_array(tensors):
    return (_vp * len(tensors))(*[None if t is None else t.data_ptr() for t in tensors])


def ptr_array_int(addrs):
    """void*[] from raw integer addresses (peer-mapped pointers)."""
    return (_vp * len(addrs))(*[int(a) for a in addrs])


def int_array(vals):
    return (C.c_int * len(vals))(*[int(v) for v in vals])


def i64_array(vals):
    return (_i64 * len(vals))(*[int(v) for v in vals])


# bumped by every in-place parameter update this package performs behind torch's back (Adam through raw pointers, a
# CUDA-graph replay that contains it): NGCF compares it between forward and backward / all_*_emb (NGCF._check_fresh)
_param_epoch = 0


def bump_param_epoch() -> None:
    global _param_epoch
    _param_epoch += 1


def param_epoch() -> int:
    return _param_epoch


def on_device(fn):
    """Decorator for the kernel-launching entry points: runs ``fn`` with the CUDA device of its first CUDA tensor (or
    module) argument current.  Kernels launch on, and ``current_stream()`` reads, the CURRENT device — a module built on
    cuda:1 must not launch on cuda:0 just because that is torch's current device."""
    import functools

    import torch

    @functools.wraps(fn)
    def wrapped(*args, **kwargs):
        dev = None
        for a in list(args) + list(kwargs.values()):
            if isinstance(a, torch.Tensor):
                if a.device.type == "cuda":
                    dev = a.device
                    break
            elif isinstance(a, torch.nn.Module):
                q = next(a.parameters(), None)
                if q is not None and q.device.type == "cuda":
                    dev = q.device
                    break
        if dev is None or dev.index is None or dev.index == torch.cuda.current_device():
            return fn(*args, **kwargs)
        with torch.cuda.device(dev):
            return fn(*args, **kwargs)
    return wrapped


def current_stream() -> int:
    """Raw cudaStream_t of torch's current stream on the current device.  (torch.cuda.current_stream() resolves the
    device through several Python layers: ~24 calls per eager step were a quarter of its host time.)"""
    import torch
    try:
        return torch._C._cuda_getCurrentRawStream(torch._C._cuda_getDevice())
    except AttributeError:                                  # private API moved: the public, slower way
        return torch.cuda.current_stream().cuda_stream

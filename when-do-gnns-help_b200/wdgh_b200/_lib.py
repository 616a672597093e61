"""ctypes binding of libwdgh_b200.so -- the C ABI declared in include/wdgh_b200.h.

There is no CPU fallback: importing this module needs the built library, and
every compute call needs a CUDA device of compute capability 10.x.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libwdgh_b200.so")

NORM_NONE, NORM_RW, NORM_SYM = 0, 1, 2
NORM_RW_SUM, NORM_SYM_RAW = 3, 4   # scale modes of wdgh_degree_scale / wdgh_scale_values only (include/wdgh_b200.h)
DTYPE_F32, DTYPE_BF16, DTYPE_F16 = 0, 1, 2   # output element type of wdgh_spmm_csr_{bf16,f16} / wdgh_pipeline_host_*
PLAN_HEADER = 16
SC_MATCH_ALL, SC_MATCH_LAB, SC_N_LAB, SC_N_SELF, SC_N_EMPTY, SC_NBINS, SC_N_NODES_NSL, SC_N_MULTI_NEG = range(8)
SC_HEADER = 8


def sc_words(c: int) -> int:
    """Length of the counters array for c classes (WDGH_SC_WORDS)."""
    return SC_HEADER + 3 * c + c * c

if not os.path.exists(LIB_PATH):
    raise ImportError(
        f"{LIB_PATH} is missing: build it with `python when-do-gnns-help_b200/build.py` "
        "(nvcc, sm_100a).  wdgh_b200 has no CPU or PyTorch fallback.")

lib = C.CDLL(LIB_PATH)

_p, _i64, _i32, _int = C.c_void_p, C.c_int64, C.c_int32, C.c_int

# name -> argtypes; every function returns int unless listed in _RESTYPE
SIGNATURES = {
    "wdgh_version": [],
    "wdgh_last_error": [],
    "wdgh_device_info": [C.POINTER(_int), C.POINTER(_int), C.POINTER(_int)],
    "wdgh_launch_count": [],
    "wdgh_coo_to_csr": [_p, _i64, _i64, _p, _p, _p],
    "wdgh_csr_to_coo_rows": [_p, _i64, _i64, _p, _p],
    "wdgh_pack_labels": [_p, _i64, _p, _p, _p],
    "wdgh_argmax_rows": [_p, _i64, _i64, _i64, _p, _p],
    "wdgh_plan_build": [_p, _i64, _i64, _i64, _p, _i64, C.POINTER(_i64), _p],
    "wdgh_degree_scale": [_p, _p, _i64, _int, _int, _p, _p, _p, _p],
    "wdgh_scale_values": [_p, _p, _p, _i64, _int, _p, _p, _p],
    "wdgh_add_self_loops": [_p, _p, _p, _i64, _p, _p, _p, _p, _p],
    "wdgh_normalize_dense": [_p, _i64, _i64, _i64, _int, _p, _p, _i64, _p],
    "wdgh_spmm_csr": [_p, _p, _p, _i64, _p, _i64, _i64, _p, _i64, _int, _int, _p, _p, _p, C.POINTER(_i64), _p, _i64,
                      _p],
    "wdgh_spmm_csr_bf16": [_p, _p, _p, _i64, _p, _i64, _i64, _p, _i64, _int, _int, _int, _p, _p, _p, C.POINTER(_i64),
                           _p, _i64, _p],
    "wdgh_spmm_csr_f16": [_p, _p, _p, _i64, _p, _i64, _i64, _p, _i64, _int, _int, _int, _p, _p, _p, C.POINTER(_i64),
                          _p, _i64, _p],
    "wdgh_column_segments": [_p, _p, _i64, _p, _i32, _p, _p],
    "wdgh_plan_heavy_flags": [_p, C.POINTER(_i64), _i64, _p, _p],
    "wdgh_spmm_csr_ranged": [_p, _p, _p, _p, _p, _i64, _p, _i64, _i64, _p, _i64, _int, _int, _p, _p, _p, _int, _int,
                             _int, _p, _i32, _i32, _i64, _i64, _i32, _p, C.POINTER(_i64), _p, _i64, _p],
    "wdgh_spmm_csr_ranged_bf16": [_p, _p, _p, _p, _p, _i64, _p, _i64, _i64, _p, _i64, _int, _int, _p, _p, _p, _int,
                                  _int, _int, _p, C.POINTER(_i64), _p, _i64, _p],
    "wdgh_spmm_csr_ranged_f16": [_p, _p, _p, _p, _p, _i64, _p, _i64, _i64, _p, _i64, _int, _int, _p, _p, _p, _int,
                                 _int, _int, _p, C.POINTER(_i64), _p, _i64, _p],
    "wdgh_structure_counts": [_p, _p, _i64, _i64, _p, _i32, _p, C.POINTER(_i64), _p, _p, _p, _p, _p, _i64, _i64, _p],
    "wdgh_spmm_structure_fused": [_p, _p, _i64, _i64, _p, _i64, _i64, _p, _i64, _int, _int, _p, _p, _p, _i32, _p,
                                  C.POINTER(_i64), _p, _p, _p, _p, _p, _p, _i64, _i64, _p],
    "wdgh_structure_counts_coo": [_p, _i64, _i64, _p, _i32, _p, _p, _p, _p, _int, _p],
    "wdgh_edge_label_rows_equal": [_p, _p, _i64, _p, _i64, _i64, _p, _p],
    "wdgh_edge_cosine": [_p, _p, _p, _i64, _p, _i64, _i64, _int, _p, _i64, _p, _p, _p],
    "wdgh_gram_workspace_floats": [_i64, _i64],
    "wdgh_gram": [_p, _i64, _i64, _i64, _p, _i64, _int, _p, _p],
    "wdgh_gather_rows": [_p, _i64, _i64, _p, _i64, _p, _i64, _p],
    "wdgh_class_colsum": [_p, _i64, _i64, _p, _i32, _int, _p, _p],
    "wdgh_class_inner_workspace_doubles": [_i64, _i64, _i32],
    "wdgh_class_inner_sums": [_p, _i64, _i64, _i64, _p, _i32, _int, _p, _p, _p],
    "wdgh_las_score": [_p, _p, _p, _i64, _i32, _int, _int, _int, _p, _p, _p],
    "wdgh_ntk_clamp_transform": [_p, _i64, _i64, _p],
    "wdgh_gntk_transform": [_p, _i64, _i64, _int, _p, _p],
    "wdgh_pipeline_host": [_p, _p, _i64, _i64, _p, _i64, _p, _i32, _int, _int, _p, _p, _p],
    "wdgh_pipeline_host_bf16": [_p, _p, _i64, _i64, _p, _i64, _p, _i32, _int, _int, _p, _int, _p, _p],
    "wdgh_pipeline_host_f16": [_p, _p, _i64, _i64, _p, _i64, _p, _i32, _int, _int, _p, _int, _p, _p],
    "wdgh_pipeline_host_release": [],
}
_RESTYPE = {"wdgh_last_error": C.c_char_p, "wdgh_launch_count": C.c_uint64, "wdgh_gram_workspace_floats": C.c_int64,
            "wdgh_class_inner_workspace_doubles": C.c_int64}

for _name, _args in SIGNATURES.items():
    _fn = getattr(lib, _name)  # AttributeError here = header / library mismatch
    _fn.argtypes = _args
    _fn.restype = _RESTYPE.get(_name, _int)


class WdghError(RuntimeError):
    pass


def last_error() -> str:
    return (lib.wdgh_last_error() or b"").decode()


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        raise WdghError(f"{what or 'wdgh'} failed (rc={rc}): {last_error()}")


def launch_count() -> int:
    return int(lib.wdgh_launch_count())


_device_checked = False


def require_device() -> None:
    """Fail loudly unless a compute-capability-10.x CUDA device is current."""
    global _device_checked
    if _device_checked:
        return
    import torch

    if not torch.cuda.is_available():
        raise WdghError("wdgh_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    torch.cuda.init()
    sm, major, minor = _int(), _int(), _int()
    check(lib.wdgh_device_info(C.byref(sm), C.byref(major), C.byref(minor)), "wdgh_device_info")
    _device_checked = True


def ptr(t) -> int:
    """Device (or host) address of a torch tensor, None -> NULL."""
    return None if t is None else t.data_ptr()


def stream_ptr() -> int:
    import torch

    return torch.cuda.current_stream().cuda_stream

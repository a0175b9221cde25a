"""ctypes binding of include/mdim.h (the C ABI of libmdim_b200.so).

The library is built in-tree by `__graft_entry__.build()` / `make -C multidimension_b200/csrc`.
There is no fallback of any kind: if the shared library is missing, loading fails loudly; if
no sm_100 device is usable, `Context()` raises.
"""
from __future__ import annotations

import ctypes as C
import os

MAX_RANK = 8
MAX_NODES = 48
MAX_PEERS = 8
ABI_VERSION = 1

# status codes (mdim_status)
OK, ERR_OOB, ERR_SIZE, ERR_UNSUPPORTED, ERR_CUDA, ERR_ARITH, ERR_INVALID, ERR_NOMEM, ERR_NCCL = range(9)
COMM_ID_BYTES = 128
REDUCE_MIN, REDUCE_MAX = 100, 101

# dtypes (mdim_dtype)
U8, I32, U32, I64, U64, F32, F64, I8, I16, U16 = range(10)
DTYPE_SIZE = {U8: 1, I32: 4, U32: 4, I64: 8, U64: 8, F32: 4, F64: 8, I8: 1, I16: 2, U16: 2}
DTYPE_NAME = {U8: "u8", I32: "i32", U32: "u32", I64: "i64", U64: "u64", F32: "f32", F64: "f64", I8: "i8", I16: "i16", U16: "u16"}

# binary ops (mdim_binary_op) — reference src/ops.rs:23-129
ADD, SUB, MUL, DIV, REM, AND, OR, XOR, SHL, SHR = range(10)
# unary ops (mdim_unary_op)
NEG, NOT, ABS, SQRT, CAST = range(5)
# node kinds
LEAF, IOTA, CONST, UNARY, BINARY, DIAG, GATHER, FOLD, CONCAT, TUPLE = range(10)
MAX_OUTS = 4

COLLECT_ASYNC, COLLECT_NO_FASTPATH, COLLECT_NO_STATIC, COLLECT_NO_JIT = 1, 2, 4, 8
IPC_HANDLE_BYTES = 64


class Scalar(C.Union):
    _fields_ = [("u64", C.c_uint64), ("i64", C.c_int64), ("f64", C.c_double), ("f32", C.c_float),
                ("u32", C.c_uint32), ("i32", C.c_int32), ("u8", C.c_uint8), ("i8", C.c_int8), ("i16", C.c_int16), ("u16", C.c_uint16)]


class Node(C.Structure):
    _fields_ = [
        ("kind", C.c_int32), ("dtype", C.c_int32), ("op", C.c_int32), ("n_comp", C.c_int32),
        ("src_dtype", C.c_int32), ("n_peers", C.c_int32),
        ("data", C.c_void_p), ("offset", C.c_int64),
        ("stride", C.c_int64 * MAX_RANK), ("gstride", C.c_int64 * MAX_RANK), ("bound", C.c_uint64 * MAX_RANK),
        ("axis_a", C.c_int32 * MAX_RANK), ("axis_b", C.c_int32 * MAX_RANK), ("axis_c", C.c_uint64 * MAX_RANK),
        ("imm", Scalar), ("peer", C.c_void_p * MAX_PEERS), ("peer_block", C.c_uint64),
    ]


class Expr(C.Structure):
    _fields_ = [("abi_version", C.c_int32), ("rank", C.c_int32), ("red_rank", C.c_int32), ("n_nodes", C.c_int32),
                ("length", C.c_uint64 * MAX_RANK), ("nodes", C.POINTER(Node))]


class ErrorInfo(C.Structure):
    _fields_ = [("status", C.c_int32), ("node", C.c_int32), ("position", C.c_uint64), ("value", C.c_uint64),
                ("bound", C.c_uint64), ("component", C.c_int32), ("reserved", C.c_int32), ("message", C.c_char * 160)]


LIB_NAME = "libmdim_b200.so"
LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), LIB_NAME)

# every symbol include/mdim.h declares: (name, restype, argtypes)
_P = C.c_void_p
_PP = C.POINTER(C.c_void_p)
SYMBOLS = [
    ("mdim_init", C.c_int, [C.c_int, _PP]),
    ("mdim_shutdown", C.c_int, [_P]),
    ("mdim_set_stream", C.c_int, [_P, _P]),
    ("mdim_get_stream", C.c_int, [_P, _PP]),
    ("mdim_sync", C.c_int, [_P]),
    ("mdim_last_error", C.c_int, [_P, C.POINTER(ErrorInfo)]),
    ("mdim_status_string", C.c_char_p, [C.c_int]),
    ("mdim_launch_count", C.c_uint64, [_P]),
    ("mdim_last_kernel", C.c_int, [_P, C.c_char_p, C.c_size_t]),
    ("mdim_device_info", C.c_int, [_P, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_size_t)]),
    ("mdim_buf_alloc", C.c_int, [_P, C.c_size_t, _PP]),
    ("mdim_buf_free", C.c_int, [_P, _P]),
    ("mdim_upload", C.c_int, [_P, _P, _P, C.c_size_t]),
    ("mdim_download", C.c_int, [_P, _P, _P, C.c_size_t]),
    ("mdim_host_alloc", C.c_int, [_P, C.c_size_t, _PP]),
    ("mdim_host_free", C.c_int, [_P, _P]),
    ("mdim_collect", C.c_int, [_P, C.POINTER(Expr), _P, C.c_uint32]),
    ("mdim_collect_host", C.c_int, [_P, C.POINTER(Expr), _P, C.c_uint32]),
    ("mdim_collect_tuple", C.c_int, [_P, C.POINTER(Expr), _PP, C.c_int, C.c_uint32]),
    ("mdim_plan_describe", C.c_int, [_P, C.POINTER(Expr), C.c_uint32, C.c_char_p, C.c_size_t]),
    ("mdim_plan_describe_nodevice", C.c_int, [C.POINTER(Expr), C.c_uint32, C.c_char_p, C.c_size_t]),
    ("mdim_ipc_export", C.c_int, [_P, _P, C.POINTER(C.c_uint8)]),
    ("mdim_ipc_open", C.c_int, [_P, C.POINTER(C.c_uint8), _PP]),
    ("mdim_ipc_close", C.c_int, [_P, _P]),
    ("mdim_comm_unique_id", C.c_int, [C.POINTER(C.c_uint8)]),
    ("mdim_comm_init", C.c_int, [_P, C.c_int, C.c_int, C.POINTER(C.c_uint8)]),
    ("mdim_comm_destroy", C.c_int, [_P]),
    ("mdim_comm_info", C.c_int, [_P, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    ("mdim_allgather", C.c_int, [_P, _P, _P, C.c_size_t]),
    ("mdim_allreduce", C.c_int, [_P, _P, C.c_size_t, C.c_int, C.c_int]),
    ("mdim_barrier", C.c_int, [_P]),
    ("mdim_peer_table", C.c_int, [_P, _P, C.c_size_t, _PP]),
    ("mdim_peer_table_close", C.c_int, [_P]),
    ("mdim_fold_sharded_axis", C.c_int, [_P, _P, C.c_uint64, C.c_uint64, C.c_int, C.c_int, Scalar, _P]),
    ("mdim_fold_sharded_axis_status", C.c_int, [_P]),
    ("mdim_fold_sharded_axis_blocked", C.c_int, [_P, _P, C.c_uint64, C.c_uint64, C.c_int, C.c_int, Scalar, _P]),
    ("mdim_jit_check_nodevice", C.c_int, [C.POINTER(Expr), C.c_uint32, C.c_char_p, C.c_size_t]),
    ("mdim_abi_version", C.c_int, []),
]

_lib = None


def lib():
    """The loaded C-ABI library.  Raises (never falls back) when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                f"or `make -C multidimension_b200/csrc`.  There is no CPU fallback.")
        L = C.CDLL(LIB_PATH)
        for name, res, args in SYMBOLS:
            fn = getattr(L, name)  # AttributeError if the library lacks a declared symbol
            fn.restype = res
            fn.argtypes = args
        if L.mdim_abi_version() != ABI_VERSION:
            raise ImportError(f"{LIB_NAME}: ABI version {L.mdim_abi_version()} != {ABI_VERSION}")
        _lib = L
    return _lib


class MdimError(RuntimeError):
    """A non-OK mdim_status.  `info` carries mdim_error_info when a context produced it."""

    def __init__(self, status, message, info=None):
        super().__init__(message)
        self.status = status
        self.info = info


class Panic(MdimError):
    """A reference panic surfaced through the C ABI (bounds, sizes, integer division)."""

"""ctypes binding of libfuse_gpu.so — the C ABI declared in include/fuse_gpu.h.

This is plumbing for the tests and bench.py (the reference-facing host mirror is C++, see
csrc/host).  It never computes anything itself and has no fallback: if the library or a CUDA device
is missing, calls raise FuseGpuError.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import List, Optional, Sequence, Tuple

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "libfuse_gpu.so")

# fq_dtype tags (datavalues/data_value.rs:19-35 order)
NULL, BOOL, I8, I16, I32, I64, U8, U16, U32, U64, F32, F64, UTF8, STRUCT = range(14)
DTYPE_NAMES = ["Null", "Boolean", "Int8", "Int16", "Int32", "Int64", "UInt8", "UInt16", "UInt32", "UInt64",
               "Float32", "Float64", "Utf8", "Struct"]
DTYPE_SIZE = {BOOL: 1, I8: 1, I16: 2, I32: 4, I64: 8, U8: 1, U16: 2, U32: 4, U64: 8, F32: 4, F64: 8}

OK, ERR_INTERNAL, ERR_PLAN, ERR_DIVIDE_BY_ZERO, ERR_UNSUPPORTED, ERR_CUDA, ERR_INVALID, ERR_CAPACITY = range(8)
EXPR_ALIAS, EXPR_CONSTANT, EXPR_FIELD, EXPR_ARITHMETIC, EXPR_COMPARISON, EXPR_LOGIC, EXPR_AGGREGATOR, EXPR_LOOKUP = range(8)
MAX_LOOKUPS = 4
PIPE_PROJECT, PIPE_AGGREGATE, PIPE_GROUPBY = 0, 1, 2
RUN_ACCUMULATE, RUN_LIMIT_EARLY_EXIT, RUN_BLOCK_STATS = 1, 2, 4
STATE_HEADER_SLOTS = 6   # FQ_STATE_HEADER_SLOTS
MAX_COLS = MAX_EXPRS = 8
MAX_KEYS = 4

AGG = {"min": 0, "max": 1, "sum": 2, "count": 3}
CMP = {"=": 0, "<": 1, "<=": 2, ">": 3, ">=": 4}
ARITH = {"+": 0, "-": 1, "*": 2, "/": 3}
LOGIC = {"and": 0, "or": 1}
_TY = {"bool": BOOL, "i8": I8, "i16": I16, "i32": I32, "i64": I64, "u8": U8, "u16": U16, "u32": U32, "u64": U64,
       "f32": F32, "f64": F64}


class ScalarBits(C.Union):
    _fields_ = [("i", C.c_int64), ("u", C.c_uint64), ("f", C.c_double)]


class ExprNode(C.Structure):
    _fields_ = [("kind", C.c_int32), ("op", C.c_int32), ("left", C.c_int32), ("right", C.c_int32),
                ("column", C.c_int32), ("dtype", C.c_int32), ("value", ScalarBits)]


class CValue(C.Structure):
    _fields_ = [("dtype", C.c_int32), ("some", C.c_int32), ("v", ScalarBits)]


class Source(C.Structure):
    _fields_ = [("n_rows", C.c_uint64), ("n_cols", C.c_int32), ("generated", C.c_int32),
                ("cols", C.POINTER(C.c_void_p)), ("numbers_begin", C.c_uint64)]


class PipeDesc(C.Structure):
    _fields_ = [("n_cols", C.c_int32), ("col_dtypes", C.c_int32 * MAX_COLS), ("col_nullable", C.c_int32 * MAX_COLS), ("generated", C.c_int32),
                ("nodes", C.POINTER(ExprNode)), ("n_nodes", C.c_int32), ("predicate", C.c_int32), ("kind", C.c_int32),
                ("n_exprs", C.c_int32), ("exprs", C.c_int32 * MAX_EXPRS), ("n_keys", C.c_int32), ("keys", C.c_int32 * MAX_KEYS)]


class FuseGpuError(Exception):
    def __init__(self, status: int, message: str):
        super().__init__(message)
        self.status = status
        self.message = message


EXPORTS = [
    "fq_abi_version", "fq_ctx_create", "fq_ctx_destroy", "fq_last_error", "fq_ctx_launch_count", "fq_ctx_sm_count",
    "fq_column_alloc", "fq_column_wrap", "fq_column_slice", "fq_column_set_validity", "fq_column_validity", "fq_column_free",
    "fq_column_upload_bits", "fq_column_download_bits",
    "fq_group_create", "fq_group_handle", "fq_group_window", "fq_group_connect", "fq_group_connect_ptrs", "fq_group_destroy",
    "fq_pipe_set_group", "fq_pipe_fetch_merged", "fq_group_gather_project", "fq_group_gather_columns", "fq_group_fetch_gather", "fq_pipe_set_variant",
    "fq_column_dtype", "fq_column_len",
    "fq_column_device_ptr", "fq_column_upload", "fq_column_download", "fq_stream_synchronize", "fq_host_alloc",
    "fq_host_free", "fq_numbers_fill", "fq_pipe_compile", "fq_pipe_destroy", "fq_pipe_is_precompiled", "fq_pipe_build_kind", "fq_pipe_source",
    "fq_pipe_expr_dtype", "fq_pipe_expr_nullable", "fq_pipe_launch_aggregate", "fq_pipe_fetch_aggregate", "fq_pipe_fetch_block_stats", "fq_pipe_aggregator_nodes",
    "fq_pipe_state_device", "fq_pipe_launch_project", "fq_pipe_fetch_project", "fq_pipe_fetch_limit_row",
    "fq_pipe_key_dtype", "fq_pipe_leaf_dtype", "fq_pipe_groupby_reserve", "fq_pipe_launch_groupby", "fq_pipe_fetch_groupby",
    "fq_pipe_export_groups", "fq_pipe_group_entry_slots", "fq_pipe_export_partials", "fq_pipe_merge_partials",
    "fq_column_set_validity_bitmap", "fq_utf8_create", "fq_utf8_free", "fq_utf8_len", "fq_utf8_compare", "fq_utf8_compare_scalar", "fq_utf8_minmax",
    "fq_utf8_bytes", "fq_utf8_download", "fq_utf8_take", "fq_utf8_dict_encode", "fq_utf8_bounds", "fq_utf8_like", "fq_pipe_set_lookup",
    "fq_sort_indices", "fq_sort_indices_limit", "fq_column_take", "fq_column_copy", "fq_ctx_trim",
    "fq_graph_begin", "fq_graph_end", "fq_graph_launch", "fq_graph_destroy", "fq_stream_create", "fq_stream_destroy",
]

_lib = None


def lib():
    """Load libfuse_gpu.so (no build here: __graft_entry__.build() / fuse_query_b200.build does that)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise FuseGpuError(ERR_CUDA, f"{LIB_PATH} is missing: run `python -m fuse_query_b200.build` (there is no CPU fallback)")
    L = C.CDLL(LIB_PATH)
    vp, u64, i32, u32, i64 = C.c_void_p, C.c_uint64, C.c_int32, C.c_uint32, C.c_int64
    sig = {
        "fq_abi_version": (u32, []),
        "fq_ctx_create": (i32, [i32, C.POINTER(vp)]),
        "fq_ctx_destroy": (None, [vp]),
        "fq_last_error": (C.c_char_p, [vp]),
        "fq_ctx_launch_count": (u64, [vp]),
        "fq_ctx_sm_count": (i32, [vp]),
        "fq_column_alloc": (i32, [vp, i32, u64, C.POINTER(vp)]),
        "fq_column_wrap": (i32, [vp, i32, u64, vp, C.POINTER(vp)]),
        "fq_column_slice": (i32, [vp, vp, u64, u64, C.POINTER(vp)]),
        "fq_column_set_validity": (i32, [vp, vp, vp]),
        "fq_column_set_validity_bitmap": (i32, [vp, vp, vp, u64]),
        "fq_column_validity": (vp, [vp]),
        "fq_column_free": (None, [vp, vp]),
        "fq_group_create": (i32, [vp, i32, i32, u64, C.POINTER(vp)]),
        "fq_group_handle": (i32, [vp, vp, vp]),
        "fq_group_window": (i32, [vp, vp, C.POINTER(vp), C.POINTER(u64)]),
        "fq_group_connect": (i32, [vp, vp, vp]),
        "fq_group_connect_ptrs": (i32, [vp, vp, C.POINTER(vp)]),
        "fq_group_destroy": (None, [vp, vp]),
        "fq_pipe_set_group": (i32, [vp, vp, vp]),
        "fq_pipe_fetch_merged": (i32, [vp, vp, C.POINTER(CValue), i32, C.POINTER(i32), C.POINTER(u64)]),
        "fq_group_gather_project": (i32, [vp, vp, vp, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), i64, vp]),
        "fq_group_gather_columns": (i32, [vp, vp, C.POINTER(vp), C.POINTER(vp), i32, u64, u64, u64, C.POINTER(vp), C.POINTER(vp), i64, vp]),
        "fq_group_fetch_gather": (i32, [vp, vp, C.POINTER(u64), C.POINTER(u64)]),
        "fq_pipe_set_variant": (i32, [vp, vp, C.c_char_p]),
        "fq_column_upload_bits": (i32, [vp, vp, u64, vp, u64, u64, vp]),
        "fq_column_download_bits": (i32, [vp, vp, u64, vp, u64, vp]),
        "fq_column_dtype": (i32, [vp]),
        "fq_column_len": (u64, [vp]),
        "fq_column_device_ptr": (vp, [vp]),
        "fq_column_upload": (i32, [vp, vp, u64, vp, u64, vp]),
        "fq_column_download": (i32, [vp, vp, u64, vp, u64, vp]),
        "fq_stream_synchronize": (i32, [vp, vp]),
        "fq_host_alloc": (i32, [vp, u64, C.POINTER(vp)]),
        "fq_host_free": (None, [vp, vp]),
        "fq_numbers_fill": (i32, [vp, vp, u64, u64, u64, vp]),
        "fq_pipe_compile": (i32, [vp, C.POINTER(PipeDesc), C.POINTER(vp)]),
        "fq_pipe_destroy": (None, [vp, vp]),
        "fq_pipe_is_precompiled": (i32, [vp]),
        "fq_pipe_build_kind": (i32, [vp]),
        "fq_pipe_source": (C.c_char_p, [vp]),
        "fq_pipe_expr_dtype": (i32, [vp, vp, i32, C.POINTER(i32)]),
        "fq_pipe_expr_nullable": (i32, [vp, vp, i32, C.POINTER(i32)]),
        "fq_pipe_launch_aggregate": (i32, [vp, vp, C.POINTER(Source), u32, vp]),
        "fq_pipe_fetch_aggregate": (i32, [vp, vp, C.POINTER(CValue), i32, C.POINTER(i32), C.POINTER(u64)]),
        "fq_pipe_fetch_block_stats": (i32, [vp, vp, C.POINTER(u64), C.POINTER(u64)]),
        "fq_pipe_aggregator_nodes": (i32, [vp, vp, C.POINTER(i32), i32, C.POINTER(i32)]),
        "fq_pipe_state_device": (i32, [vp, vp, C.POINTER(vp), C.POINTER(u64)]),
        "fq_pipe_launch_project": (i32, [vp, vp, C.POINTER(Source), C.POINTER(vp), C.POINTER(vp), u64, i64, u32, vp]),
        "fq_pipe_fetch_project": (i32, [vp, vp, C.POINTER(u64), C.POINTER(u64)]),
        "fq_pipe_fetch_limit_row": (i32, [vp, vp, C.POINTER(u64)]),
        "fq_pipe_key_dtype": (i32, [vp, vp, i32, C.POINTER(i32), C.POINTER(i32)]),
        "fq_pipe_leaf_dtype": (i32, [vp, vp, i32, C.POINTER(i32), C.POINTER(i32)]),
        "fq_pipe_groupby_reserve": (i32, [vp, vp, u64]),
        "fq_pipe_launch_groupby": (i32, [vp, vp, C.POINTER(Source), u32, vp]),
        "fq_pipe_fetch_groupby": (i32, [vp, vp, C.POINTER(u64)]),
        "fq_pipe_export_groups": (i32, [vp, vp, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), u64, vp]),
        "fq_pipe_group_entry_slots": (i32, [vp, vp, C.POINTER(i32)]),
        "fq_pipe_export_partials": (i32, [vp, vp, i32, vp, C.POINTER(u64), vp]),
        "fq_pipe_merge_partials": (i32, [vp, vp, vp, u64, u32, vp]),
        "fq_utf8_create": (i32, [vp, vp, vp, u64, vp, vp, C.POINTER(vp)]),
        "fq_utf8_free": (None, [vp, vp]),
        "fq_utf8_len": (u64, [vp]),
        "fq_utf8_compare": (i32, [vp, i32, vp, vp, vp, vp, vp]),
        "fq_utf8_compare_scalar": (i32, [vp, i32, vp, vp, u64, vp, vp, vp]),
        "fq_utf8_minmax": (i32, [vp, i32, vp, C.POINTER(i64), vp]),
        "fq_utf8_bytes": (u64, [vp]),
        "fq_utf8_download": (i32, [vp, vp, vp, vp, vp]),
        "fq_utf8_take": (i32, [vp, vp, vp, u64, vp, C.POINTER(vp), vp]),
        "fq_utf8_dict_encode": (i32, [vp, vp, vp, C.POINTER(vp), vp]),
        "fq_utf8_bounds": (i32, [vp, vp, vp, u64, C.POINTER(u64), C.POINTER(u64), vp]),
        "fq_utf8_like": (i32, [vp, vp, vp, u64, i32, vp, vp]),
        "fq_pipe_set_lookup": (i32, [vp, vp, i32, vp, u64]),
        "fq_sort_indices": (i32, [vp, vp, vp, i32, u64, vp, vp]),
        "fq_sort_indices_limit": (i32, [vp, vp, vp, i32, u64, u64, vp, C.POINTER(u64), vp]),
        "fq_column_take": (i32, [vp, vp, vp, u64, vp, vp, vp]),
        "fq_column_copy": (i32, [vp, vp, u64, vp, u64, u64, vp]),
        "fq_ctx_trim": (i32, [vp]),
        "fq_stream_create": (i32, [vp, C.POINTER(vp)]),
        "fq_stream_destroy": (None, [vp, vp]),
        "fq_graph_begin": (i32, [vp, vp]),
        "fq_graph_end": (i32, [vp, vp, C.POINTER(vp)]),
        "fq_graph_launch": (i32, [vp, vp, vp]),
        "fq_graph_destroy": (None, [vp, vp]),
    }
    for name, (res, args) in sig.items():
        f = getattr(L, name)
        f.restype = res
        f.argtypes = args
    _lib = L
    return L


# ---------------------------------------------------------------------------------------------
# s-expression -> fq_expr_node[]  (the test-side s-expression syntax: (col x) (u64 1) (+ a b) (sum a) (alias n a) ...)
# ---------------------------------------------------------------------------------------------
def _tokens(text: str) -> List[str]:
    return text.replace("(", " ( ").replace(")", " ) ").split()


class ExprBuilder:
    """Accumulates the flat node array shared by a pipe's predicate and select expressions."""

    def __init__(self, columns: Sequence[str]):
        self.columns = list(columns)
        self.nodes: List[ExprNode] = []

    def _push(self, **kw) -> int:
        n = ExprNode(left=-1, right=-1)
        for k, v in kw.items():
            setattr(n, k, v)
        self.nodes.append(n)
        return len(self.nodes) - 1

    def add(self, sexpr: str) -> int:
        toks = _tokens(sexpr)
        root, rest = self._parse(toks, 0)
        if rest != len(toks):
            raise ValueError(f"trailing tokens in {sexpr!r}")
        return root

    def _parse(self, t: List[str], i: int) -> Tuple[int, int]:
        if t[i] != "(":
            raise ValueError(f"expected ( at {t[i:]}")
        head = t[i + 1]
        i += 2
        if head == "col":
            idx = self.columns.index(t[i])
            node = self._push(kind=EXPR_FIELD, column=idx)
            i += 1
        elif head in _TY:
            ty = _TY[head]
            lit = t[i]
            i += 1
            bits = ScalarBits()
            if ty == BOOL:
                bits.i = 1 if lit == "true" else 0
            elif ty in (F32, F64):
                bits.f = float(lit)
            elif ty in (U8, U16, U32, U64):
                bits.u = int(lit)
            else:
                bits.i = int(lit)
            node = self._push(kind=EXPR_CONSTANT, dtype=ty, value=bits)
        elif head == "alias":
            i += 1
            child, i = self._parse(t, i)
            node = self._push(kind=EXPR_ALIAS, left=child)
        elif head == "lookup":   # (lookup <slot> <index expression>)
            slot = int(t[i])
            child, i = self._parse(t, i + 1)
            node = self._push(kind=EXPR_LOOKUP, op=slot, left=child)
        elif head.lower() in AGG:
            child, i = self._parse(t, i)
            node = self._push(kind=EXPR_AGGREGATOR, op=AGG[head.lower()], left=child)
        else:
            for table, kind in ((ARITH, EXPR_ARITHMETIC), (CMP, EXPR_COMPARISON), (LOGIC, EXPR_LOGIC)):
                if head.lower() in table:
                    l, i = self._parse(t, i)
                    r, i = self._parse(t, i)
                    node = self._push(kind=kind, op=table[head.lower()], left=l, right=r)
                    break
            else:
                raise ValueError(f"unknown head {head!r}")
        if t[i] != ")":
            raise ValueError(f"expected ) at {t[i:]}")
        return node, i + 1

    def array(self):
        arr = (ExprNode * max(1, len(self.nodes)))(*self.nodes)
        return arr


# ---------------------------------------------------------------------------------------------
# thin object wrappers
# ---------------------------------------------------------------------------------------------
class Context:
    def __init__(self, device: int = 0):
        self._h = C.c_void_p()
        st = lib().fq_ctx_create(device, C.byref(self._h))
        if st:
            raise FuseGpuError(st, lib().fq_last_error(None).decode())
        self.device = device

    def check(self, st: int):
        if st:
            raise FuseGpuError(st, lib().fq_last_error(self._h).decode())

    def close(self):
        if self._h:
            lib().fq_ctx_destroy(self._h)
            self._h = C.c_void_p()

    @property
    def launch_count(self) -> int:
        return lib().fq_ctx_launch_count(self._h)

    @property
    def sm_count(self) -> int:
        return lib().fq_ctx_sm_count(self._h)

    # ---- columns ----
    def column(self, dtype: int, n: int) -> "Column":
        h = C.c_void_p()
        self.check(lib().fq_column_alloc(self._h, dtype, n, C.byref(h)))
        return Column(self, h)

    def wrap(self, dtype: int, n: int, device_ptr: int) -> "Column":
        h = C.c_void_p()
        self.check(lib().fq_column_wrap(self._h, dtype, n, C.c_void_p(device_ptr), C.byref(h)))
        return Column(self, h)

    def numbers(self, begin: int, n: int, stream: int = 0) -> "Column":
        """Materialised system.numbers_mt shard [begin, begin+n) (one fill kernel)."""
        col = self.column(U64, n)
        self.check(lib().fq_numbers_fill(self._h, col._h, 0, begin, n, C.c_void_p(stream)))
        return col

    def group(self, rank: int, world: int, row_bytes: int = 1 << 16) -> "Group":
        """This rank's end of the cross-GPU merge point (exchange window in this GPU's memory)."""
        h = C.c_void_p()
        self.check(lib().fq_group_create(self._h, rank, world, row_bytes, C.byref(h)))
        return Group(self, h, rank, world)

    def from_bitmap(self, bits, n: int, bit_offset: int = 0, stream: int = 0) -> "Column":
        """Boolean column (values or validity) from an Arrow LSB-first bitmap (bytes / numpy uint8), expanded on the device."""
        import numpy as np
        b = np.ascontiguousarray(np.frombuffer(bits, dtype=np.uint8) if not isinstance(bits, np.ndarray) else bits)
        col = self.column(BOOL, n)
        self.check(lib().fq_column_upload_bits(self._h, col._h, 0, C.c_void_p(b.ctypes.data), bit_offset, n, C.c_void_p(stream)))
        self.synchronize(stream)
        return col

    def fill_numbers(self, col: "Column", begin: int, n: int, stream: int = 0, row_offset: int = 0) -> None:
        """col[row_offset : row_offset + n] = begin .. begin + n - 1 (NumbersStream::poll_next on the device)."""
        self.check(lib().fq_numbers_fill(self._h, col._h, row_offset, begin, n, C.c_void_p(stream)))

    def from_numpy(self, a, valid=None, stream: int = 0, *, valid_bitmap=None, bit_offset: int = 0) -> "Column":
        """Upload values; `valid` (bool / 0-1 array, one entry per row) attaches a byte-per-row validity column,
        `valid_bitmap` (numpy uint8: an Arrow LSB-first bitmap, row 0 = bit `bit_offset`) attaches it bit-packed."""
        import numpy as np
        if valid_bitmap is not None:
            col = self.from_numpy(a, None, stream)
            bits = self.from_numpy(np.ascontiguousarray(np.asarray(valid_bitmap, dtype=np.uint8)), None, stream)
            self.check(lib().fq_column_set_validity_bitmap(self._h, col._h, bits._h, bit_offset))
            col._validity = bits
            return col
        if valid is not None:
            col = self.from_numpy(a, None, stream)
            v = np.ascontiguousarray(np.asarray(valid).astype(np.uint8))
            vcol = self.column(BOOL, len(v))
            if len(v):
                self.check(lib().fq_column_upload(self._h, vcol._h, 0, C.c_void_p(v.ctypes.data), len(v), C.c_void_p(stream)))
                self.synchronize(stream)
            self.check(lib().fq_column_set_validity(self._h, col._h, vcol._h))
            col._validity = vcol
            return col
        tag = {np.dtype(np.int8): I8, np.dtype(np.int16): I16, np.dtype(np.int32): I32, np.dtype(np.int64): I64,
               np.dtype(np.uint8): U8, np.dtype(np.uint16): U16, np.dtype(np.uint32): U32, np.dtype(np.uint64): U64,
               np.dtype(np.float32): F32, np.dtype(np.float64): F64}[a.dtype]
        a = np.ascontiguousarray(a)
        col = self.column(tag, len(a))
        if len(a):
            self.check(lib().fq_column_upload(self._h, col._h, 0, C.c_void_p(a.ctypes.data), len(a), C.c_void_p(stream)))
            self.synchronize(stream)
        return col

    def synchronize(self, stream: int = 0):
        self.check(lib().fq_stream_synchronize(self._h, C.c_void_p(stream)))

    # ---- ORDER BY ----
    def sort_indices(self, keys: Sequence["Column"], n: int, descending: Optional[Sequence[bool]] = None, stream: int = 0,
                     out: Optional["Column"] = None) -> "Column":
        """Row indexes (UInt32) that put `keys` in order: lexicographic, keys[0] most significant, NULLs first, stable."""
        out = out if out is not None else self.column(U32, max(1, n))
        arr = (C.c_void_p * len(keys))(*[k._h for k in keys])
        desc = (C.c_uint8 * len(keys))(*[1 if (descending and descending[j]) else 0 for j in range(len(keys))])
        self.check(lib().fq_sort_indices(self._h, arr, desc, len(keys), n, out._h, C.c_void_p(stream)))
        return out

    def sort_indices_limit(self, keys: Sequence["Column"], n: int, limit: int, descending: Optional[Sequence[bool]] = None,
                           stream: int = 0) -> Tuple["Column", int]:
        """ORDER BY ... LIMIT: the first min(limit, n) row indexes of the order sort_indices gives -> (column, count)."""
        out = self.column(U32, max(1, min(limit, n)))
        arr = (C.c_void_p * len(keys))(*[k._h for k in keys])
        desc = (C.c_uint8 * len(keys))(*[1 if (descending and descending[j]) else 0 for j in range(len(keys))])
        count = C.c_uint64()
        self.check(lib().fq_sort_indices_limit(self._h, arr, desc, len(keys), n, limit, out._h, C.byref(count), C.c_void_p(stream)))
        return out, count.value

    def take(self, src: "Column", rows: "Column", n: int, stream: int = 0) -> "Column":
        """out[i] = src[rows[i]]; the result carries byte validity when the source has validity of either form."""
        out = self.column(src.dtype, max(1, n))
        nullable = src.validity is not None or getattr(src, "_validity", None) is not None
        valid = self.column(BOOL, max(1, n)) if nullable else None
        self.check(lib().fq_column_take(self._h, src._h, rows._h, n, out._h, valid._h if valid is not None else None, C.c_void_p(stream)))
        if valid is not None:
            self.check(lib().fq_column_set_validity(self._h, out._h, valid._h))
            out._validity = valid
        return out

    def trim(self) -> None:
        """give cached scratch memory (ORDER BY) back to the device"""
        self.check(lib().fq_ctx_trim(self._h))

    def stream_create(self) -> int:
        """a non-blocking stream on this context's device (callers with CUDA bindings of their own pass their streams)"""
        s = C.c_void_p()
        self.check(lib().fq_stream_create(self._h, C.byref(s)))
        return s.value

    def stream_destroy(self, stream: int) -> None:
        lib().fq_stream_destroy(self._h, C.c_void_p(stream))

    # ---- recorded launches (CUDA graph) ----
    def graph_begin(self, stream: int) -> None:
        """Start recording: fq_pipe_launch_* calls on `stream` are recorded, not run, until graph_end."""
        self.check(lib().fq_graph_begin(self._h, C.c_void_p(stream)))

    def graph_end(self, stream: int) -> "Graph":
        g = C.c_void_p()
        self.check(lib().fq_graph_end(self._h, C.c_void_p(stream), C.byref(g)))
        return Graph(self, g)

    # ---- Utf8 arrays ----
    def utf8(self, values: Sequence[Optional[str]], stream: int = 0) -> "Utf8Array":
        """Arrow string array on the device from python strings (None = NULL)."""
        import numpy as np
        raw = [b"" if v is None else v.encode() for v in values]
        offsets = np.zeros(len(raw) + 1, dtype=np.int32)
        if raw:
            offsets[1:] = np.cumsum([len(b) for b in raw])
        data = b"".join(raw)
        valid = None
        if any(v is None for v in values):
            flags = np.array([0 if v is None else 1 for v in values], dtype=np.uint8)
            valid = self.column(BOOL, len(flags))
            self.check(lib().fq_column_upload(self._h, valid._h, 0, C.c_void_p(flags.ctypes.data), len(flags), C.c_void_p(stream)))
            self.synchronize(stream)
        h = C.c_void_p()
        buf = C.create_string_buffer(data, max(1, len(data)))
        self.check(lib().fq_utf8_create(self._h, C.c_void_p(offsets.ctypes.data), buf, len(raw), valid._h if valid is not None else None,
                                        C.c_void_p(stream), C.byref(h)))
        return Utf8Array(self, h, valid)

    # ---- pipes ----
    def pipe(self, exprs: Sequence[str], *, columns: Sequence[str] = ("number",), dtypes: Sequence[int] = (U64,),
             predicate: Optional[str] = None, aggregate: bool = False, generated: bool = False,
             nullable: Sequence[bool] = (), keys: Sequence[str] = ()) -> "Pipe":
        """`keys` (GROUP BY expressions) makes it a hash-aggregation pipe; `exprs` are then the aggregate expressions."""
        b = ExprBuilder(columns)
        pred = b.add(predicate) if predicate else -1
        roots = [b.add(e) for e in exprs]
        key_roots = [b.add(k) for k in keys]
        d = PipeDesc()
        d.n_cols = len(columns)
        for i, t in enumerate(dtypes):
            d.col_dtypes[i] = t
        for i, f in enumerate(nullable):
            d.col_nullable[i] = int(f) if int(f) in (0, 1, 2) else 1      # 1: byte validity, 2: Arrow bitmap validity
        d.generated = int(generated)
        nodes = b.array()
        d.nodes = C.cast(nodes, C.POINTER(ExprNode))
        d.n_nodes = len(b.nodes)
        d.predicate = pred
        d.kind = PIPE_GROUPBY if key_roots else (PIPE_AGGREGATE if aggregate else PIPE_PROJECT)
        d.n_exprs = len(roots)
        for i, r in enumerate(roots):
            d.exprs[i] = r
        d.n_keys = len(key_roots)
        for i, r in enumerate(key_roots):
            d.keys[i] = r
        h = C.c_void_p()
        self.check(lib().fq_pipe_compile(self._h, C.byref(d), C.byref(h)))
        p = Pipe(self, h, b, roots, aggregate or bool(key_roots), generated)
        p.n_keys = len(key_roots)
        return p


class Column:
    def __init__(self, ctx: Context, h):
        self.ctx, self._h = ctx, h

    def free(self):
        if self._h:
            lib().fq_column_free(self.ctx._h, self._h)
            self._h = None

    @property
    def dtype(self) -> int:
        return lib().fq_column_dtype(self._h)

    def __len__(self) -> int:
        return lib().fq_column_len(self._h)

    @property
    def device_ptr(self) -> int:
        return lib().fq_column_device_ptr(self._h) or 0

    def slice(self, offset: int, n: int) -> "Column":
        """A view of rows [offset, offset+n); the validity column, when there is one, is sliced alongside."""
        h = C.c_void_p()
        self.ctx.check(lib().fq_column_slice(self.ctx._h, self._h, offset, n, C.byref(h)))
        out = Column(self.ctx, h)
        out._parent = self
        return out

    @property
    def validity(self) -> Optional["Column"]:
        """The attached validity column (one BOOL byte per row, 1 = valid), or None for a NOT NULL column."""
        h = lib().fq_column_validity(self._h)
        return Column(self.ctx, h) if h else None

    def to_bitmap(self, n: Optional[int] = None, stream: int = 0):
        """Boolean column -> Arrow LSB-first bitmap (numpy uint8 of ceil(n / 8) bytes), packed on the device."""
        import numpy as np
        n = len(self) if n is None else n
        out = np.zeros((n + 7) // 8, dtype=np.uint8)
        if n:
            self.ctx.check(lib().fq_column_download_bits(self.ctx._h, self._h, 0, C.c_void_p(out.ctypes.data), n, C.c_void_p(stream)))
            self.ctx.synchronize(stream)
        return out

    def to_numpy(self, n: Optional[int] = None, stream: int = 0):
        import numpy as np
        npdt = {BOOL: np.uint8, I8: np.int8, I16: np.int16, I32: np.int32, I64: np.int64, U8: np.uint8, U16: np.uint16,
                U32: np.uint32, U64: np.uint64, F32: np.float32, F64: np.float64}[self.dtype]
        n = len(self) if n is None else n
        out = np.empty(n, dtype=npdt)
        if n:
            self.ctx.check(lib().fq_column_download(self.ctx._h, self._h, 0, C.c_void_p(out.ctypes.data), n, C.c_void_p(stream)))
            self.ctx.synchronize(stream)
        return out


class Graph:
    """fq_graph: the launches of one or more pipes, replayed with one graph launch; fetch from the pipes as usual."""

    def __init__(self, ctx: "Context", handle):
        self.ctx, self._h = ctx, handle

    def launch(self, stream: int) -> None:
        self.ctx.check(lib().fq_graph_launch(self.ctx._h, self._h, C.c_void_p(stream)))

    def destroy(self) -> None:
        if self._h:
            lib().fq_graph_destroy(self.ctx._h, self._h)
            self._h = None


class Utf8Array:
    """fq_utf8: Arrow string layout on the device (offsets + bytes, optional validity)."""

    def __init__(self, ctx: Context, h, valid: Optional[Column]):
        self.ctx, self._h, self._valid = ctx, h, valid

    def __len__(self) -> int:
        return lib().fq_utf8_len(self._h)

    def compare(self, op: str, other, stream: int = 0):
        """-> list of bool / None per row; `other` is another Utf8Array or a python string (array (op) scalar)"""
        n = len(self)
        out = self.ctx.column(BOOL, max(1, n))
        nullable = self._valid is not None or (isinstance(other, Utf8Array) and other._valid is not None)
        out_valid = self.ctx.column(BOOL, max(1, n)) if nullable else None
        ov = out_valid._h if out_valid is not None else None
        if isinstance(other, Utf8Array):
            self.ctx.check(lib().fq_utf8_compare(self.ctx._h, CMP[op], self._h, other._h, out._h, ov, C.c_void_p(stream)))
        else:
            b = other.encode()
            self.ctx.check(lib().fq_utf8_compare_scalar(self.ctx._h, CMP[op], self._h, C.create_string_buffer(b, max(1, len(b))), len(b), out._h, ov,
                                                         C.c_void_p(stream)))
        vals = [bool(x) for x in out.to_numpy(n, stream)]
        if out_valid is not None:
            ok = out_valid.to_numpy(n, stream)
            vals = [v if f else None for v, f in zip(vals, ok)]
        return vals

    def minmax(self, op: str, stream: int = 0) -> int:
        """row index of the min / max valid string (first occurrence), -1 when there is none"""
        row = C.c_int64()
        self.ctx.check(lib().fq_utf8_minmax(self.ctx._h, AGG[op], self._h, C.byref(row), C.c_void_p(stream)))
        return row.value

    def nbytes(self) -> int:
        return lib().fq_utf8_bytes(self._h)

    def to_list(self, stream: int = 0) -> List[Optional[bytes]]:
        """the strings as bytes (None where the array's validity says NULL)"""
        import numpy as np
        n = len(self)
        offsets = np.zeros(n + 1, dtype=np.int32)
        data = C.create_string_buffer(max(1, self.nbytes()))
        self.ctx.check(lib().fq_utf8_download(self.ctx._h, self._h, C.c_void_p(offsets.ctypes.data), data, C.c_void_p(stream)))
        self.ctx.synchronize(stream)
        raw = data.raw
        vals = [raw[offsets[i]:offsets[i + 1]] for i in range(n)]
        if self._valid is not None:
            ok = self._valid.to_numpy(n, stream)
            vals = [v if f else None for v, f in zip(vals, ok)]
        return vals

    def take(self, rows: Column, n: int, valid: Optional[Column] = None, stream: int = 0) -> "Utf8Array":
        """strings rows[0 .. n) (UInt32 column); `valid` (Boolean column) marks NULL output slots and must outlive the result"""
        h = C.c_void_p()
        self.ctx.check(lib().fq_utf8_take(self.ctx._h, self._h, rows._h, n, valid._h if valid is not None else None, C.byref(h), C.c_void_p(stream)))
        return Utf8Array(self.ctx, h, valid)

    def dict_encode(self, stream: int = 0):
        """-> (codes: UInt32 Column, one slot per row, dictionary: Utf8Array of the distinct valid strings in bytewise order)"""
        codes = self.ctx.column(U32, max(1, len(self)))
        h = C.c_void_p()
        self.ctx.check(lib().fq_utf8_dict_encode(self.ctx._h, self._h, codes._h, C.byref(h), C.c_void_p(stream)))
        return codes, Utf8Array(self.ctx, h, None)

    def bounds(self, value, stream: int = 0):
        """(lower, upper) bound of `value` (str or bytes) in this array, which must be sorted"""
        b = value.encode() if isinstance(value, str) else bytes(value)
        lo, hi = C.c_uint64(), C.c_uint64()
        self.ctx.check(lib().fq_utf8_bounds(self.ctx._h, self._h, C.create_string_buffer(b, max(1, len(b))), len(b), C.byref(lo), C.byref(hi),
                                            C.c_void_p(stream)))
        return lo.value, hi.value

    def like(self, pattern, negate: bool = False, stream: int = 0) -> Column:
        """fq_utf8_like: a UInt8 column of ceil(len / 8) bytes, bit i = string i LIKE `pattern` (str or bytes), negated by
        `negate`; NULL rows and the padding bits get 0.  An empty array gets one zero byte (a column is never empty)."""
        import numpy as np
        b = pattern.encode() if isinstance(pattern, str) else bytes(pattern)
        n = len(self)
        bits = self.ctx.column(U8, (n + 7) // 8) if n else self.ctx.from_numpy(np.zeros(1, dtype=np.uint8))
        self.ctx.check(lib().fq_utf8_like(self.ctx._h, self._h, C.create_string_buffer(b, max(1, len(b))), len(b), int(negate), bits._h,
                                          C.c_void_p(stream)))
        return bits

    def free(self):
        if self._h:
            lib().fq_utf8_free(self.ctx._h, self._h)
            self._h = None


class Group:
    """fq_group: the merge point across GPUs over peer memory (one process per GPU; see include/fuse_gpu.h)."""

    def __init__(self, ctx: Context, h, rank: int, world: int):
        self.ctx, self._h, self.rank, self.world = ctx, h, rank, world

    def handle(self) -> bytes:
        """64-byte CUDA IPC handle of this rank's window (to be sent to the peer processes)."""
        buf = C.create_string_buffer(64)
        self.ctx.check(lib().fq_group_handle(self.ctx._h, self._h, buf))
        return buf.raw

    @property
    def window(self) -> int:
        p, n = C.c_void_p(), C.c_uint64()
        self.ctx.check(lib().fq_group_window(self.ctx._h, self._h, C.byref(p), C.byref(n)))
        return p.value

    def connect(self, handles: Sequence[bytes]) -> None:
        """handles[r] = rank r's handle() (own entry ignored)."""
        blob = b"".join(bytes(h).ljust(64, b"\0")[:64] for h in handles)
        self.ctx.check(lib().fq_group_connect(self.ctx._h, self._h, C.c_char_p(blob)))

    def connect_ptrs(self, windows: Sequence[int]) -> None:
        """Ranks living in one process: the device addresses of every rank's window."""
        arr = (C.c_void_p * self.world)(*[C.c_void_p(w) for w in windows])
        self.ctx.check(lib().fq_group_connect_ptrs(self.ctx._h, self._h, arr))

    def gather_project(self, pipe: "Pipe", local_cols: Sequence[Column], final_cols: Sequence[Column], *, limit: int = -1,
                       local_valid: Optional[Sequence[Optional[Column]]] = None,
                       final_valid: Optional[Sequence[Optional[Column]]] = None, stream: int = 0) -> None:
        def arr(cols):
            if cols is None:
                return None
            return (C.c_void_p * max(1, len(cols)))(*[None if c is None else c._h for c in cols])
        self.ctx.check(lib().fq_group_gather_project(self.ctx._h, self._h, pipe._h, arr(local_cols), arr(local_valid), arr(final_cols),
                                                      arr(final_valid), limit, C.c_void_p(stream)))

    def fetch_gather(self) -> Tuple[int, int]:
        """-> (rows selected by all ranks, rows in the final columns)"""
        sel, fin = C.c_uint64(), C.c_uint64()
        self.ctx.check(lib().fq_group_fetch_gather(self.ctx._h, self._h, C.byref(sel), C.byref(fin)))
        return sel.value, fin.value

    def destroy(self):
        if self._h:
            lib().fq_group_destroy(self.ctx._h, self._h)
            self._h = None


def make_source(cols: Sequence[Column], n_rows: int, *, generated: bool = False, begin: int = 0):
    arr = (C.c_void_p * max(1, len(cols)))(*[c._h for c in cols])
    s = Source()
    s.n_rows = n_rows
    s.n_cols = len(cols)
    s.generated = int(generated)
    s.cols = C.cast(arr, C.POINTER(C.c_void_p))
    s.numbers_begin = begin
    s._keep = arr
    return s


class Pipe:
    def __init__(self, ctx: Context, h, builder: ExprBuilder, roots: List[int], aggregate: bool, generated: bool):
        self.ctx, self._h, self.builder, self.roots = ctx, h, builder, roots
        self.aggregate, self.generated = aggregate, generated

    def destroy(self):
        if self._h:
            lib().fq_pipe_destroy(self.ctx._h, self._h)
            self._h = None

    @property
    def precompiled(self) -> bool:
        return bool(lib().fq_pipe_is_precompiled(self._h))

    @property
    def build_kind(self) -> int:
        """0 = precompiled table, 1 = NVRTC in this process, 2 = on-disk JIT cache."""
        return lib().fq_pipe_build_kind(self._h)

    @property
    def source(self) -> str:
        return lib().fq_pipe_source(self._h).decode()

    def set_group(self, group: Optional["Group"]) -> None:
        """Aggregate launches end with the in-kernel merge across the group's ranks (fetch_merged reads it)."""
        self.ctx.check(lib().fq_pipe_set_group(self.ctx._h, self._h, group._h if group is not None else None))

    def set_lookup(self, slot: int, bits: Column, n_bits: int) -> None:
        """Binds bit table `slot` of the pipe's (lookup <slot> ...) nodes: a UInt8 column, LSB-first, read by later launches
        (keep it alive as long as they run)."""
        self.ctx.check(lib().fq_pipe_set_lookup(self.ctx._h, self._h, slot, bits._h, n_bits))

    def set_variant(self, variant: str) -> None:
        """Kernel variant for the next launches: "tma" | "u4" (aggregate), "tma" | "sparse" | "dense" | "ldg" (filter +
        projection), "tma" | "ldg" (projection); GROUP BY pipes have none."""
        self.ctx.check(lib().fq_pipe_set_variant(self.ctx._h, self._h, variant.encode()))

    def expr_nullable(self, i: int) -> bool:
        out = C.c_int32()
        self.ctx.check(lib().fq_pipe_expr_nullable(self.ctx._h, self._h, i, C.byref(out)))
        return bool(out.value)

    def expr_dtype(self, i: int) -> int:
        out = C.c_int32()
        self.ctx.check(lib().fq_pipe_expr_dtype(self.ctx._h, self._h, i, C.byref(out)))
        return out.value

    def aggregator_nodes(self) -> List[int]:
        n = C.c_int32()
        buf = (C.c_int32 * 64)()
        self.ctx.check(lib().fq_pipe_aggregator_nodes(self.ctx._h, self._h, buf, 64, C.byref(n)))
        return [buf[i] for i in range(n.value)]

    def state_device(self) -> Tuple[int, int]:
        p, n = C.c_void_p(), C.c_uint64()
        self.ctx.check(lib().fq_pipe_state_device(self.ctx._h, self._h, C.byref(p), C.byref(n)))
        return p.value, n.value

    # ---- aggregate ----
    def launch_aggregate(self, source: Source, *, accumulate: bool = False, block_stats: bool = False, stream: int = 0):
        flags = (RUN_ACCUMULATE if accumulate else 0) | (RUN_BLOCK_STATS if block_stats else 0)
        self.ctx.check(lib().fq_pipe_launch_aggregate(self.ctx._h, self._h, C.byref(source), flags, C.c_void_p(stream)))

    def fetch_block_stats(self) -> Tuple[int, int]:
        """(reference 10 000-row blocks scanned, blocks in which the predicate kept no row)"""
        b, e = C.c_uint64(), C.c_uint64()
        self.ctx.check(lib().fq_pipe_fetch_block_stats(self.ctx._h, self._h, C.byref(b), C.byref(e)))
        return b.value, e.value

    def fetch_merged(self):
        """fetch_aggregate for the state merged over every rank of the pipe's group by the last launch."""
        return self.fetch_aggregate(merged=True)

    def fetch_aggregate(self, merged: bool = False):
        """-> (list of (dtype, value|None) per Aggregator leaf, or None for DataValue::Null; rows_selected)"""
        vals = (CValue * 64)()
        n, rows = C.c_int32(), C.c_uint64()
        fetch = lib().fq_pipe_fetch_merged if merged else lib().fq_pipe_fetch_aggregate
        self.ctx.check(fetch(self.ctx._h, self._h, vals, 64, C.byref(n), C.byref(rows)))
        out = []
        for i in range(n.value):
            v = vals[i]
            if v.dtype == NULL:
                out.append(None)
            elif not v.some:
                out.append((v.dtype, None))
            elif v.dtype in (F32, F64):
                out.append((v.dtype, v.v.f))
            elif v.dtype in (U8, U16, U32, U64):
                out.append((v.dtype, v.v.u))
            else:
                out.append((v.dtype, v.v.i))
        return out, rows.value

    # ---- group by ----
    def key_dtype(self, j: int) -> Tuple[int, bool]:
        t, nl = C.c_int32(), C.c_int32()
        self.ctx.check(lib().fq_pipe_key_dtype(self.ctx._h, self._h, j, C.byref(t), C.byref(nl)))
        return t.value, bool(nl.value)

    def leaf_dtype(self, k: int) -> Tuple[int, bool]:
        t, nl = C.c_int32(), C.c_int32()
        self.ctx.check(lib().fq_pipe_leaf_dtype(self.ctx._h, self._h, k, C.byref(t), C.byref(nl)))
        return t.value, bool(nl.value)

    def groupby_reserve(self, groups: int) -> None:
        self.ctx.check(lib().fq_pipe_groupby_reserve(self.ctx._h, self._h, groups))

    def launch_groupby(self, source: Source, *, accumulate: bool = False, stream: int = 0) -> None:
        self.ctx.check(lib().fq_pipe_launch_groupby(self.ctx._h, self._h, C.byref(source), RUN_ACCUMULATE if accumulate else 0, C.c_void_p(stream)))

    def fetch_groupby(self) -> int:
        n = C.c_uint64()
        self.ctx.check(lib().fq_pipe_fetch_groupby(self.ctx._h, self._h, C.byref(n)))
        return n.value

    def run_groupby(self, source: Source, *, groups_hint: int = 1 << 16, stream: int = 0) -> int:
        """reserve -> launch -> fetch, growing the table until the groups fit; returns the number of groups.

        Every reservation after the first rehashes the keys with a new seed.  A scan has at most as many groups as rows,
        so the table grows to room for every row and no further: two overflows at that size raise."""
        hint, rows, full_overflows = groups_hint, source.n_rows, 0
        while True:
            self.groupby_reserve(hint)
            self.launch_groupby(source, stream=stream)
            try:
                return self.fetch_groupby()
            except FuseGpuError as e:
                if e.status != ERR_CAPACITY:
                    raise
                if hint >= rows:
                    full_overflows += 1
                    if full_overflows == 2:
                        raise FuseGpuError(ERR_CAPACITY, f"GROUP BY: two hash tables with room for all {rows} rows scanned overflowed") from e
                hint = max(1, min(hint * 8, rows))

    def export_groups(self, n_groups: int, stream: int = 0):
        """-> (key columns, key validity columns or None, leaf columns, leaf validity columns or None), device-resident"""
        ctx = self.ctx
        n_leaves = len(self.aggregator_nodes())
        keys, kval, leaves, lval = [], [], [], []
        for j in range(self.n_keys):
            t, nl = self.key_dtype(j)
            keys.append(ctx.column(t, max(1, n_groups)))
            kval.append(ctx.column(BOOL, max(1, n_groups)) if nl else None)
        for k in range(n_leaves):
            t, nl = self.leaf_dtype(k)
            leaves.append(ctx.column(t, max(1, n_groups)))
            lval.append(ctx.column(BOOL, max(1, n_groups)) if nl else None)

        def arr(cols):
            return (C.c_void_p * max(1, len(cols)))(*[None if c is None else c._h for c in cols])
        ctx.check(lib().fq_pipe_export_groups(ctx._h, self._h, arr(keys), arr(kval), arr(leaves), arr(lval), n_groups, C.c_void_p(stream)))
        ctx.synchronize(stream)
        return keys, kval, leaves, lval

    def group_entry_slots(self) -> int:
        n = C.c_int32()
        self.ctx.check(lib().fq_pipe_group_entry_slots(self.ctx._h, self._h, C.byref(n)))
        return n.value

    def export_partials(self, world: int, entries: "Column", stream: int = 0) -> List[int]:
        counts = (C.c_uint64 * 8)()
        self.ctx.check(lib().fq_pipe_export_partials(self.ctx._h, self._h, world, entries._h, counts, C.c_void_p(stream)))
        return [counts[i] for i in range(world)]

    def merge_partials(self, entries: Optional["Column"], n_entries: int, *, accumulate: bool = False, stream: int = 0) -> None:
        self.ctx.check(lib().fq_pipe_merge_partials(self.ctx._h, self._h, entries._h if entries is not None else None, n_entries,
                                                     RUN_ACCUMULATE if accumulate else 0, C.c_void_p(stream)))

    # ---- projection / filter ----
    def launch_project(self, source: Source, outs: Sequence[Column], capacity: int, *, limit: int = -1, early_exit: bool = False,
                       out_valid: Optional[Sequence[Optional[Column]]] = None, stream: int = 0):
        arr = (C.c_void_p * max(1, len(outs)))(*[c._h for c in outs])
        varr = None
        if out_valid is not None:
            varr = (C.c_void_p * max(1, len(outs)))(*[None if c is None else c._h for c in out_valid])
        self.ctx.check(lib().fq_pipe_launch_project(self.ctx._h, self._h, C.byref(source), arr, varr, capacity, limit,
                                                     RUN_LIMIT_EARLY_EXIT if early_exit else 0, C.c_void_p(stream)))

    def fetch_limit_row(self) -> int:
        """Source row that produced the last output row of a launch that filled its capacity (completes the LIMIT)."""
        row = C.c_uint64()
        self.ctx.check(lib().fq_pipe_fetch_limit_row(self.ctx._h, self._h, C.byref(row)))
        return row.value

    def fetch_project(self) -> Tuple[int, int]:
        sel, wr = C.c_uint64(), C.c_uint64()
        self.ctx.check(lib().fq_pipe_fetch_project(self.ctx._h, self._h, C.byref(sel), C.byref(wr)))
        return sel.value, wr.value

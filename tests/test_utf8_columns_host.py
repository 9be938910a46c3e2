"""Utf8 table columns, host side: the array -> (offsets, bytes, validity) conversion register_table uploads, and the
dictionary entry points of the C ABI (exported, bound in cabi, present in the generated Rust bindings).  No device."""
import ctypes
import os

import numpy as np
import pyarrow as pa
import pytest

from fuse_query_b200 import cabi
from fuse_query_b200.tables import utf8_parts

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEW_SYMBOLS = ["fq_utf8_bytes", "fq_utf8_download", "fq_utf8_take", "fq_utf8_dict_encode", "fq_utf8_bounds"]


def decode(parts):
    offsets, data, valid = parts
    assert offsets.dtype == np.int32 and offsets[0] == 0 and offsets[-1] == len(data)
    out = [data[offsets[i]:offsets[i + 1]].decode() for i in range(len(offsets) - 1)]
    if valid is not None:
        assert valid.dtype == np.uint8 and len(valid) == len(out)
        out = [v if ok else None for v, ok in zip(out, valid)]
    return out


VALUES = ["paris", None, "", "a\0b", "日本", "paris", None, "x" * 300]


@pytest.mark.parametrize("make", [
    lambda: pa.array(VALUES, type=pa.string()),
    lambda: pa.array(VALUES, type=pa.large_string()),
    lambda: pa.array(VALUES, type=pa.string()).dictionary_encode(),
    lambda: pa.chunked_array([VALUES[:3], VALUES[3:]], type=pa.string()),
    lambda: pa.chunked_array([pa.array(VALUES[:5]).dictionary_encode(), pa.array(VALUES[5:]).dictionary_encode()]),
    lambda: np.array(VALUES, dtype=object),
], ids=["string", "large_string", "dictionary", "chunked", "chunked_dictionary", "numpy_object"])
def test_string_columns_convert(make):
    assert decode(utf8_parts(make())) == VALUES


def test_sliced_arrays_are_rebased():
    arr = pa.array(["skip", "me", "a", None, "bc"])[2:]
    offsets, data, valid = utf8_parts(arr)
    assert offsets.tolist() == [0, 1, 1, 3] and data == b"abc" and valid.tolist() == [1, 0, 1]
    big = pa.array(["skip", "me", "a", "bc"], type=pa.large_string())[2:]
    assert decode(utf8_parts(big)) == ["a", "bc"]


def test_no_nulls_means_no_validity():
    offsets, data, valid = utf8_parts(np.array(["b", "aa", ""]))
    assert valid is None and data == b"baa" and offsets.tolist() == [0, 1, 3, 3]


def test_all_null_and_empty_columns():
    assert decode(utf8_parts(pa.array([None, None], type=pa.string()))) == [None, None]
    assert utf8_parts(pa.array([], type=pa.string()))[0].tolist() == [0]
    assert utf8_parts(pa.chunked_array([], type=pa.string()))[1] == b""


def test_non_string_columns_are_left_alone():
    assert utf8_parts(np.arange(3)) is None
    assert utf8_parts(pa.array([1, 2])) is None
    assert utf8_parts(np.array([1, "a"], dtype=object)) is None
    assert utf8_parts(pa.array([1, 2]).dictionary_encode()) is None


def test_dictionary_entry_points_are_exported_and_bound():
    lib = ctypes.CDLL(cabi.LIB_PATH)
    rust = open(os.path.join(ROOT, "ffi", "fuse-gpu-sys", "src", "lib.rs")).read()
    for name in NEW_SYMBOLS:
        assert hasattr(lib, name) and name in cabi.EXPORTS
        assert f"pub fn {name}(" in rust
    for method in ("nbytes", "to_list", "take", "dict_encode", "bounds"):
        assert callable(getattr(cabi.Utf8Array, method))

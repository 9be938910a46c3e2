"""Registering host data (numpy / pyarrow) as HBM-resident tables of a FuseQueryContext."""
from __future__ import annotations

from typing import Mapping

import numpy as np

from . import _fuse_host as h

_TAG = {np.dtype(np.bool_): h.DataType.Boolean, np.dtype(np.int8): h.DataType.Int8, np.dtype(np.int16): h.DataType.Int16,
        np.dtype(np.int32): h.DataType.Int32, np.dtype(np.int64): h.DataType.Int64, np.dtype(np.uint8): h.DataType.UInt8,
        np.dtype(np.uint16): h.DataType.UInt16, np.dtype(np.uint32): h.DataType.UInt32, np.dtype(np.uint64): h.DataType.UInt64,
        np.dtype(np.float32): h.DataType.Float32, np.dtype(np.float64): h.DataType.Float64}


def _arrow_column(col):
    """pyarrow ChunkedArray/Array -> (values, validity or None).  The validity comes back as ("bitmap", buffer, bit
    offset): the arrow null bitmap itself (1 bit per row, LSB first), which the device expands to its own layout (one
    byte per row) — no host-side unpacking."""
    import pyarrow as pa
    arr = col.combine_chunks() if isinstance(col, pa.ChunkedArray) else col
    if not arr.null_count:
        return arr.to_numpy(zero_copy_only=False), None
    zero = False if pa.types.is_boolean(arr.type) else 0
    values = arr.fill_null(zero).to_numpy(zero_copy_only=False)   # the payload of a NULL slot is never read as a value
    return values, ("bitmap", arr.buffers()[0], arr.offset)


_INT32_MAX = 2**31 - 1


def utf8_parts(col):
    """A string column -> (offsets, data, valid), or None when `col` holds no strings.

    `offsets` is int32 with len + 1 entries starting at 0, `data` the UTF-8 bytes, `valid` a uint8 array (1 = not NULL) or
    None when no slot is NULL.  Strings: pyarrow `string`, `large_string` and `dictionary<..., string>` arrays (chunked or
    sliced), numpy `str_` arrays and numpy `object` arrays of `str` / None.  More than 2 GiB of bytes is an error: the
    device keeps int32 offsets, like Arrow's `string`."""
    if isinstance(col, np.ndarray):
        if col.dtype.kind == "U":
            values = col.ravel().tolist()
        elif col.dtype == object and col.size and all(v is None or isinstance(v, str) for v in col.ravel().tolist()) \
                and any(isinstance(v, str) for v in col.ravel().tolist()):
            values = col.ravel().tolist()
        else:
            return None
        raw = [b"" if v is None else v.encode() for v in values]
        lens = np.fromiter((len(b) for b in raw), dtype=np.int64, count=len(raw))
        offsets = np.zeros(len(raw) + 1, dtype=np.int64)
        np.cumsum(lens, out=offsets[1:])
        _check_bytes(int(offsets[-1]))
        valid = None
        if any(v is None for v in values):
            valid = np.fromiter((v is not None for v in values), dtype=np.uint8, count=len(values))
        return offsets.astype(np.int32), b"".join(raw), valid
    if not hasattr(col, "null_count"):
        return None
    import pyarrow as pa

    def is_str(t):
        return pa.types.is_string(t) or pa.types.is_large_string(t)

    def plain(a):   # dictionary<..., string> -> its strings
        return a.dictionary_decode() if pa.types.is_dictionary(a.type) else a

    t = col.type
    if not (is_str(t) or (pa.types.is_dictionary(t) and is_str(t.value_type))):
        return None
    if isinstance(col, pa.ChunkedArray):
        chunks = [plain(c) for c in col.chunks]
        value_type = t.value_type if pa.types.is_dictionary(t) else t
        arr = pa.concat_arrays(chunks) if chunks else pa.array([], type=value_type)
    else:
        arr = plain(col)
    n = len(arr)
    if n == 0:
        return np.zeros(1, dtype=np.int32), b"", None
    wide = pa.types.is_large_string(arr.type)
    offs = np.frombuffer(arr.buffers()[1], dtype=np.int64 if wide else np.int32, count=n + 1, offset=arr.offset * (8 if wide else 4))
    begin, end = int(offs[0]), int(offs[-1])
    _check_bytes(end - begin)
    data_buf = arr.buffers()[2]
    data = data_buf.to_pybytes()[begin:end] if data_buf is not None else b""
    valid = np.asarray(arr.is_valid()).astype(np.uint8) if arr.null_count else None
    return (offs - begin).astype(np.int32), data, valid


def _check_bytes(n: int):
    if n > _INT32_MAX:
        raise h.FuseQueryError(f"Internal Error: Unsupported on the device path: a Utf8 column of {n} bytes (at most 2 GiB)")


def register_table(ctx, gpu, db: str, name: str, columns: Mapping[str, "np.ndarray"]):
    """Upload `columns` to HBM and register them as table `db.name`.  Returns the MemoryTable.

    A column is a numpy array (NOT NULL), a numpy masked array, a `(values, valid)` pair (valid: 1 = not NULL), or a
    pyarrow array; a pyarrow.Table is taken column by column.  Columns with NULLs become nullable fields whose validity
    rides beside the values as one byte per row.  String columns (see `utf8_parts`) become Utf8 fields, dictionary-encoded
    on the device: UInt32 codes over the sorted distinct strings, so that queries over them run as integer work."""
    if hasattr(columns, "column_names"):  # pyarrow.Table
        tbl = columns
        columns = {n: tbl.column(n) for n in tbl.column_names}
    fields, arrays = [], []
    for n, a in columns.items():
        parts = None if isinstance(a, tuple) else utf8_parts(a)
        if parts is not None:
            offsets, data, valid = parts
            fields.append(h.DataField(n, h.DataType.Utf8, valid is not None))
            arrays.append(h.DataArray.from_utf8(gpu, offsets, data, valid))
            continue
        valid = None
        if isinstance(a, tuple):
            a, valid = a
        elif isinstance(a, np.ma.MaskedArray):
            a, valid = a.filled(0), (None if a.mask is np.ma.nomask else (~np.ma.getmaskarray(a)).astype(np.uint8))
        elif hasattr(a, "null_count"):          # pyarrow Array / ChunkedArray
            a, valid = _arrow_column(a)
        a = np.ascontiguousarray(np.asarray(a))
        if a.dtype not in _TAG:
            raise h.FuseQueryError(f"Internal Error: Unsupported on the device path: column {n} of dtype {a.dtype}")
        fields.append(h.DataField(n, _TAG[a.dtype], valid is not None))
        if valid is None:
            arrays.append(h.DataArray.from_numpy(gpu, a))
        elif isinstance(valid, tuple) and valid[0] == "bitmap":
            arr = h.DataArray.from_numpy(gpu, a)
            arr.set_validity(h.DataArray.from_arrow_bitmap(gpu, valid[1].address, valid[2], len(a)))
            arrays.append(arr)
        else:
            arrays.append(h.DataArray.from_numpy_masked(gpu, a, np.asarray(valid)))
    table = h.MemoryTable(db, name, h.DataSchema(fields), arrays)
    ds = ctx.datasource()
    ds.add_database(db) if not _has_db(ds, db) else None
    ds.add_table(db, table)
    return table


def register_parquet(ctx, gpu, db: str, name: str, path, columns=None):
    """Read a Parquet file (or a directory of them) column by column into HBM and register it as table `db.name`:
    the reference's "table storage engine" slot (`datasources/table.rs:13-22`, README "Remote (S3 or other table
    storage engine)") filled with the one format this image can decode (pyarrow).  Decoding is host work done once at
    registration; queries then run against the resident columns.  `columns` restricts what is loaded."""
    import pyarrow.parquet as pq
    return register_table(ctx, gpu, db, name, pq.read_table(str(path), columns=list(columns) if columns else None))


def register_arrow_ipc(ctx, gpu, db: str, name: str, path, columns=None):
    """Same for an Arrow IPC (Feather v2) file, memory-mapped: the uploads read straight from the page cache."""
    import pyarrow as pa
    import pyarrow.ipc as ipc
    with pa.memory_map(str(path), "r") as f:
        tbl = ipc.open_file(f).read_all()
        if columns:
            tbl = tbl.select(list(columns))
        return register_table(ctx, gpu, db, name, tbl)


def _has_db(ds, db: str) -> bool:
    try:
        ds.get_table(db, "\0")
    except h.FuseQueryError as e:
        return "Cannot find the database" not in str(e)
    return True

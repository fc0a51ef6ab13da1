"""ctypes binding of libllkv_gpu.so (include/llkv_gpu.h) + the host-side mirror of the reference's call shape.

`DeviceTable` stands where a `Table` backed by a `ColumnStore` stands in the reference (llkv-table/src/table.rs:231-490):
chunks are appended column by column (`ColumnStore::append`, llkv-column-map/src/store/core.rs:787), then
`filter_row_ids` / aggregate scans run against it (llkv-executor/src/lib.rs:5357-5682, 4405-4542).

There is NO CPU fallback: importing works anywhere, but `Context()` raises `LlkvError(Io)` without a CUDA device and
`load()` raises if the CUDA library has not been built.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np

from . import ffi
from .expr import (AggregateSpec, AggregateValue, Expr, ProgramCompiler, decode_group_key, flatten_aggregates)
from .table import HostColumn, HostTable, LlkvError, Snapshot

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(os.path.dirname(_HERE), "csrc", "libllkv_gpu.so")

# LogicalStorageNamespace (llkv-types/src/ids.rs:20-62)
NS_USER, NS_ROW_ID_SHADOW, NS_TXN_CREATED_BY, NS_TXN_DELETED_BY = 0, 1, 2, 3
# chunk sizes the reference's append path produces (llkv-column-map/src/store/constants.rs:14-28, slicing.rs:33-43,155-166)
TARGET_CHUNK_BYTES = 1 << 20
VARWIDTH_FALLBACK_ROWS = 4096

_lib = None
# llkv_chunk_visitor: (user, prim_type, values, row_ids, n_rows) -> status
CHUNK_VISITOR = C.CFUNCTYPE(C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.POINTER(C.c_uint64), C.c_uint64)


def load():
    """dlopens libllkv_gpu.so; raises if it is missing (the product path has no other implementation)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"{LIB_PATH} is missing: build it with rust-llkv_b200/csrc/build.sh (there is no CPU fallback)")
    lib = C.CDLL(LIB_PATH)
    P = C.POINTER
    vp, u64, i32, u8, i8 = C.c_void_p, C.c_uint64, C.c_int32, C.c_uint8, C.c_int8
    sig = {
        "llkv_gpu_abi_version": (i32, []),
        "llkv_gpu_last_error": (C.c_size_t, [C.c_char_p, C.c_size_t]),
        "llkv_gpu_device_count": (i32, []),
        "llkv_gpu_ctx_create": (i32, [i32, i32, u64, P(vp)]),
        "llkv_gpu_ctx_destroy": (None, [vp]),
        "llkv_gpu_ctx_synchronize": (i32, [vp]),
        "llkv_gpu_ctx_stream": (i32, [vp, P(vp)]),
        "llkv_gpu_ctx_set_timing": (i32, [vp, i32]),
        "llkv_gpu_ctx_set_tuning": (i32, [vp, i32, i32, i32, i32, i32]),
        "llkv_gpu_ctx_set_jit": (i32, [vp, i32]),
        "llkv_gpu_ctx_set_partitioning": (i32, [vp, i32]),
        "llkv_gpu_ctx_set_pruning": (i32, [vp, i32]),
        "llkv_gpu_debug_plan": (i32, [vp, i32, vp, i32, i32, u64, u64, vp, i32, vp, i32, vp, i32, i32, u64, i32, i32, i32, i32, i32,
                                       C.c_char_p, C.c_char_p, u64]),
        "llkv_gpu_descriptor_parse": (i32, [vp, u64, vp]),
        "llkv_gpu_descriptor_page_parse": (i32, [vp, u64, P(u64), vp, u64, P(u64)]),
        "llkv_gpu_sortable_u64": (u64, [i32, u64]),
        "llkv_gpu_chunk_stats": (i32, [i32, vp, u64, vp, vp]),
        "llkv_gpu_chunk_overlaps": (i32, [i32, u64, u64, vp, vp]),
        "llkv_gpu_host_alloc": (i32, [u64, P(vp)]),
        "llkv_gpu_host_free": (i32, [vp]),
        "llkv_gpu_host_register": (i32, [vp, u64]),
        "llkv_gpu_host_unregister": (i32, [vp]),
        "llkv_gpu_column_register": (i32, [vp, u64, i32, u8, i8, P(vp)]),
        "llkv_gpu_column_reserve": (i32, [vp, u64]),
        "llkv_gpu_column_append_chunk": (i32, [vp, u64, vp, u64, vp, vp, u64, vp]),
        "llkv_gpu_column_append_blob": (i32, [vp, u64, vp, u64, vp, u64]),
        "llkv_gpu_column_seal": (i32, [vp]),
        "llkv_gpu_column_flush": (i32, [vp]),
        "llkv_gpu_column_delete_rows": (i32, [vp, vp, u64]),
        "llkv_gpu_column_present_rows": (i32, [vp, P(u64)]),
        "llkv_gpu_column_dict_size": (i32, [vp, P(u64)]),
        "llkv_gpu_column_dict_entry": (i32, [vp, u64, P(vp), P(u64)]),
        "llkv_gpu_column_build_sort_index": (i32, [vp, u64]),
        "llkv_gpu_column_sort_index_blob": (i32, [vp, u64, vp, u64, P(u64)]),
        "llkv_gpu_column_gather": (i32, [vp, vp, u64, vp, u64, vp]),
        "llkv_gpu_column_visit": (i32, [vp, u64, i32, CHUNK_VISITOR, vp]),
        "llkv_gpu_column_scan": (i32, [vp, vp, P(ffi.ScanOptions), u64, CHUNK_VISITOR, vp]),
        "llkv_gpu_column_h2d_bytes": (i32, [vp, P(u64)]),
        "llkv_gpu_ctx_set_upload_threads": (i32, [vp, i32]),
        "llkv_gpu_ctx_set_dma_share": (i32, [vp, i32]),
        "llkv_gpu_column_rows": (i32, [vp, P(u64)]),
        "llkv_gpu_column_read": (i32, [vp, u64, u64, vp, u64]),
        "llkv_gpu_column_clear": (i32, [vp]),
        "llkv_gpu_column_destroy": (i32, [vp]),
        "llkv_gpu_program_compile": (i32, [vp, vp, i32, vp, i32, vp, i32, vp, i32, P(vp)]),
        "llkv_gpu_program_destroy": (None, [vp]),
        "llkv_gpu_mvcc_set": (i32, [vp, u64, vp, vp, u64, u64, vp, i32]),
        "llkv_gpu_mvcc_clear": (i32, [vp, u64]),
        "llkv_gpu_filter_bitmap": (i32, [vp, u64, vp, i32, u64, u64, vp, u64, P(u64)]),
        "llkv_gpu_agg_create": (i32, [vp, u64, vp, i32, vp, i32, vp, i32, i32, u64, P(vp)]),
        "llkv_gpu_agg_reset": (i32, [vp]),
        "llkv_gpu_agg_run": (i32, [vp, vp, i32, u64, u64]),
        "llkv_gpu_agg_merge": (i32, [vp]),
        "llkv_gpu_agg_execute": (i32, [vp, vp, i32, u64, u64, i32]),
        "llkv_gpu_ctx_set_graphs": (i32, [vp, i32]),
        "llkv_gpu_agg_group_count": (i32, [vp, P(u64)]),
        "llkv_gpu_agg_finalize": (i32, [vp, vp, vp, u64, P(u64)]),
        "llkv_gpu_agg_run_info": (i32, [vp, P(ffi.RunInfo)]),
        "llkv_gpu_agg_set_output": (i32, [vp, vp, i32, vp, i32, u64, u64]),
        "llkv_gpu_agg_destroy": (None, [vp]),
        "llkv_gpu_comm_unique_id": (i32, [vp]),
        "llkv_gpu_comm_init": (i32, [vp, vp, i32, i32]),
        "llkv_gpu_comm_destroy": (i32, [vp]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if lib.llkv_gpu_abi_version() != 1:
        raise RuntimeError("libllkv_gpu.so ABI version mismatch")
    _lib = lib
    return lib


def last_error() -> str:
    buf = C.create_string_buffer(2048)
    load().llkv_gpu_last_error(buf, 2048)
    return buf.value.decode(errors="replace")


def _check(rc: int):
    if rc:
        raise LlkvError(rc, last_error())


def logical_field_id(table_id: int, field_id: int, namespace: int = NS_USER) -> int:
    """LogicalFieldId::from_parts (llkv-types/src/ids.rs:133-175): field 32 | table 16 | namespace 16."""
    return (field_id & 0xFFFFFFFF) | ((table_id & 0xFFFF) << 32) | ((namespace & 0xFFFF) << 48)


def device_count() -> int:
    return int(load().llkv_gpu_device_count())


class Context:
    """One per GPU (llkv_gpu_ctx)."""

    def __init__(self, device: int = 0, n_streams: int = 4, pinned_bytes: int = 64 << 20):
        self.lib = load()
        h = C.c_void_p()
        _check(self.lib.llkv_gpu_ctx_create(device, n_streams, pinned_bytes, C.byref(h)))
        self.handle = h
        self.device = device

    def close(self):
        if self.handle:
            self.lib.llkv_gpu_ctx_destroy(self.handle)
            self.handle = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def synchronize(self):
        _check(self.lib.llkv_gpu_ctx_synchronize(self.handle))

    def stream(self) -> int:
        s = C.c_void_p()
        _check(self.lib.llkv_gpu_ctx_stream(self.handle, C.byref(s)))
        return int(s.value or 0)

    def set_timing(self, enabled: bool):
        _check(self.lib.llkv_gpu_ctx_set_timing(self.handle, int(enabled)))

    def set_tuning(self, ctas_per_sm=0, block_threads=0, stages=0, rows_per_thread=0, force_wide=0):
        _check(self.lib.llkv_gpu_ctx_set_tuning(self.handle, ctas_per_sm, block_threads, stages, rows_per_thread, force_wide))

    def set_jit(self, mode: int):
        """0 = interpret the lean program, 1 = specialise a plan shape from its second run on (default), 2 = always."""
        _check(self.lib.llkv_gpu_ctx_set_jit(self.handle, mode))

    def set_partitioning(self, mode: int):
        """Partitioned high-cardinality GROUP BY: 0 = never, 1 = when the group table exceeds L2 (default), 2 = whenever
        the plan allows it."""
        _check(self.lib.llkv_gpu_ctx_set_partitioning(self.handle, mode))

    def set_pruning(self, mode: int):
        """Zone-map tile skipping: 0 = never, 1 = for columns scanned again unchanged when >= 1/8 of the tiles drop out
        (default), 2 = from the first scan, whenever any tile drops out."""
        _check(self.lib.llkv_gpu_ctx_set_pruning(self.handle, mode))

    def set_graphs(self, mode: int):
        """Aggregation.execute replays a captured CUDA graph once a step repeats unchanged: 1 (default) / 0."""
        _check(self.lib.llkv_gpu_ctx_set_graphs(self.handle, mode))

    def set_upload_threads(self, n_threads: int):
        """Host workers narrowing Decimal128 chunks from page-locked sources before the DMA: -1 default, 0 off."""
        _check(self.lib.llkv_gpu_ctx_set_upload_threads(self.handle, n_threads))

    def set_dma_share(self, percent: int = -1):
        """Share of a hybrid Decimal128 upload that goes to the copy engine as it lies (narrowed on the device); -1 = automatic."""
        _check(self.lib.llkv_gpu_ctx_set_dma_share(self.handle, percent))

    # ---- multi-GPU (NCCL over NVLink): the unique id travels through whatever the host uses for rendezvous
    def comm_unique_id(self) -> bytes:
        buf = (C.c_uint8 * ffi.UNIQUE_ID_BYTES)()
        _check(self.lib.llkv_gpu_comm_unique_id(buf))
        return bytes(buf)

    def comm_init(self, unique_id: bytes, n_ranks: int, rank: int):
        buf = (C.c_uint8 * ffi.UNIQUE_ID_BYTES)(*unique_id)
        _check(self.lib.llkv_gpu_comm_init(self.handle, buf, n_ranks, rank))

    def comm_destroy(self):
        _check(self.lib.llkv_gpu_comm_destroy(self.handle))


def pinned_empty(nbytes: int) -> Tuple[np.ndarray, int]:
    """Page-locked host buffer as a uint8 numpy view (llkv_gpu_host_alloc); free with pinned_free(ptr)."""
    p = C.c_void_p()
    _check(load().llkv_gpu_host_alloc(nbytes, C.byref(p)))
    arr = np.ctypeslib.as_array((C.c_uint8 * max(1, nbytes)).from_address(p.value))
    return arr[:nbytes], int(p.value)


def pinned_free(ptr: int):
    _check(load().llkv_gpu_host_free(C.c_void_p(ptr)))


def host_register(buf) -> int:
    """Page-locks a buffer the caller owns (numpy array or mmap: the pager's blob memory) so appends DMA straight out of
    it; returns the address to pass to host_unregister."""
    arr = np.frombuffer(buf, dtype=np.uint8) if not isinstance(buf, np.ndarray) else buf
    ptr = arr.ctypes.data
    _check(load().llkv_gpu_host_register(C.c_void_p(ptr), arr.nbytes))
    return ptr


def host_unregister(ptr: int):
    _check(load().llkv_gpu_host_unregister(C.c_void_p(ptr)))


def chunk_rows_for(dtype_type: int) -> int:
    """Rows per chunk the reference's append path produces for a column of this type (slicing.rs:33-43,155-166)."""
    w = {ffi.PT_UINT64: 8, ffi.PT_INT64: 8, ffi.PT_FLOAT64: 8, ffi.PT_INT32: 4, ffi.PT_UINT32: 4, ffi.PT_FLOAT32: 4,
         ffi.PT_INT16: 2, ffi.PT_UINT16: 2, ffi.PT_INT8: 1, ffi.PT_UINT8: 1}.get(dtype_type)
    return TARGET_CHUNK_BYTES // w if w else VARWIDTH_FALLBACK_ROWS


class DeviceColumn:
    def __init__(self, ctx: Context, lfid: int, col: HostColumn):
        self.ctx = ctx
        self.lib = ctx.lib
        self.dtype = col.dtype
        self.lfid = lfid
        h = C.c_void_p()
        _check(self.lib.llkv_gpu_column_register(ctx.handle, lfid, col.dtype.type, col.dtype.precision, col.dtype.scale, C.byref(h)))
        self.handle = h
        self.next_pk = 1

    def reserve(self, n_rows: int):
        _check(self.lib.llkv_gpu_column_reserve(self.handle, n_rows))

    def append(self, col: HostColumn, chunk_rows: Optional[int] = None, row_id_base: Optional[int] = None, as_blob: bool = False):
        """Appends `col` in chunks of `chunk_rows` rows (default: the reference's chunking for the type)."""
        n = col.n_rows
        if chunk_rows is None:
            chunk_rows = chunk_rows_for(col.dtype.type)
        base = self.rows() if row_id_base is None else row_id_base
        t = col.dtype.type
        for lo in range(0, max(n, 0), chunk_rows):
            hi = min(n, lo + chunk_rows)
            m = hi - lo
            validity = None
            if col.validity is not None:
                bits = np.unpackbits(col.validity, bitorder="little")[lo:hi]
                validity = np.packbits(bits, bitorder="little")
            vptr = C.c_void_p(validity.ctypes.data) if validity is not None else None
            if t == ffi.PT_UTF8:
                offs = col.values[lo:hi + 1]
                _check(self.lib.llkv_gpu_column_append_chunk(self.handle, self.next_pk, C.c_void_p(offs.ctypes.data), m, vptr, None,
                                                              base + lo, C.c_void_p(col.aux.ctypes.data) if col.aux.size else None))
            elif as_blob and validity is None:
                blob = HostColumn(col.field_id, col.dtype, col.values[lo:hi]).serialize()
                _check(self.lib.llkv_gpu_column_append_blob(self.handle, self.next_pk, blob, len(blob), None, base + lo))
            else:
                vals = col.values[lo:hi]
                _check(self.lib.llkv_gpu_column_append_chunk(self.handle, self.next_pk, C.c_void_p(vals.ctypes.data), m, vptr, None,
                                                              base + lo, None))
            self.next_pk += 1

    def append_raw(self, ptr: int, n_rows: int, row_id_base: int):
        """One chunk from a raw pointer: host memory (e.g. a slice of a pinned buffer) or device memory of this GPU."""
        _check(self.lib.llkv_gpu_column_append_chunk(self.handle, self.next_pk, C.c_void_p(ptr), n_rows, None, None, row_id_base, None))
        self.next_pk += 1

    def append_rows(self, values: np.ndarray, row_ids: np.ndarray, first_row_id: int = 0, validity: Optional[np.ndarray] = None,
                    aux: Optional[np.ndarray] = None):
        """One chunk with its row-id shadow column (ColumnStore::append with arbitrary row ids): rows land at position
        row id - first_row_id; a row id that is already there is overwritten (last writer wins).  For a Utf8 column
        `values` is the chunk's int32 offsets (one more than the row ids) and `aux` its data bytes."""
        vals = np.ascontiguousarray(values, dtype=np.int32) if self.dtype.type == ffi.PT_UTF8 else np.ascontiguousarray(values)
        ids = np.ascontiguousarray(row_ids, dtype=np.uint64)
        vptr = C.c_void_p(validity.ctypes.data) if validity is not None else None
        data = np.ascontiguousarray(aux, dtype=np.uint8) if aux is not None else None
        aptr = C.c_void_p(data.ctypes.data) if data is not None and data.size else None
        _check(self.lib.llkv_gpu_column_append_chunk(self.handle, self.next_pk, C.c_void_p(vals.ctypes.data), ids.shape[0], vptr,
                                                      C.c_void_p(ids.ctypes.data), first_row_id, aptr))
        self.next_pk += 1

    def delete_rows(self, row_ids):
        ids = np.ascontiguousarray(row_ids, dtype=np.uint64)
        _check(self.lib.llkv_gpu_column_delete_rows(self.handle, C.c_void_p(ids.ctypes.data), ids.shape[0]))

    def gather(self, row_ids):
        """gather_rows(IncludeNulls): [value or None, ...] for the row ids, in request order (fixed-width columns)."""
        ids = np.ascontiguousarray(row_ids, dtype=np.uint64)
        t = self.dtype.type
        if t == ffi.PT_DECIMAL128:
            out = np.zeros((ids.shape[0], 2), dtype=np.uint64)
        else:
            np_t = {ffi.PT_UINT64: np.uint64, ffi.PT_INT64: np.int64, ffi.PT_FLOAT64: np.float64, ffi.PT_INT32: np.int32, ffi.PT_UINT32: np.uint32,
                    ffi.PT_FLOAT32: np.float32, ffi.PT_DATE32: np.int32, ffi.PT_INT16: np.int16, ffi.PT_UINT16: np.uint16, ffi.PT_INT8: np.int8,
                    ffi.PT_UINT8: np.uint8, ffi.PT_BOOLEAN: np.uint8, ffi.PT_DATE64: np.int64}[t]
            out = np.zeros(ids.shape[0], dtype=np_t)
        valid = np.zeros(ids.shape[0], dtype=np.uint8)
        _check(self.lib.llkv_gpu_column_gather(self.handle, C.c_void_p(ids.ctypes.data), ids.shape[0], C.c_void_p(out.ctypes.data), out.nbytes,
                                               C.c_void_p(valid.ctypes.data)))
        if t == ffi.PT_DECIMAL128:
            return [ffi.words_to_i128(int(lo), int(hi)) if v else None for (lo, hi), v in zip(out, valid)]
        return [x.item() if v else None for x, v in zip(out, valid)]

    def visit(self, on_chunk, chunk_rows: int = 0, with_row_ids: bool = False):
        """ColumnStore::scan with an unsorted visitor: on_chunk(values ndarray[, row_ids ndarray]) per chunk
        (PrimitiveVisitor::*_chunk / PrimitiveWithRowIdsVisitor::*_chunk_with_rids)."""
        t = self.dtype.type
        np_t = {ffi.PT_UINT64: np.uint64, ffi.PT_INT64: np.int64, ffi.PT_FLOAT64: np.float64, ffi.PT_INT32: np.int32, ffi.PT_UINT32: np.uint32,
                ffi.PT_FLOAT32: np.float32, ffi.PT_DATE32: np.int32, ffi.PT_INT16: np.int16, ffi.PT_UINT16: np.uint16, ffi.PT_INT8: np.int8,
                ffi.PT_UINT8: np.uint8, ffi.PT_BOOLEAN: np.uint8, ffi.PT_DATE64: np.int64, ffi.PT_DECIMAL128: np.uint64}[t]
        per_row = 2 if t == ffi.PT_DECIMAL128 else 1

        def trampoline(_user, prim_type, values, row_ids, n):
            assert prim_type == t
            vals = np.ctypeslib.as_array(C.cast(values, C.POINTER(np.ctypeslib.as_ctypes_type(np_t))), shape=(n * per_row,)).copy()
            if per_row == 2:
                vals = vals.reshape(n, 2)
            if with_row_ids:
                on_chunk(vals, np.ctypeslib.as_array(row_ids, shape=(n,)).copy())
            else:
                on_chunk(vals)
            return 0

        cb = CHUNK_VISITOR(trampoline)
        _check(self.lib.llkv_gpu_column_visit(self.handle, chunk_rows, int(with_row_ids), cb, None))

    def scan(self, on_run, sorted: bool = False, reverse: bool = False, with_row_ids: bool = False, limit: Optional[int] = None, offset: int = 0,
             include_nulls: bool = False, nulls_first: bool = False, anchor: Optional["DeviceColumn"] = None, lower=None, upper=None,
             chunk_rows: int = 0):
        """ColumnStore::scan(field, ScanOptions, visitor): on_run(values | None, row_ids | None) per chunk; values None = a null run.
        lower / upper: (value, inclusive) bounds in the column's type."""
        t = self.dtype.type
        np_t = {ffi.PT_UINT64: np.uint64, ffi.PT_INT64: np.int64, ffi.PT_FLOAT64: np.float64, ffi.PT_INT32: np.int32, ffi.PT_UINT32: np.uint32,
                ffi.PT_FLOAT32: np.float32, ffi.PT_DATE32: np.int32, ffi.PT_INT16: np.int16, ffi.PT_UINT16: np.uint16, ffi.PT_INT8: np.int8,
                ffi.PT_UINT8: np.uint8, ffi.PT_BOOLEAN: np.uint8, ffi.PT_DATE64: np.int64, ffi.PT_DECIMAL128: np.uint64}[t]
        per_row = 2 if t == ffi.PT_DECIMAL128 else 1
        o = ffi.ScanOptions()
        o.sorted, o.reverse, o.with_row_ids, o.include_nulls, o.nulls_first = int(sorted), int(reverse), int(with_row_ids), int(include_nulls), int(nulls_first)
        o.offset, o.limit = offset, 0 if limit is None else limit
        if limit == 0:
            return

        def bits_of(v):
            if np_t in (np.float64,):
                return int(np.array([v], np.float64).view(np.uint64)[0])
            if np_t in (np.float32,):
                return int(np.array([v], np.float32).view(np.uint32)[0])
            return int(v) & 0xFFFFFFFFFFFFFFFF

        if lower is not None:
            o.has_lower, o.lower_inclusive, o.lower_bits = 1, int(lower[1]), bits_of(lower[0])
        if upper is not None:
            o.has_upper, o.upper_inclusive, o.upper_bits = 1, int(upper[1]), bits_of(upper[0])

        def trampoline(_user, prim_type, values, row_ids, n):
            ids = np.ctypeslib.as_array(row_ids, shape=(n,)).copy() if row_ids else None
            if not values:
                on_run(None, ids)
                return 0
            vals = np.ctypeslib.as_array(C.cast(values, C.POINTER(np.ctypeslib.as_ctypes_type(np_t))), shape=(n * per_row,)).copy()
            on_run(vals.reshape(n, 2) if per_row == 2 else vals, ids)
            return 0

        cb = CHUNK_VISITOR(trampoline)
        _check(self.lib.llkv_gpu_column_scan(self.handle, anchor.handle if anchor else None, C.byref(o), chunk_rows, cb, None))

    def build_sort_index(self, chunk_rows: int = 0):
        _check(self.lib.llkv_gpu_column_build_sort_index(self.handle, chunk_rows))

    def sort_index_blob(self, chunk_index: int) -> bytes:
        """The chunk's value_order_perm blob ("ARR0", UInt32 indices) as the pager would store it."""
        n = C.c_uint64()
        _check(self.lib.llkv_gpu_column_sort_index_blob(self.handle, chunk_index, None, 0, C.byref(n)))
        buf = (C.c_uint8 * n.value)()
        _check(self.lib.llkv_gpu_column_sort_index_blob(self.handle, chunk_index, buf, n.value, C.byref(n)))
        return bytes(buf)

    def dict_size(self) -> int:
        """Distinct strings of a Utf8 column that holds strings longer than 7 bytes (0: the column is not dictionary-coded)."""
        n = C.c_uint64()
        _check(self.lib.llkv_gpu_column_dict_size(self.handle, C.byref(n)))
        return n.value

    def dict_entry(self, code: int) -> str:
        ptr = C.c_void_p()
        n = C.c_uint64()
        _check(self.lib.llkv_gpu_column_dict_entry(self.handle, code, C.byref(ptr), C.byref(n)))
        return C.string_at(ptr, n.value).decode("utf-8") if n.value else ""

    def present_rows(self) -> int:
        n = C.c_uint64()
        _check(self.lib.llkv_gpu_column_present_rows(self.handle, C.byref(n)))
        return int(n.value)

    def seal(self):
        _check(self.lib.llkv_gpu_column_seal(self.handle))

    def flush(self):
        """Issues and waits for the copies the appends left pending; page-locked sources may be reused afterwards."""
        _check(self.lib.llkv_gpu_column_flush(self.handle))

    def h2d_bytes(self) -> int:
        n = C.c_uint64()
        _check(self.lib.llkv_gpu_column_h2d_bytes(self.handle, C.byref(n)))
        return int(n.value)

    def read(self, row_begin: int = 0, n_rows: Optional[int] = None) -> np.ndarray:
        """Rows of the resident image back in the Arrow values layout (what a PrimitiveVisitor chunk callback would see)."""
        n_rows = self.rows() - row_begin if n_rows is None else n_rows
        t = self.dtype.type
        if t == ffi.PT_DECIMAL128:
            out = np.empty((n_rows, 2), dtype=np.uint64)
        else:
            np_t = {ffi.PT_UINT64: np.uint64, ffi.PT_INT64: np.int64, ffi.PT_FLOAT64: np.float64, ffi.PT_INT32: np.int32, ffi.PT_UINT32: np.uint32,
                    ffi.PT_FLOAT32: np.float32, ffi.PT_DATE32: np.int32, ffi.PT_INT16: np.int16, ffi.PT_UINT16: np.uint16, ffi.PT_INT8: np.int8,
                    ffi.PT_UINT8: np.uint8, ffi.PT_BOOLEAN: np.uint8, ffi.PT_DATE64: np.int64}[t]
            out = np.empty(n_rows, dtype=np_t)
        _check(self.lib.llkv_gpu_column_read(self.handle, row_begin, n_rows, C.c_void_p(out.ctypes.data), out.nbytes))
        return out

    def clear(self):
        _check(self.lib.llkv_gpu_column_clear(self.handle))

    def rows(self) -> int:
        n = C.c_uint64()
        _check(self.lib.llkv_gpu_column_rows(self.handle, C.byref(n)))
        return int(n.value)

    def destroy(self):
        if self.handle:
            self.lib.llkv_gpu_column_destroy(self.handle)
            self.handle = None


class Program:
    """A compiled predicate (llkv_gpu_program): ProgramCompiler::compile output crossing the boundary."""

    def __init__(self, ctx: Context, expr: Expr):
        self.lib = ctx.lib
        cp = ProgramCompiler(expr).compile()
        ops, n_ops, lits, n_lits, nodes, n_nodes, roots, n_roots = cp.c_arrays()
        h = C.c_void_p()
        _check(self.lib.llkv_gpu_program_compile(ctx.handle, ops, n_ops, lits, n_lits, nodes, n_nodes, roots, n_roots, C.byref(h)))
        self.handle = h

    def destroy(self):
        if self.handle:
            self.lib.llkv_gpu_program_destroy(self.handle)
            self.handle = None


class Aggregation:
    """A set of AggregateStates fused with the scan that feeds them (llkv_gpu_agg)."""

    def __init__(self, table: "DeviceTable", specs: Sequence[AggregateSpec], group_by: Sequence[int] = (),
                 expr_mode: Optional[int] = None, cardinality_hint: int = 0):
        self.table = table
        self.lib = table.ctx.lib
        self.n_aggs = len(specs)
        self.n_keys = len(group_by)
        self.group_by = tuple(group_by)
        if expr_mode is None:
            expr_mode = ffi.EXPR_EXACT if group_by else ffi.EXPR_ARROW
        aggs, n_aggs, nodes, n_nodes = flatten_aggregates(specs)
        keys = (C.c_uint64 * max(1, len(group_by)))(*group_by)
        h = C.c_void_p()
        _check(self.lib.llkv_gpu_agg_create(table.ctx.handle, table.table_id, aggs, n_aggs, nodes, n_nodes, keys, len(group_by),
                                            expr_mode, cardinality_hint, C.byref(h)))
        self.handle = h

    def reset(self):
        _check(self.lib.llkv_gpu_agg_reset(self.handle))

    def run(self, program: Optional[Program] = None, apply_mvcc: bool = False, row_begin: int = 0, row_end: Optional[int] = None):
        row_end = self.table.n_rows if row_end is None else row_end
        _check(self.lib.llkv_gpu_agg_run(self.handle, program.handle if program else None, int(apply_mvcc), row_begin, row_end))

    def merge(self):
        _check(self.lib.llkv_gpu_agg_merge(self.handle))

    def execute(self, program: Optional[Program] = None, apply_mvcc: bool = False, row_begin: int = 0, row_end: Optional[int] = None,
                merge: bool = True):
        """reset + run + (merge, when the context has peers) in one call (llkv_gpu_agg_execute)."""
        row_end = self.table.n_rows if row_end is None else row_end
        _check(self.lib.llkv_gpu_agg_execute(self.handle, program.handle if program else None, int(apply_mvcc), row_begin, row_end, int(merge)))

    def set_output(self, having=(), order_by=(), offset: int = 0, limit: int = 0):
        """HAVING / ORDER BY / OFFSET / LIMIT over the finalized rows.  having: [("agg" | "key", index, CompareOp code, literal)],
        order_by: [("agg" | "key", index, descending, nulls_first)]."""
        from .expr import lit
        h = (ffi.HavingTerm * max(1, len(having)))()
        for i, (what, index, op, value) in enumerate(having):
            h[i].is_aggregate = int(what == "agg")
            h[i].index = index
            h[i].cmp_op = op
            h[i].literal = lit(value).to_c()
        o = (ffi.OrderKey * max(1, len(order_by)))()
        for i, (what, index, descending, nulls_first) in enumerate(order_by):
            o[i].is_aggregate = int(what == "agg")
            o[i].index = index
            o[i].descending = int(descending)
            o[i].nulls_first = int(nulls_first)
        _check(self.lib.llkv_gpu_agg_set_output(self.handle, h, len(having), o, len(order_by), offset, limit))

    def group_count(self) -> int:
        n = C.c_uint64()
        _check(self.lib.llkv_gpu_agg_group_count(self.handle, C.byref(n)))
        return int(n.value)

    def finalize_raw(self, group_capacity: int):
        """llkv_gpu_agg_finalize into C arrays (llkv_agg_value / llkv_group_key), kept and reused per capacity."""
        buf = getattr(self, "_raw", None)
        if buf is None or buf[0] != group_capacity:
            buf = (group_capacity, (ffi.AggValue * (group_capacity * max(1, self.n_aggs)))(),
                   (ffi.GroupKey * (group_capacity * max(1, self.n_keys)))())
            self._raw = buf
        _, vals, keys = buf
        n = C.c_uint64()
        _check(self.lib.llkv_gpu_agg_finalize(self.handle, vals, keys, group_capacity, C.byref(n)))
        return vals, keys, int(n.value)

    AGG_VALUE_DTYPE = np.dtype([("lo", "<u8"), ("hi", "<u8"), ("type", "<i4"), ("precision", "u1"), ("scale", "i1"), ("valid", "u1"), ("_pad", "u1")])
    GROUP_KEY_DTYPE = np.dtype([("bits", "<u8"), ("type", "<i4"), ("valid", "u1"), ("dict", "u1"), ("_pad", "u1", (2,))])

    def finalize_numpy(self, group_capacity: int):
        """The finalized cells as numpy structured arrays [groups, aggregates] / [groups, keys] (for results with millions of
        groups: no Python object per cell)."""
        vals, keys, n = self.finalize_raw(group_capacity)
        v = np.frombuffer(vals, dtype=self.AGG_VALUE_DTYPE, count=n * self.n_aggs).reshape(n, self.n_aggs)
        k = np.frombuffer(keys, dtype=self.GROUP_KEY_DTYPE, count=n * self.n_keys).reshape(n, self.n_keys) if self.n_keys else None
        return v, k, n

    def decode(self, vals, keys, n):
        rows = []
        for g in range(n):
            key = tuple(decode_group_key(keys[g * self.n_keys + k], lambda kind, code, k=k: self.table.columns[self.group_by[k]].dict_entry(code))
                        for k in range(self.n_keys))
            rows.append((key, [AggregateValue.from_c(vals[g * self.n_aggs + a]) for a in range(self.n_aggs)]))
        return rows

    def finalize(self, group_capacity: Optional[int] = None):
        """[(key_tuple, [AggregateValue, ...]), ...] in first-appearance order of the groups."""
        if group_capacity is None:
            group_capacity = self.group_count() if self.n_keys else 1
            group_capacity = max(1, group_capacity)
        vals, keys, n = self.finalize_raw(group_capacity)
        return self.decode(vals, keys, n)

    def run_info(self) -> ffi.RunInfo:
        info = ffi.RunInfo()
        _check(self.lib.llkv_gpu_agg_run_info(self.handle, C.byref(info)))
        return info

    def destroy(self):
        if self.handle:
            self.lib.llkv_gpu_agg_destroy(self.handle)
            self.handle = None


def shard_rows(n_rows: int, world: int, rank: int, align: int = 131072) -> Tuple[int, int]:
    """Row range [begin, end) of `rank` among `world` GPUs: contiguous, aligned to `align` rows (a chunk boundary:
    131 072 = one 1 MiB Int64 chunk, llkv-column-map/src/store/slicing.rs:33-43) so every column of a shard covers the
    same chunks; the last rank takes the remainder (SURVEY.md §8e)."""
    if world <= 0 or not (0 <= rank < world):
        raise ValueError("bad rank/world")
    units = (n_rows + align - 1) // align
    lo = units * rank // world * align
    hi = units * (rank + 1) // world * align
    return min(lo, n_rows), (n_rows if rank == world - 1 else min(hi, n_rows))


def merge_partial_results(parts, rules):
    """Host-side statement of what llkv_gpu_agg_merge does on the device for SUM/COUNT/MIN/MAX states: folds per-rank
    finalized rows [(key, [AggregateValue...])] in rank order; `rules[i]` is "sum", "min" or "max" for aggregate i
    (COUNT merges as "sum"; AVG is merged as its (sum, count) pair and divided afterwards, as the device keeps it).
    NULL (no rows seen on that rank) is the identity.  Used by the multi-rank CPU tests."""
    import dataclasses
    merged, order = {}, []
    for rows in parts:
        for key, vals in rows:
            if key not in merged:
                merged[key] = list(vals)
                order.append(key)
                continue
            cur = merged[key]
            for i, v in enumerate(vals):
                if v.value is None:
                    continue
                if cur[i].value is None:
                    cur[i] = v
                elif rules[i] == "sum":
                    cur[i] = dataclasses.replace(cur[i], value=cur[i].value + v.value)
                elif rules[i] == "min":
                    cur[i] = cur[i] if cur[i].value <= v.value else v
                elif rules[i] == "max":
                    cur[i] = cur[i] if cur[i].value >= v.value else v
                else:
                    raise ValueError("unknown merge rule %r" % (rules[i],))
    return [(k, merged[k]) for k in order]


def debug_plan(table: HostTable, expr: Optional[Expr], specs: Sequence[AggregateSpec], snapshot: Optional[Snapshot] = None,
               group_by: Sequence[int] = (), expr_mode: Optional[int] = None, cardinality_hint: int = 0, block_threads: int = 0,
               rows_per_thread: int = 0, stages: int = 0, ctas_per_sm: int = 0, jit: bool = False, cubin_path: Optional[str] = None,
               partition: bool = False, tile_list: bool = False, packed: bool = False, continues: bool = False) -> str:
    """llkv_gpu_debug_plan: compiles the plan against the host table's column statistics (no GPU needed) and returns the
    listing of the lean program; with jit=True the lean kernel is also specialised with NVRTC.  continues=True: the step
    form of a run that follows another run without a reset."""
    lib = load()
    cols = []
    host_cols = list(table.columns.values())
    lfids = [logical_field_id(table.table_id, c.field_id) for c in host_cols]
    created = deleted = -1
    if table.created_by is not None and snapshot is not None:
        created, deleted = len(host_cols), len(host_cols) + 1
        host_cols += [table.created_by, table.deleted_by]
        lfids += [logical_field_id(table.table_id, 0xFFFFFFFF, NS_TXN_CREATED_BY), logical_field_id(table.table_id, 0xFFFFFFFE, NS_TXN_DELETED_BY)]
    arr = (ffi.DebugColumn * len(host_cols))()
    for i, (c, lfid) in enumerate(zip(host_cols, lfids)):
        d = arr[i]
        d.nullable = int(c.validity is not None)
        d.logical_field_id = lfid
        d.prim_type = c.dtype.type
        d.precision = c.dtype.precision
        d.scale = c.dtype.scale
        d.n_rows = c.n_rows
        t = c.dtype.type
        if t == ffi.PT_UTF8:
            lens = np.diff(c.values.astype(np.int64))
            d.max_strlen = int(lens.max()) if lens.size else 0
        elif t == ffi.PT_DECIMAL128:
            v = c.values.reshape(-1, 2) if c.values.ndim == 1 else c.values
            lo = v[:, 0].view(np.int64)
            hi = v[:, 1].view(np.int64)
            fits = bool(np.all(hi == (lo >> 63)))
            d.dec_fits_i64 = int(fits)
            if fits and lo.size:
                d.has_minmax, d.min_value, d.max_value = 1, int(lo.min()), int(lo.max())
        elif t in (ffi.PT_FLOAT32, ffi.PT_FLOAT64):
            pass
        elif c.n_rows:
            if t == ffi.PT_UINT64:
                d.has_minmax, d.min_value, d.max_value = 1, int(np.int64(np.uint64(c.values.min()))), int(np.int64(np.uint64(c.values.max())))
            else:
                d.has_minmax, d.min_value, d.max_value = 1, int(c.values.min()), int(c.values.max())
    prog = None
    if expr is not None:
        cp = ProgramCompiler(expr).compile()
        ops, n_ops, lits, n_lits, nodes, n_nodes, roots, n_roots = cp.c_arrays()
        prog = C.c_void_p()
        _check(lib.llkv_gpu_program_compile(None, ops, n_ops, lits, n_lits, nodes, n_nodes, roots, n_roots, C.byref(prog)))
    try:
        if expr_mode is None:
            expr_mode = ffi.EXPR_EXACT if group_by else ffi.EXPR_ARROW
        aggs, n_aggs, anodes, n_anodes = flatten_aggregates(specs)
        keys = (C.c_uint64 * max(1, len(group_by)))(*group_by)
        out = C.create_string_buffer(1 << 16)
        _check(lib.llkv_gpu_debug_plan(arr, len(host_cols), prog, created, deleted, snapshot.txn_id if snapshot else 0,
                                       snapshot.snapshot_id if snapshot else 0, aggs, n_aggs, anodes, n_anodes, keys, len(group_by), expr_mode,
                                       cardinality_hint, block_threads, rows_per_thread, stages, ctas_per_sm, int(jit) | (2 if partition or packed else 0) | (4 if tile_list else 0) | (8 if packed else 0) | (16 if continues else 0),
                                       cubin_path.encode() if cubin_path else None, out, len(out)))
        return out.value.decode()
    finally:
        if prog is not None:
            lib.llkv_gpu_program_destroy(prog)


class DeviceTable:
    """The HBM-resident image of one table: every column concatenated chunk by chunk, dense row ids."""

    def __init__(self, ctx: Context, table_id: int = 1):
        self.ctx = ctx
        self.table_id = table_id
        self.columns: Dict[int, DeviceColumn] = {}
        self.created_by: Optional[DeviceColumn] = None
        self.deleted_by: Optional[DeviceColumn] = None
        self.n_rows = 0

    @staticmethod
    def from_host(ctx: Context, table: HostTable, chunk_rows: Optional[int] = None, as_blob: bool = False) -> "DeviceTable":
        dt = DeviceTable(ctx, table.table_id)
        for col in table.columns.values():
            dt.add_column(col, chunk_rows, as_blob)
        if table.created_by is not None:
            dt.add_mvcc(table.created_by, table.deleted_by, chunk_rows)
        dt.seal()
        return dt

    def add_column(self, col: HostColumn, chunk_rows: Optional[int] = None, as_blob: bool = False) -> DeviceColumn:
        dc = DeviceColumn(self.ctx, logical_field_id(self.table_id, col.field_id), col)
        dc.reserve(col.n_rows)
        dc.append(col, chunk_rows, as_blob=as_blob)
        self.columns[col.field_id] = dc
        self.n_rows = col.n_rows
        return dc

    def add_mvcc(self, created_by: HostColumn, deleted_by: HostColumn, chunk_rows: Optional[int] = None):
        self.created_by = DeviceColumn(self.ctx, logical_field_id(self.table_id, 0xFFFFFFFF, NS_TXN_CREATED_BY), created_by)
        self.created_by.reserve(created_by.n_rows)
        self.created_by.append(created_by, chunk_rows)
        self.deleted_by = DeviceColumn(self.ctx, logical_field_id(self.table_id, 0xFFFFFFFE, NS_TXN_DELETED_BY), deleted_by)
        self.deleted_by.reserve(deleted_by.n_rows)
        self.deleted_by.append(deleted_by, chunk_rows)

    def seal(self):
        for c in self._all():
            c.seal()

    def _all(self) -> List[DeviceColumn]:
        cols = list(self.columns.values())
        if self.created_by is not None:
            cols += [self.created_by, self.deleted_by]
        return cols

    def set_snapshot(self, snapshot: Optional[Snapshot]):
        """MvccRowIdFilter::new(txn_manager, snapshot) (llkv-transaction/src/helpers.rs:259-312)."""
        lib = self.ctx.lib
        if snapshot is None or self.created_by is None:
            _check(lib.llkv_gpu_mvcc_clear(self.ctx.handle, self.table_id))
            return
        nc = list(snapshot.noncommitted)
        arr = (C.c_uint64 * max(1, len(nc)))(*nc)
        _check(lib.llkv_gpu_mvcc_set(self.ctx.handle, self.table_id, self.created_by.handle, self.deleted_by.handle,
                                     snapshot.txn_id, snapshot.snapshot_id, arr, len(nc)))

    def filter_bitmap(self, expr: Optional[Expr], snapshot: Optional[Snapshot] = None, row_begin: int = 0,
                      row_end: Optional[int] = None) -> Tuple[np.ndarray, int]:
        """Selection bitmap over row positions + its popcount (ScanStorage::filter_leaf / RowIdFilter::filter)."""
        row_end = self.n_rows if row_end is None else row_end
        prog = Program(self.ctx, expr) if expr is not None else None
        self.set_snapshot(snapshot)
        n_words = (row_end - row_begin + 63) // 64
        words = np.zeros(max(1, n_words), dtype=np.uint64)
        count = C.c_uint64()
        try:
            _check(self.ctx.lib.llkv_gpu_filter_bitmap(self.ctx.handle, self.table_id, prog.handle if prog else None,
                                                       int(snapshot is not None), row_begin, row_end,
                                                       C.c_void_p(words.ctypes.data), n_words, C.byref(count)))
        finally:
            if prog:
                prog.destroy()
        return words[:n_words], int(count.value)

    def aggregate(self, expr: Optional[Expr], specs: Sequence[AggregateSpec], snapshot: Optional[Snapshot] = None,
                  group_by: Sequence[int] = (), expr_mode: Optional[int] = None, row_begin: int = 0,
                  row_end: Optional[int] = None, cardinality_hint: int = 0, group_capacity: Optional[int] = None):
        """One-shot: new accumulators, one fused scan, finalize.  Same result shape as oracle.aggregate."""
        prog = Program(self.ctx, expr) if expr is not None else None
        self.set_snapshot(snapshot)
        agg = Aggregation(self, specs, group_by, expr_mode, cardinality_hint)
        try:
            agg.run(prog, snapshot is not None, row_begin, row_end)
            return agg.finalize(group_capacity)
        finally:
            agg.destroy()
            if prog:
                prog.destroy()

    def destroy(self):
        for c in self._all():
            c.destroy()
        self.columns.clear()
        self.created_by = self.deleted_by = None

"""ctypes mirror of include/llkv_gpu.h (structs + enums).

Shared by the GPU binding (gpu.py) and by the test-only oracle wrapper (oracle/oracle.py) so both sides
receive byte-identical flattened trees.  Nothing here computes anything.
"""
import ctypes as C

# status codes — llkv_result::Error variant order (llkv-result/src/error.rs:31-176)
OK, ERR_IO, ERR_ARROW, ERR_INVALID_ARGUMENT, ERR_NOT_FOUND = 0, 1, 2, 3, 4
ERR_CATALOG, ERR_CONSTRAINT, ERR_TRANSACTION, ERR_INTERNAL = 5, 6, 7, 8
ERR_EXPR_CAST, ERR_PREDICATE_BUILD, ERR_RESERVED_TABLE_ID = 9, 10, 11
ERROR_NAMES = {
    1: "Io", 2: "Arrow", 3: "InvalidArgumentError", 4: "NotFound", 5: "CatalogError", 6: "ConstraintError",
    7: "TransactionContextError", 8: "Internal", 9: "ExprCast", 10: "PredicateBuild", 11: "ReservedTableId",
}

# PrimType codes (llkv-column-map/src/serialization.rs:146-166)
PT_NULL, PT_UINT64, PT_INT32, PT_UINT32, PT_FLOAT32 = 0, 1, 2, 3, 4
PT_INT64, PT_INT16, PT_INT8, PT_UINT16, PT_UINT8, PT_FLOAT64, PT_UTF8 = 6, 7, 8, 9, 10, 11, 12
PT_BOOLEAN, PT_DATE32, PT_DATE64, PT_DECIMAL128 = 15, 16, 17, 18
PT_WIDTH = {
    PT_UINT64: 8, PT_INT32: 4, PT_UINT32: 4, PT_FLOAT32: 4, PT_INT64: 8, PT_INT16: 2, PT_INT8: 1, PT_UINT16: 2,
    PT_UINT8: 1, PT_FLOAT64: 8, PT_BOOLEAN: 1, PT_DATE32: 4, PT_DATE64: 8, PT_DECIMAL128: 16,
}

LIT_NULL, LIT_INT128, LIT_FLOAT64, LIT_DECIMAL128, LIT_STRING, LIT_BOOLEAN, LIT_DATE32 = range(7)
SE_COLUMN, SE_LITERAL, SE_BINARY, SE_NOT, SE_IS_NULL, SE_CAST, SE_COMPARE, SE_COALESCE = 0, 1, 2, 3, 4, 7, 8, 9
BIN_ADD, BIN_SUB, BIN_MUL, BIN_DIV, BIN_MOD, BIN_AND, BIN_OR, BIN_SHL, BIN_SHR = range(9)
CMP_EQ, CMP_NE, CMP_LT, CMP_LE, CMP_GT, CMP_GE = range(6)
EV_PUSH_PREDICATE, EV_PUSH_COMPARE, EV_PUSH_IN_LIST, EV_PUSH_IS_NULL, EV_PUSH_LITERAL = 0, 1, 2, 3, 4
EV_FUSED_AND, EV_AND, EV_OR, EV_NOT, EV_FILTER_ITEM = 5, 6, 7, 8, 100
OP_EQUALS, OP_RANGE, OP_GT, OP_GTE, OP_LT, OP_LTE, OP_IN = range(7)
OP_STARTS_WITH, OP_ENDS_WITH, OP_CONTAINS, OP_IS_NULL, OP_IS_NOT_NULL = 7, 8, 9, 10, 11
BOUND_INCLUDED, BOUND_EXCLUDED, BOUND_UNBOUNDED = 0, 1, 2
AGG_COUNT, AGG_SUM, AGG_TOTAL, AGG_AVG, AGG_MIN, AGG_MAX, AGG_COUNT_NULLS = range(7)
EXPR_ARROW, EXPR_EXACT = 0, 1
UNIQUE_ID_BYTES = 128


class Literal(C.Structure):
    _fields_ = [("kind", C.c_int32), ("precision", C.c_uint8), ("scale", C.c_int8), ("_pad", C.c_uint8 * 2),
                ("lo", C.c_uint64), ("hi", C.c_uint64)]


class ScalarNode(C.Structure):
    _fields_ = [("tag", C.c_int32), ("op", C.c_int32), ("left", C.c_int32), ("right", C.c_int32),
                ("field_id", C.c_uint64), ("literal", Literal), ("cast_type", C.c_int32),
                ("cast_precision", C.c_uint8), ("cast_scale", C.c_int8), ("_pad", C.c_uint8 * 2)]


class EvalOp(C.Structure):
    _fields_ = [("tag", C.c_int32), ("operator_tag", C.c_int32), ("field_id", C.c_uint64),
                ("lower_kind", C.c_int32), ("upper_kind", C.c_int32), ("lit_begin", C.c_int32),
                ("lit_count", C.c_int32), ("expr_left", C.c_int32), ("expr_right", C.c_int32),
                ("cmp_op", C.c_int32), ("negated", C.c_int32), ("child_count", C.c_int32),
                ("literal_bool", C.c_int32)]


class AggSpec(C.Structure):
    _fields_ = [("kind", C.c_int32), ("expr_root", C.c_int32), ("data_type", C.c_int32),
                ("precision", C.c_uint8), ("scale", C.c_int8), ("distinct", C.c_uint8), ("_pad", C.c_uint8)]


class HavingTerm(C.Structure):
    _fields_ = [("is_aggregate", C.c_int32), ("index", C.c_int32), ("cmp_op", C.c_int32), ("_pad", C.c_int32), ("literal", Literal)]


class OrderKey(C.Structure):
    _fields_ = [("is_aggregate", C.c_int32), ("index", C.c_int32), ("descending", C.c_int32), ("nulls_first", C.c_int32)]


class AggValue(C.Structure):
    _fields_ = [("lo", C.c_uint64), ("hi", C.c_uint64), ("type", C.c_int32), ("precision", C.c_uint8),
                ("scale", C.c_int8), ("valid", C.c_uint8), ("_pad", C.c_uint8)]


class GroupKey(C.Structure):
    _fields_ = [("bits", C.c_uint64), ("type", C.c_int32), ("valid", C.c_uint8), ("dict", C.c_uint8),
                ("_pad", C.c_uint8 * 2)]


class ScanOptions(C.Structure):
    """llkv_scan_options = ScanOptions (llkv-column-map/src/store/scan/options.rs:13-37)."""
    _fields_ = [("sorted", C.c_int32), ("reverse", C.c_int32), ("with_row_ids", C.c_int32), ("include_nulls", C.c_int32),
                ("nulls_first", C.c_int32), ("has_lower", C.c_int32), ("lower_inclusive", C.c_int32), ("has_upper", C.c_int32),
                ("upper_inclusive", C.c_int32), ("_pad", C.c_int32), ("lower_bits", C.c_uint64), ("upper_bits", C.c_uint64),
                ("offset", C.c_uint64), ("limit", C.c_uint64)]


class RunInfo(C.Structure):
    _fields_ = [("rows", C.c_uint64), ("kernel_launches", C.c_uint32), ("used_wide_path", C.c_uint32),
                ("algorithmic_bytes_per_row", C.c_uint32), ("physical_bytes_per_row", C.c_uint32),
                ("grid", C.c_uint32), ("block", C.c_uint32), ("rows_per_tile", C.c_uint32), ("stages", C.c_uint32),
                ("smem_bytes", C.c_uint32), ("fast_groups", C.c_uint32), ("last_kernel_ms", C.c_float),
                ("used_fast_kernel", C.c_uint32), ("used_jit_kernel", C.c_uint32), ("partitions", C.c_uint32), ("tiles_pruned", C.c_uint32),
                ("graph_replays", C.c_uint32), ("merged_p2p", C.c_uint32), ("last_merge_ms", C.c_float), ("packed_tuples", C.c_uint32),
                ("published_steps", C.c_uint32)]


class DebugColumn(C.Structure):
    _fields_ = [("logical_field_id", C.c_uint64), ("prim_type", C.c_int32), ("precision", C.c_uint8), ("scale", C.c_int8),
                ("has_minmax", C.c_uint8), ("dec_fits_i64", C.c_uint8), ("min_value", C.c_int64), ("max_value", C.c_int64),
                ("n_rows", C.c_uint64), ("max_strlen", C.c_uint8), ("nullable", C.c_uint8), ("_pad", C.c_uint8 * 6)]


def i128_to_words(v: int):
    v &= (1 << 128) - 1
    return v & 0xFFFFFFFFFFFFFFFF, v >> 64


def words_to_i128(lo: int, hi: int) -> int:
    v = (hi << 64) | lo
    return v - (1 << 128) if v >> 127 else v

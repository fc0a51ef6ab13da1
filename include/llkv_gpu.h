/*
 * llkv_gpu.h — C ABI of the B200-native scan -> filter -> MVCC -> aggregate path for LLKV.
 *
 * This header is the drop-in boundary (SURVEY.md §8b).  Every entry point is
 * `extern "C"`, takes plain pointers and sizes, and replaces one reference
 * interface, cited as `crate/path.rs:line` relative to jzombie/rust-llkv
 * v0.8.5-alpha.  A Rust `-sys` crate binds these 1:1 (see INTEGRATION.md and
 * ffi/llkv-gpu-sys/src/lib.rs; authored, the image has no Rust toolchain); the
 * same symbols are driven from Python ctypes (`rust-llkv_b200/llkv_b200/gpu.py`),
 * the host-side mirror of the reference's types that the tests use.
 *
 * Conventions
 *   - Every call returns an `int32_t` status.  0 is success; non-zero values
 *     follow the variant order of `llkv_result::Error`
 *     (llkv-result/src/error.rs:31-176).  The message for the last failing
 *     call on the calling thread is read with `llkv_gpu_last_error`.
 *   - The caller owns every host buffer; the library owns all device memory
 *     behind opaque handles.  Handles may move between threads, but calls on
 *     one handle must be serialised by the caller (mirrors `&mut self`).
 *     Columns, programs and aggregates are children of their context and
 *     share its state (column registry, staging ring, stream, snapshots):
 *     the library serialises calls that touch one context with a lock inside
 *     the context, so different handles of one context may be used from
 *     different threads.  A child handle must not outlive its context.
 *   - There is no CPU fallback.  Without a usable CUDA device
 *     `llkv_gpu_ctx_create` fails with LLKV_ERR_IO and nothing else works.
 */
#ifndef LLKV_GPU_H
#define LLKV_GPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LLKV_GPU_ABI_VERSION 1

/* ---- status codes: llkv_result::Error variant order (llkv-result/src/error.rs:31-176) ---- */
enum {
  LLKV_OK = 0,
  LLKV_ERR_IO = 1,               /* Error::Io — also "no CUDA device / CUDA runtime failure" */
  LLKV_ERR_ARROW = 2,            /* Error::Arrow — arithmetic overflow raised by arrow-arith kernels */
  LLKV_ERR_INVALID_ARGUMENT = 3, /* Error::InvalidArgumentError — e.g. "integer overflow" from SumInt64 */
  LLKV_ERR_NOT_FOUND = 4,        /* Error::NotFound */
  LLKV_ERR_CATALOG = 5,
  LLKV_ERR_CONSTRAINT = 6,
  LLKV_ERR_TRANSACTION = 7,
  LLKV_ERR_INTERNAL = 8,         /* Error::Internal */
  LLKV_ERR_EXPR_CAST = 9,        /* Error::ExprCast */
  LLKV_ERR_PREDICATE_BUILD = 10, /* Error::PredicateBuild — literal cast / unsupported operator */
  LLKV_ERR_RESERVED_TABLE_ID = 11
};

/* ---- column element types: on-disk PrimType codes (llkv-column-map/src/serialization.rs:146-166) ---- */
enum {
  LLKV_PT_NULL = 0, /* DataType::Null (only as an expression type) */
  LLKV_PT_UINT64 = 1,
  LLKV_PT_INT32 = 2,
  LLKV_PT_UINT32 = 3,
  LLKV_PT_FLOAT32 = 4,
  LLKV_PT_INT64 = 6,
  LLKV_PT_INT16 = 7,
  LLKV_PT_INT8 = 8,
  LLKV_PT_UINT16 = 9,
  LLKV_PT_UINT8 = 10,
  LLKV_PT_FLOAT64 = 11,
  LLKV_PT_UTF8 = 12,     /* typed predicates and GROUP BY keys; <= 7 bytes as packed keys, longer ones dictionary-coded
                            (see "Utf8 columns" below) */
  LLKV_PT_BOOLEAN = 15,  /* one byte per value at this boundary (0/1) */
  LLKV_PT_DATE32 = 16,
  LLKV_PT_DATE64 = 17,
  LLKV_PT_DECIMAL128 = 18
};

/* ---- llkv_types::Literal (llkv-types/src/literal.rs:26-41), variant order ---- */
enum {
  LLKV_LIT_NULL = 0,
  LLKV_LIT_INT128 = 1,     /* lo/hi = two's complement i128 */
  LLKV_LIT_FLOAT64 = 2,    /* lo = IEEE-754 bits */
  LLKV_LIT_DECIMAL128 = 3, /* lo/hi = raw i128, scale = DecimalValue::scale */
  LLKV_LIT_STRING = 4,     /* precision = byte length (<= 15), bytes little-endian in lo/hi; or precision = 255
                              (LLKV_LIT_STRING_BY_REF): lo = address of the bytes, hi = byte length — the call that
                              receives the literal copies the bytes before it returns */
  LLKV_LIT_BOOLEAN = 5,    /* lo = 0/1 */
  LLKV_LIT_DATE32 = 6      /* lo = sign-extended days since epoch */
};

#define LLKV_LIT_STRING_BY_REF 255
typedef struct llkv_literal {
  int32_t kind;
  uint8_t precision; /* Decimal128: informational; String: length */
  int8_t scale;
  uint8_t _pad[2];
  uint64_t lo;
  uint64_t hi;
} llkv_literal;

/* ---- llkv_expr::ScalarExpr (llkv-expr/src/expr.rs:127-182), flattened, children before parents ---- */
enum {
  LLKV_SE_COLUMN = 0,
  LLKV_SE_LITERAL = 1,
  LLKV_SE_BINARY = 2,
  LLKV_SE_NOT = 3,
  LLKV_SE_IS_NULL = 4,
  LLKV_SE_CAST = 7,
  LLKV_SE_COMPARE = 8,
  LLKV_SE_COALESCE = 9
};
/* llkv_expr::BinaryOp (expr.rs:311-321) */
enum { LLKV_BIN_ADD = 0, LLKV_BIN_SUB = 1, LLKV_BIN_MUL = 2, LLKV_BIN_DIV = 3, LLKV_BIN_MOD = 4,
       LLKV_BIN_AND = 5, LLKV_BIN_OR = 6, LLKV_BIN_SHL = 7, LLKV_BIN_SHR = 8 };
/* llkv_expr::CompareOp (expr.rs:342-349) */
enum { LLKV_CMP_EQ = 0, LLKV_CMP_NE = 1, LLKV_CMP_LT = 2, LLKV_CMP_LE = 3, LLKV_CMP_GT = 4, LLKV_CMP_GE = 5 };

typedef struct llkv_scalar_node {
  int32_t tag;       /* LLKV_SE_* */
  int32_t op;        /* BINARY: LLKV_BIN_*; COMPARE: LLKV_CMP_*; IS_NULL: negated flag */
  int32_t left;      /* child node index or -1 */
  int32_t right;     /* child node index or -1 */
  uint64_t field_id; /* COLUMN: LogicalFieldId as u64 (llkv-types/src/ids.rs:133-152) */
  llkv_literal literal;
  int32_t cast_type; /* CAST: LLKV_PT_* */
  uint8_t cast_precision;
  int8_t cast_scale;
  uint8_t _pad[2];
} llkv_scalar_node;

/* ---- llkv_compute::program::EvalOp (llkv-compute/src/program.rs:48-78), postfix ---- */
enum {
  LLKV_EV_PUSH_PREDICATE = 0,
  LLKV_EV_PUSH_COMPARE = 1,
  LLKV_EV_PUSH_IN_LIST = 2,
  LLKV_EV_PUSH_IS_NULL = 3,
  LLKV_EV_PUSH_LITERAL = 4,
  LLKV_EV_FUSED_AND = 5, /* followed by child_count LLKV_EV_FILTER_ITEM entries */
  LLKV_EV_AND = 6,
  LLKV_EV_OR = 7,
  LLKV_EV_NOT = 8,
  LLKV_EV_FILTER_ITEM = 100
};
/* OwnedOperator (program.rs:87-112) */
enum {
  LLKV_OP_EQUALS = 0,
  LLKV_OP_RANGE = 1,
  LLKV_OP_GT = 2,
  LLKV_OP_GTE = 3,
  LLKV_OP_LT = 4,
  LLKV_OP_LTE = 5,
  LLKV_OP_IN = 6,
  LLKV_OP_STARTS_WITH = 7, /* Utf8 columns; one string literal (the pattern); llkv_eval_op.literal_bool = 1 asks for the */
  LLKV_OP_ENDS_WITH = 8,   /* case-insensitive form (typed_predicate.rs:187-209: both sides through to_lowercase()), which this  */
  LLKV_OP_CONTAINS = 9,    /* path serves for ASCII patterns over columns without non-ASCII bytes, else LLKV_ERR_PREDICATE_BUILD */
  LLKV_OP_IS_NULL = 10,
  LLKV_OP_IS_NOT_NULL = 11
};
/* std::ops::Bound */
enum { LLKV_BOUND_INCLUDED = 0, LLKV_BOUND_EXCLUDED = 1, LLKV_BOUND_UNBOUNDED = 2 };

typedef struct llkv_eval_op {
  int32_t tag;          /* LLKV_EV_* */
  int32_t operator_tag; /* PUSH_PREDICATE / FILTER_ITEM: LLKV_OP_* */
  uint64_t field_id;    /* PUSH_PREDICATE / FUSED_AND / FILTER_ITEM */
  int32_t lower_kind;   /* RANGE: LLKV_BOUND_* */
  int32_t upper_kind;
  int32_t lit_begin;    /* first literal in literals[]; RANGE: lower (if bounded) then upper (if bounded); IN: the list */
  int32_t lit_count;
  int32_t expr_left;    /* PUSH_COMPARE: lhs root; PUSH_IN_LIST / PUSH_IS_NULL: operand root (index into nodes[]) */
  int32_t expr_right;   /* PUSH_COMPARE: rhs root; PUSH_IN_LIST: first entry in list_roots[] */
  int32_t cmp_op;       /* PUSH_COMPARE: LLKV_CMP_* */
  int32_t negated;      /* PUSH_IN_LIST / PUSH_IS_NULL */
  int32_t child_count;  /* AND / OR / FUSED_AND; PUSH_IN_LIST: list length */
  int32_t literal_bool; /* PUSH_LITERAL; STARTS_WITH / ENDS_WITH / CONTAINS leaves: 1 = case-insensitive */
} llkv_eval_op;

/* ---- llkv_aggregate::AggregateKind (llkv-aggregate/src/lib.rs:32-69) ---- */
enum {
  LLKV_AGG_COUNT = 0,       /* expr_root < 0 => COUNT(*) (CountStar), else CountColumn */
  LLKV_AGG_SUM = 1,
  LLKV_AGG_TOTAL = 2,
  LLKV_AGG_AVG = 3,
  LLKV_AGG_MIN = 4,
  LLKV_AGG_MAX = 5,
  LLKV_AGG_COUNT_NULLS = 6
};

typedef struct llkv_agg_spec {
  int32_t kind;      /* LLKV_AGG_* */
  int32_t expr_root; /* argument expression root in nodes[], -1 for COUNT(*) */
  int32_t data_type; /* AggregateKind::*.data_type as LLKV_PT_* — selects the accumulator (lib.rs:463-748) */
  uint8_t precision;
  int8_t scale;
  uint8_t distinct;  /* DISTINCT (llkv-aggregate/src/lib.rs:103-204): ungrouped COUNT / SUM / TOTAL / AVG over one bare integer column,
                        and then every aggregate of the query must be DISTINCT over that column; otherwise 0 */
  uint8_t _pad;
} llkv_agg_spec;

/* How scalar expressions that feed aggregates are typed and rounded (SURVEY.md §8a notes D1/D2). */
enum {
  LLKV_EXPR_ARROW = 0, /* ungrouped path: arrow-arith kernels + cast to the inferred type
                          (llkv-compute/src/eval.rs:565-614, kernels.rs:99-177) */
  LLKV_EXPR_EXACT = 1  /* GROUP BY path: exact DecimalValue ops per row
                          (llkv-executor/src/lib.rs:7229-7332, llkv-compute/src/scalar/decimal.rs:128-170) */
};

/* One finalized aggregate cell: what AggregateAccumulator::finalize puts in its 1-row array (lib.rs:1488-1939). */
typedef struct llkv_agg_value {
  uint64_t lo;       /* Int64 / f64 bits / low half of i128 */
  uint64_t hi;       /* high half of i128 (Decimal128) */
  int32_t type;      /* LLKV_PT_INT64 / LLKV_PT_FLOAT64 / LLKV_PT_DECIMAL128 / ... */
  uint8_t precision;
  int8_t scale;
  uint8_t valid;     /* 0 => NULL */
  uint8_t _pad;
} llkv_agg_value;

/* One GROUP BY key cell (llkv-executor/src/lib.rs:99-106 GroupKeyValue). */
typedef struct llkv_group_key {
  uint64_t bits;  /* Int: i64; Bool: 0/1; String: bytes big-endian from the top byte, length in the low byte — or, when
                     `dict` = 1, the string's code in the key column's dictionary (llkv_gpu_column_dict_entry) */
  int32_t type;   /* LLKV_PT_* of the key column */
  uint8_t valid;  /* 0 => NULL key (its own group) */
  uint8_t dict;   /* Utf8 keys of a column that holds strings longer than 7 bytes: 1 = `bits` is a dictionary code
                     (2 is used by the test oracle only: `bits` is the position of a row holding the string) */
  uint8_t _pad[2];
} llkv_group_key;

/* Facts about the most recent llkv_gpu_agg_run / llkv_gpu_filter_bitmap on a handle (for bench.py and ncu notes). */
typedef struct llkv_run_info {
  uint64_t rows;                /* rows scanned */
  uint32_t kernel_launches;     /* CUDA kernels launched by the call */
  uint32_t used_wide_path;      /* 1 when the 128-bit interpreter ran (narrow path overflowed or not applicable) */
  uint32_t algorithmic_bytes_per_row; /* sum of Arrow value widths of the columns read (SURVEY.md §8d) */
  uint32_t physical_bytes_per_row;    /* bytes per row the kernels read from HBM */
  uint32_t grid, block, rows_per_tile, stages, smem_bytes;
  uint32_t fast_groups;         /* CTA-local group slots with per-thread accumulators */
  float last_kernel_ms;         /* device time of the scan kernel (CUDA events) when timing is enabled, else 0 */
  uint32_t used_fast_kernel;    /* 1 when the lean kernel (lean_kernel.cuh) ran, 0 for the general interpreter */
  uint32_t used_jit_kernel;     /* 1 when the lean kernel ran as a build specialised on this plan shape (jit.cpp) */
  uint32_t partitions;          /* hash partitions of a partitioned high-cardinality GROUP BY run, 0 = not partitioned */
  uint32_t tiles_pruned;        /* tiles the scan skipped because no conjunct range predicate can match their zones */
  uint32_t graph_replays;       /* steps of this aggregate that llkv_gpu_agg_execute replayed from its captured CUDA graph */
  uint32_t merged_p2p;          /* 1 when the last merge was one kernel over NVLink peer mailboxes (no collective, no host wait) */
  float last_merge_ms;          /* device time of that merge kernel, waiting for the slowest peer included (timing enabled) */
  uint32_t packed_tuples;       /* partitioned run in its packed form (64-bit tuples, partitions aggregated in shared memory):
                                   1 = partitions are hash ranges, 2 = key ranges (dense integer keys); 0 = first form / not partitioned */
  uint32_t published_steps;     /* steps of this aggregate whose scan published the result to page-locked memory and re-armed
                                   the state (a repeated step that is one kernel), replays included */
} llkv_run_info;

typedef struct llkv_gpu_ctx llkv_gpu_ctx;
typedef struct llkv_gpu_column llkv_gpu_column;
typedef struct llkv_gpu_program llkv_gpu_program;
typedef struct llkv_gpu_agg llkv_gpu_agg;

/* ---- library / context ---- */
int32_t llkv_gpu_abi_version(void);
/* Copies the calling thread's last error message (NUL terminated) and returns its full length. */
size_t llkv_gpu_last_error(char* buf, size_t cap);
/* Number of CUDA devices, or 0.  Never fails. */
int32_t llkv_gpu_device_count(void);

/* One context per GPU.  `n_streams` copy streams feed the pinned staging ring of `pinned_bytes`
 * bytes that stands where `Pager::batch_get` hands out blobs (llkv-storage/src/pager/mod.rs:89-104). */
int32_t llkv_gpu_ctx_create(int32_t device_ordinal, int32_t n_streams, uint64_t pinned_bytes, llkv_gpu_ctx** out);
void llkv_gpu_ctx_destroy(llkv_gpu_ctx* ctx);
int32_t llkv_gpu_ctx_synchronize(llkv_gpu_ctx* ctx);
/* The cudaStream_t the scan kernels are launched on (for CUDA-event timing by the caller). */
int32_t llkv_gpu_ctx_stream(llkv_gpu_ctx* ctx, void** out_stream);
/* Turns per-run CUDA-event timing of the scan kernel on/off (llkv_run_info.last_kernel_ms). */
int32_t llkv_gpu_ctx_set_timing(llkv_gpu_ctx* ctx, int32_t enabled);
/* Tuning knobs: 0 keeps the default.  rows_per_thread in {1,2,4,8} (8: lean kernel only).  force_wide: 1 = always the 128-bit general
 * interpreter, 2 = always the 64-bit general interpreter (never the lean kernel). */
int32_t llkv_gpu_ctx_set_tuning(llkv_gpu_ctx* ctx, int32_t ctas_per_sm, int32_t block_threads, int32_t stages,
                                int32_t rows_per_thread, int32_t force_wide);

/* Run-time specialisation of the lean kernel on a plan shape (program + layout), compiled with NVRTC and cached per
 * device: 0 = never (always interpret the lowered program), 1 = from the second run of a shape on (default), 2 = from
 * the first run.  Literals, row ranges and snapshots are run-time parameters of the specialised kernel.  Without NVRTC
 * on the machine the lean kernel keeps interpreting on the GPU. */
int32_t llkv_gpu_ctx_set_jit(llkv_gpu_ctx* ctx, int32_t mode);

/* High-cardinality GROUP BY (cardinality_hint > 128; the reference's hash-map GROUP BY, llkv-executor/src/lib.rs:
 * 5028-5355) updates the global open-addressing table once per row.  When the table is much larger than L2 that is one
 * random DRAM sector read-modify-write per row and word; the partitioned form writes (key, row id, operands) tuples into
 * hash partitions whose table slice fits in L2 and folds them partition by partition (two streaming passes instead of
 * random access).  When the keys, a launch-relative row number and the SUM operands of a row fit one 64-bit word the tuples
 * are packed, the partitions are made small enough (a few thousand groups) for one CTA to aggregate a whole partition in
 * shared memory, and every group is written to the table once per launch.  mode: 0 = never, 1 = when the table exceeds L2
 * and the scan is long enough (default), 2 = whenever the plan allows it (tests), 3 = as 2 but never the packed form
 * (tests).  Results are identical in every mode.  Needs the specialised kernel (jit mode != 0). */
int32_t llkv_gpu_ctx_set_partitioning(llkv_gpu_ctx* ctx, int32_t mode);

/* Zone-map pruning on the device-resident image — the chunk skip of the reference's scans (ChunkMetadata min/max against
 * the predicate range, llkv-column-map/src/store/pruning.rs:104-258, scan/unsorted.rs:222-227) at a granularity of 4096
 * rows, with Decimal128 columns included (the reference keeps no statistics for them, store/core.rs:1029-1032).  Minima /
 * maxima per zone are computed on the device the first time they are wanted; a fused scan whose filter is a conjunction
 * containing range predicates then visits only the tiles whose zones can match.  mode: 0 = never, 1 = for columns scanned
 * again without having changed, when at least 1/8 of the tiles drop out (default), 2 = from the first scan, whenever any
 * tile drops out (tests).  Results are identical in every mode. */
int32_t llkv_gpu_ctx_set_pruning(llkv_gpu_ctx* ctx, int32_t mode);

/* Page-locked host memory so chunk uploads DMA straight from the caller's buffer.
 *
 * LIFETIME OF PAGE-LOCKED SOURCES.  When the `values` / `blob` / `aux` / `validity` buffer of an append is page-locked
 * (llkv_gpu_host_alloc, llkv_gpu_host_register), the library reads it AFTER the append returns: consecutive chunks are
 * coalesced into larger DMA transfers and Decimal128 chunks are narrowed by host workers in the background.  Such a
 * buffer must stay valid and unmodified until llkv_gpu_column_flush or llkv_gpu_column_seal of that column has
 * returned.  llkv_gpu_host_free and llkv_gpu_host_unregister first issue and wait for every pending copy of every
 * context, so releasing the memory through them is always safe.  Pageable sources are copied before the append returns. */
int32_t llkv_gpu_host_alloc(uint64_t bytes, void** out);
int32_t llkv_gpu_host_free(void* p);
/* Host worker threads that narrow Decimal128 chunks arriving from page-locked memory to 8 or 4 bytes per value before the
 * DMA, as long as every value of the column is a sign-extended i64 / i32 (a chunk that does not fit sends the column back
 * to the Arrow layout, nothing is lost): half or a quarter of the bytes cross PCIe and the device skips its own narrowing
 * pass at seal.  -1 = default (min(32, hardware threads - 1)), 0 = off (16-byte DMA, narrowed on the device at seal). */
int32_t llkv_gpu_ctx_set_upload_threads(llkv_gpu_ctx* ctx, int32_t n_threads);
/* Hybrid upload: `percent` of a Decimal128 column's Arrow bytes (in 8 MiB blocks) cross the link as they lie, issued by a
 * thread of the pool, and are narrowed and checked by a kernel on the device, while the workers narrow the rest before
 * their DMA.  Both ways read the same host memory, which is the limit they share: the copy engine helps when there are
 * few workers (8 workers: 56 ms -> 48 ms per 2.9 GB) and not when the workers alone saturate the host (15 workers:
 * 37 ms either way).  -1 = default: what the workers leave of the host's streaming budget (0 from 12 workers up);
 * 0 = workers only; 100 = copy engine only. */
int32_t llkv_gpu_ctx_set_dma_share(llkv_gpu_ctx* ctx, int32_t percent);
/* Page-locks memory the caller already owns — the pager's mmap-backed blobs (EntryHandle, llkv-storage/src/pager/
 * simd_r_drive_pager.rs; SURVEY.md §8f rank 3) — so llkv_gpu_column_append_blob / _append_chunk DMA straight out of it
 * instead of staging through the context's pinned ring.  Read-only mappings are registered read-only.  Unregister before
 * the mapping goes away. */
int32_t llkv_gpu_host_register(const void* p, uint64_t bytes);
int32_t llkv_gpu_host_unregister(const void* p);

/* ---- column metadata in front of the scan (host only, no device work): the descriptor walk of
 * llkv-column-map/src/store/scan/unsorted.rs:202-241.  The caller fetches the blobs (ColumnCatalog -> descriptor pk ->
 * page chain, one Pager::batch_get per page, llkv-column-map/src/store/descriptor.rs:380-444), these entries read them;
 * the chunk pks they return are what the caller then fetches in one batched get and hands to
 * llkv_gpu_column_append_blob. ---- */

/* ChunkMetadata (llkv-column-map/src/store/descriptor.rs:23-32): 64 bytes little endian on disk. */
typedef struct llkv_chunk_metadata {
  uint64_t chunk_pk;
  uint64_t value_order_perm_pk; /* 0 = none */
  uint64_t row_count;
  uint64_t serialized_bytes;
  uint64_t min_val_u64; /* order-preserving u64 image of the chunk's minimum (llkv_gpu_sortable_u64) */
  uint64_t max_val_u64;
  uint64_t null_count;
  uint64_t distinct_count;
} llkv_chunk_metadata;

/* ColumnDescriptor (descriptor.rs:87-98; from_le_bytes :263-299).  The index metadata bytes follow the fixed part in
 * the blob at offset 52 (index_meta_len of them). */
typedef struct llkv_column_descriptor {
  uint64_t field_id; /* LogicalFieldId as u64 */
  uint64_t head_page_pk;
  uint64_t tail_page_pk;
  uint64_t total_row_count;
  uint64_t total_chunk_count;
  uint32_t data_type_code; /* 0 = unknown (older files) */
  uint32_t index_meta_len;
} llkv_column_descriptor;

int32_t llkv_gpu_descriptor_parse(const void* bytes, uint64_t len, llkv_column_descriptor* out);

/* One descriptor page: DescriptorPageHeader {next_page_pk u64, entry_count u32, 4 bytes padding} followed by
 * entry_count packed ChunkMetadata (descriptor.rs:344-378).  *next_page_pk == 0 ends the chain.  LLKV_ERR_IO when the
 * blob is shorter than its header says (a truncated page), LLKV_ERR_INVALID_ARGUMENT when `capacity` is too small
 * (*n_entries then holds the count; a page holds at most 256 entries, store/constants.rs:14). */
int32_t llkv_gpu_descriptor_page_parse(const void* bytes, uint64_t len, uint64_t* next_page_pk, llkv_chunk_metadata* out,
                                       uint64_t capacity, uint64_t* n_entries);

/* Order-preserving u64 image of a value given as raw bits in the low bytes (llkv-column-map/src/codecs.rs:33-65:
 * signed integers and dates flip the sign bit of their own width, floats use the sign-flip trick (Float32 through f64),
 * unsigned integers are themselves). */
uint64_t llkv_gpu_sortable_u64(int32_t prim_type, uint64_t value_bits);

typedef struct llkv_range_bound {
  int32_t kind;        /* LLKV_BOUND_* (std::ops::Bound; the same codes as llkv_eval_op ranges) */
  int32_t _pad;
  uint64_t value_bits; /* raw bits of the bound in the column's type */
} llkv_range_bound;

/* IntRanges::matches for the range of one type (llkv-column-map/src/store/pruning.rs:104-258): 1 when a chunk whose
 * metadata says [chunk_min_u64, chunk_max_u64] may hold rows inside (lower, upper), 0 when it cannot (the scan skips
 * the chunk).  NULL bounds mean Unbounded. */
int32_t llkv_gpu_chunk_overlaps(int32_t prim_type, uint64_t chunk_min_u64, uint64_t chunk_max_u64, const llkv_range_bound* lower,
                                const llkv_range_bound* upper);

/* compute_chunk_stats (llkv-column-map/src/store/pruning.rs:272-470) for one chunk of a primitive column: fills
 * min_val_u64 / max_val_u64 (sortable images), null_count and distinct_count of `out` (the other fields are left alone).
 * `validity` is an optional Arrow bitmap (LSB first), NULL = all valid.  An empty chunk is LLKV_ERR_NOT_FOUND (the
 * reference returns None); a chunk of NULLs only has zero statistics; float chunks skip NaN as a bound (strict < / >
 * from +-infinity) and count distinct bit patterns.  Host only: the append path's bookkeeping, for wrappers that write
 * ChunkMetadata themselves. */
int32_t llkv_gpu_chunk_stats(int32_t prim_type, const void* values, uint64_t n_rows, const uint8_t* validity, llkv_chunk_metadata* out);

/* ---- columns: ColumnStore::append / scan source (llkv-column-map/src/store/core.rs:787, scan/mod.rs:191) ---- */
int32_t llkv_gpu_column_register(llkv_gpu_ctx* ctx, uint64_t logical_field_id, int32_t prim_type, uint8_t precision,
                                 int8_t scale, llkv_gpu_column** out);
/* Optional capacity hint (rows). */
int32_t llkv_gpu_column_reserve(llkv_gpu_column* col, uint64_t n_rows);
/* Appends one chunk.  `values` is the Arrow values buffer (pager blob + 24, serialization.rs:41-53).
 * `validity` is an optional Arrow validity bitmap (LSB first) for the chunk; NULL = all valid (the
 * reference's chunk format stores no nulls, serialization.rs:265-269).  `row_ids` is the chunk's
 * row-id shadow column or NULL for the dense run starting at `row_id_base`.  Row ids that do not continue the column
 * densely (rows appended after deletes, updates, columns that skip the rows where they are NULL) make the column
 * row-id sparse: a row lands at position row id - the column's first row id (name the table's first row id in
 * `row_id_base` with a first chunk of scattered ids), its validity bit is set, a row the chunk marks NULL is not written,
 * and a row id written again takes the later chunk's value (last writer wins).  Row ids within one chunk must be distinct.
 * For LLKV_PT_UTF8 `values` is the i32 offsets buffer (n_rows+1) and `aux` the data bytes, for dense and sparse chunks
 * alike (see "Utf8 columns" below).
 * `values` may also point into device memory of the context's GPU (fixed-width types): the chunk is then copied device to
 * device in stream order, and the page-locked lifetime rule above applies to it. */
int32_t llkv_gpu_column_append_chunk(llkv_gpu_column* col, uint64_t chunk_pk, const void* values, uint64_t n_rows,
                                     const uint8_t* validity, const uint64_t* row_ids, uint64_t row_id_base,
                                     const void* aux);
/* Appends a serialized chunk blob exactly as the pager stores it ("ARR0" header, serialization.rs:41-53,264-307). */
int32_t llkv_gpu_column_append_blob(llkv_gpu_column* col, uint64_t chunk_pk, const void* blob, uint64_t blob_len,
                                    const uint64_t* row_ids, uint64_t row_id_base);
/* Issues and waits for every copy the column's appends left pending; afterwards page-locked sources may be reused.
 * (The column stays open for more chunks; llkv_gpu_column_seal implies a flush.) */
int32_t llkv_gpu_column_flush(llkv_gpu_column* col);
/* Waits for outstanding uploads of this column; after this the column is scannable. */
int32_t llkv_gpu_column_seal(llkv_gpu_column* col);
/* ColumnStore::delete_rows (llkv-column-map/src/store/core.rs:1392-1776): the rows leave the column (ids it does not hold
 * are ignored); their positions stay as gaps. */
int32_t llkv_gpu_column_delete_rows(llkv_gpu_column* col, const uint64_t* row_ids, uint64_t n);
/* ColumnStore::gather_rows / gather_row_window under GatherNullPolicy::IncludeNulls (llkv-column-map/src/store/projection.rs:
 * 41-48,929-1352): the values of `row_ids` in request order, Arrow values layout; out_valid[i] = 0 where the column holds no
 * such row (the value is then zero).  For tests and B2-level callers; aggregates never gather.  Not for Utf8. */
int32_t llkv_gpu_column_gather(llkv_gpu_column* col, const uint64_t* row_ids, uint64_t n, void* out_values, uint64_t out_bytes,
                               uint8_t* out_valid);
/* Utf8 columns.  Strings of up to 7 bytes are resident as packed 8-byte keys.  A column that receives a longer string
 * becomes dictionary-coded: the host side of append_chunk interns every string (the bytes of such a column never cross
 * PCIe: 8 bytes per row do), `seal` orders the dictionary byte-wise (Rust's str: Ord) and the resident codes become ranks,
 * so equality, IN, ranges and prefixes are integer leaves on the specialised kernel, suffix / substring / case-insensitive
 * patterns are evaluated once per dictionary entry at plan time (at most 255 matching entries, else
 * LLKV_ERR_PREDICATE_BUILD), and GROUP BY keys take ceil(log2(entries)) bits (GroupKeyValue::String,
 * llkv-executor/src/lib.rs:99-106,9362-9456).  Group keys of such a column come back with llkv_group_key.dict = 1.
 * Limits: 2^24 distinct strings per column; scalar
 * expressions over a dictionary-coded column are LLKV_ERR_INVALID_ARGUMENT.  Across GPUs the ranks agree on one dictionary
 * per Utf8 key column before a grouped plan is compiled (an all-gather of their entries; a rank whose shard holds short
 * strings only switches to dictionary form with the others), so codes mean the same string on every rank.
 * Row-id-sparse chunks (llkv_gpu_column_append_chunk) take the same forms: short strings are packed on the device as they
 * are scattered to their positions; a chunk with a longer string re-codes the column (only the strings of rows that exist
 * are interned: a gap or a deleted row adds no entry) and later chunks are interned on the host and scattered as codes.
 * A string replaced by a later write, or whose rows were deleted, stays in the dictionary until llkv_gpu_column_clear.
 * At seal the statistics of a sparse short-string column (longest and shortest string, non-ASCII bytes) are recomputed
 * over the rows that exist, so a column whose present strings are all one byte long is kept at one byte per row.
 * llkv_gpu_column_dict_entry: the bytes stay valid until the next append to / clear of the column. */
int32_t llkv_gpu_column_dict_size(llkv_gpu_column* col, uint64_t* out_entries);
int32_t llkv_gpu_column_dict_entry(llkv_gpu_column* col, uint64_t code, const uint8_t** out_bytes, uint64_t* out_len);
/* Sort index (SURVEY.md §8f rank 3; SortIndexOps::stage_build_for_chunk / stage_update_for_new_chunk,
 * llkv-column-map/src/store/indexing/sort.rs:126-172): for every chunk of `chunk_rows` rows (0 = the append path's chunk size
 * for the type) the permutation that lists the chunk's rows in ascending value order — what `lexsort_to_indices` gives the
 * reference (floats by total order; equal values in row order) — built on the device, one CTA per chunk.
 * llkv_gpu_column_sort_index_blob serialises one chunk's permutation exactly as the pager stores it under
 * ChunkMetadata.value_order_perm_pk ("ARR0" header, PrimType UInt32; serialization.rs:41-53): `out_blob` NULL asks for the
 * length only.  Columns with gaps / NULLs, Utf8 and Decimal128 columns that do not fit i64 have no sort index here. */
int32_t llkv_gpu_column_build_sort_index(llkv_gpu_column* col, uint64_t chunk_rows);
int32_t llkv_gpu_column_sort_index_blob(llkv_gpu_column* col, uint64_t chunk_index, void* out_blob, uint64_t cap, uint64_t* out_len);
/* Rows the column holds (llkv_gpu_column_rows counts positions, gaps included). */
int32_t llkv_gpu_column_present_rows(llkv_gpu_column* col, uint64_t* out_rows);
/* Bytes the column's appends have put on the host-to-device link since it was registered (for end-to-end accounting). */
int32_t llkv_gpu_column_h2d_bytes(const llkv_gpu_column* col, uint64_t* out_bytes);
int32_t llkv_gpu_column_rows(const llkv_gpu_column* col, uint64_t* out_rows);
/* Reads rows [row_begin, row_begin + n_rows) of a sealed fixed-width column back into `out` in the Arrow values layout
 * the chunks were appended in (Decimal128 columns kept as i64 on the device are widened again): what a
 * PrimitiveVisitor::*_chunk callback would be handed for that row range (llkv-column-map/src/store/scan/visitors.rs:89-148,
 * scan/unsorted.rs:202-345).  For tests and diagnostics of the resident image; aggregates never copy rows back.
 * LLKV_PT_UTF8 is not supported here. */
int32_t llkv_gpu_column_read(llkv_gpu_column* col, uint64_t row_begin, uint64_t n_rows, void* out, uint64_t out_bytes);
/* Visitor-level boundary (B3): ColumnStore::scan with an unsorted visitor — PrimitiveVisitor::{u64,i64,...}_chunk and
 * PrimitiveWithRowIdsVisitor::*_chunk_with_rids (llkv-column-map/src/store/scan/visitors.rs:89-148, src/lib.rs:174-359,
 * scan/unsorted.rs:202-345).  `visit` is called on the calling thread once per chunk of at most `chunk_rows` positions
 * (0 = the append path's chunk size for the type) with the chunk's values in the Arrow layout (`prim_type` names the
 * element type: the per-dtype method the reference would dispatch to) and, when `with_row_ids` is set, their row ids
 * (NULL otherwise); rows the column does not hold are skipped (ScanOptions::include_nulls = false).  The buffers are only
 * valid during the call.  A non-zero return from `visit` stops the scan and becomes the call's status. */
typedef int32_t (*llkv_chunk_visitor)(void* user, int32_t prim_type, const void* values, const uint64_t* row_ids, uint64_t n_rows);
int32_t llkv_gpu_column_visit(llkv_gpu_column* col, uint64_t chunk_rows, int32_t with_row_ids, llkv_chunk_visitor visit, void* user);
/* ColumnStore::scan(field, ScanOptions, visitor) with the options of llkv-column-map/src/store/scan/options.rs:13-37:
 * unsorted (append order) or sorted by value (ascending, or descending with `reverse`; floats in total order; equal values
 * in row order), paginated by offset / limit across chunks (PaginateVisitor; limit 0 = unbounded), restricted to a value
 * range (`ranges`; bounds are the values' bits in the column's type, signed ones sign-extended), and — sorted scans with
 * row ids only — with the rows of `anchor` that the column does not hold as null runs (`visit` is then called with
 * values = NULL and the row ids: PrimitiveSortedWithRowIdsVisitor::null_run), before or after the values (nulls_first),
 * ascending by row id (descending for reverse scans).  The sort runs on the device (a whole-column stable radix sort: the
 * reference merges its per-chunk value_order_perm runs on the CPU, scan/sorted.rs); pages are gathered and handed to
 * `visit` chunk by chunk in the Arrow layout.  Utf8 and wide Decimal128 columns are LLKV_ERR_INVALID_ARGUMENT. */
typedef struct llkv_scan_options {
  int32_t sorted, reverse, with_row_ids, include_nulls, nulls_first;
  int32_t has_lower, lower_inclusive, has_upper, upper_inclusive;
  int32_t _pad;
  uint64_t lower_bits, upper_bits;
  uint64_t offset, limit;
} llkv_scan_options;
int32_t llkv_gpu_column_scan(llkv_gpu_column* col, llkv_gpu_column* anchor, const llkv_scan_options* options, uint64_t chunk_rows,
                             llkv_chunk_visitor visit, void* user);
/* Drops the rows but keeps the device allocation (re-upload the next batch into the same buffer). */
int32_t llkv_gpu_column_clear(llkv_gpu_column* col);
int32_t llkv_gpu_column_destroy(llkv_gpu_column* col);

/* ---- predicates: ProgramCompiler::compile (llkv-compute/src/program.rs:271-298) ---- */
int32_t llkv_gpu_program_compile(llkv_gpu_ctx* ctx, const llkv_eval_op* ops, int32_t n_ops,
                                 const llkv_literal* literals, int32_t n_literals, const llkv_scalar_node* nodes,
                                 int32_t n_nodes, const int32_t* list_roots, int32_t n_list_roots,
                                 llkv_gpu_program** out);
void llkv_gpu_program_destroy(llkv_gpu_program* prog);

/* ---- MVCC: MvccRowIdFilter (llkv-transaction/src/helpers.rs:259-312), RowVersion::is_visible_for
 *      (llkv-transaction/src/mvcc.rs:282-334).  `noncommitted` lists every txn id whose
 *      TxnIdManager::status is Active or Aborted (mvcc.rs:157-171); unknown ids are Committed. ---- */
int32_t llkv_gpu_mvcc_set(llkv_gpu_ctx* ctx, uint64_t table_id, llkv_gpu_column* created_by,
                          llkv_gpu_column* deleted_by, uint64_t txn_id, uint64_t snapshot_id,
                          const uint64_t* noncommitted, int32_t n_noncommitted);
int32_t llkv_gpu_mvcc_clear(llkv_gpu_ctx* ctx, uint64_t table_id);

/* ---- selection bitmap over row positions (B2: ScanStorage::filter_leaf / RowIdFilter::filter,
 *      llkv-scan/src/lib.rs:163-229).  Bit i of out_words is row (row_begin + i).  `prog` NULL = all rows. ---- */
int32_t llkv_gpu_filter_bitmap(llkv_gpu_ctx* ctx, uint64_t table_id, const llkv_gpu_program* prog, int32_t apply_mvcc,
                               uint64_t row_begin, uint64_t row_end, uint64_t* out_words, uint64_t n_words,
                               uint64_t* out_count);

/* ---- aggregates: AggregateAccumulator::{new_with_projection_index,update,finalize}
 *      (llkv-aggregate/src/lib.rs:463,759,1488) fused with the scan that feeds them
 *      (llkv-executor/src/lib.rs:5357-5682 ungrouped, 4405-4542 + 5028-5355 GROUP BY). ---- */
/* GROUP BY keys (group_key_value, llkv-executor/src/lib.rs:9362-9456: integers, Date32, Boolean, Utf8) are packed into
 * one 64-bit word from the columns' value ranges when they fit.  Wider key tuples are grouped by a 64-bit hash of the key
 * values: after the run a verification pass proves that no two different tuples share a group (otherwise
 * LLKV_ERR_INTERNAL, never a wrong answer) and finalize reads each group's key values from the columns at the group's
 * first row; such aggregates do not merge across GPUs (LLKV_ERR_INVALID_ARGUMENT). */
int32_t llkv_gpu_agg_create(llkv_gpu_ctx* ctx, uint64_t table_id, const llkv_agg_spec* specs, int32_t n_aggs,
                            const llkv_scalar_node* nodes, int32_t n_nodes, const uint64_t* group_key_fields,
                            int32_t n_keys, int32_t expr_mode, uint64_t cardinality_hint, llkv_gpu_agg** out);
/* Resets all accumulators / group tables (a fresh set of AggregateStates). */
int32_t llkv_gpu_agg_reset(llkv_gpu_agg* agg);
/* update(): scans rows [row_begin,row_end) of the table's columns, applies `prog` (NULL = no filter) and,
 * if apply_mvcc, the snapshot set by llkv_gpu_mvcc_set, and folds the survivors into the accumulators.
 * Asynchronous on the context stream. */
int32_t llkv_gpu_agg_run(llkv_gpu_agg* agg, const llkv_gpu_program* prog, int32_t apply_mvcc, uint64_t row_begin,
                         uint64_t row_end);
/* Merges the partial states of all ranks of the communicator bound to the context (SURVEY.md §8e). */
int32_t llkv_gpu_agg_merge(llkv_gpu_agg* agg);
/* One step of a prepared aggregate in one call: llkv_gpu_agg_reset + llkv_gpu_agg_run + (merge != 0 and the context has
 * peers) llkv_gpu_agg_merge — what the executor branch of INTEGRATION.md issues per query (llkv-executor/src/lib.rs:
 * 5357-5682: new states, scan, finalize).  Once a step repeats with nothing changed it is captured as one CUDA graph and
 * replayed with a single launch (llkv_gpu_ctx_set_graphs: 1 = default, 0 = never).  Results are identical either way. */
int32_t llkv_gpu_agg_execute(llkv_gpu_agg* agg, const llkv_gpu_program* prog, int32_t apply_mvcc, uint64_t row_begin,
                             uint64_t row_end, int32_t merge);
int32_t llkv_gpu_ctx_set_graphs(llkv_gpu_ctx* ctx, int32_t mode);
/* Number of groups currently held (1 for ungrouped). Synchronises. */
int32_t llkv_gpu_agg_group_count(llkv_gpu_agg* agg, uint64_t* out_groups);
/* finalize(): writes n_groups*n_aggs values (group-major) and n_groups*n_keys keys, groups in first-appearance
 * order when the aggregate tracks it (low cardinality), otherwise ascending key order.  Errors the reference
 * raises during update (integer overflow, Decimal128 sum overflow, arrow arithmetic overflow) surface here. */
int32_t llkv_gpu_agg_finalize(llkv_gpu_agg* agg, llkv_agg_value* out_values, llkv_group_key* out_keys,
                              uint64_t group_capacity, uint64_t* out_groups);
/* HAVING / ORDER BY / OFFSET / LIMIT over the finalized rows (llkv-executor/src/lib.rs:5306-5348; plans.rs:1205-1225
 * OrderByPlan).  A HAVING term compares one output column (group key or aggregate) with a literal; terms are ANDed and a
 * row stays only when every term is TRUE (a NULL cell is not).  ORDER BY keys sort the remaining rows (stable; ties keep the
 * first-appearance order), NULLs first or last as asked whatever the direction (arrow SortOptions).  limit 0 = no limit.
 * Applies to every later llkv_gpu_agg_finalize of the handle; n_having = n_order = 0 with offset = limit = 0 restores the
 * plain first-appearance output.  The group capacity then bounds the rows that come out, not the groups held. */
typedef struct llkv_order_key {
  int32_t is_aggregate; /* 0: index counts GROUP BY keys, 1: aggregates */
  int32_t index;
  int32_t descending;
  int32_t nulls_first;
} llkv_order_key;
typedef struct llkv_having_term {
  int32_t is_aggregate;
  int32_t index;
  int32_t cmp_op; /* LLKV_CMP_* : cell cmp literal */
  int32_t _pad;
  llkv_literal literal;
} llkv_having_term;
int32_t llkv_gpu_agg_set_output(llkv_gpu_agg* agg, const llkv_having_term* having, int32_t n_having, const llkv_order_key* order,
                                int32_t n_order, uint64_t offset, uint64_t limit);
int32_t llkv_gpu_agg_run_info(const llkv_gpu_agg* agg, llkv_run_info* out);
void llkv_gpu_agg_destroy(llkv_gpu_agg* agg);

/* ---- diagnostics (no GPU needed) ----
 * Compiles a plan against column *descriptions* exactly as llkv_gpu_agg_run would against registered columns and writes a
 * listing (lean program, geometry, accumulator layout) to `out_text`.  With `jit` != 0 the lean kernel is also
 * specialised on the plan shape with NVRTC (cubin written to `cubin_path` when not NULL).  Used by the CPU test-suite
 * and for reading SASS / register counts without a GPU.  Decimal128 columns whose values fit i64 are described as
 * resident i64 (as llkv_gpu_column_seal stores them), one-byte Utf8 columns as one byte per row. */
typedef struct llkv_debug_column {
  uint64_t logical_field_id;
  int32_t prim_type;
  uint8_t precision;
  int8_t scale;
  uint8_t has_minmax;    /* min_value / max_value are valid (integers, dates, decimals that fit i64) */
  uint8_t dec_fits_i64;  /* Decimal128: every value is a sign-extended i64 */
  int64_t min_value, max_value;
  uint64_t n_rows;
  uint8_t max_strlen;    /* Utf8 */
  uint8_t nullable;      /* the column carries a validity bitmap */
  uint8_t _pad[6];
} llkv_debug_column;
int32_t llkv_gpu_debug_plan(const llkv_debug_column* cols, int32_t n_cols, const llkv_gpu_program* prog, int32_t created_by_col,
                            int32_t deleted_by_col, uint64_t txn_id, uint64_t snapshot_id, const llkv_agg_spec* specs, int32_t n_aggs,
                            const llkv_scalar_node* nodes, int32_t n_nodes, const uint64_t* group_key_fields, int32_t n_keys,
                            int32_t expr_mode, uint64_t cardinality_hint, int32_t block_threads, int32_t rows_per_thread, int32_t stages,
                            int32_t ctas_per_sm, int32_t jit /* bit 0: specialise with NVRTC, bit 1: as the partitioned GROUP BY scan, bit 2: as the scan that walks a tile list, bit 3: the partitioned scan with packed tuples, bit 4: the step form of a run that continues the previous one without a reset */, const char* cubin_path, char* out_text, uint64_t out_cap);

/* ---- multi-GPU: one context per rank, NCCL over NVLink (SURVEY.md §8e) ---- */
#define LLKV_GPU_UNIQUE_ID_BYTES 128
int32_t llkv_gpu_comm_unique_id(uint8_t out_id[LLKV_GPU_UNIQUE_ID_BYTES]);
int32_t llkv_gpu_comm_init(llkv_gpu_ctx* ctx, const uint8_t id[LLKV_GPU_UNIQUE_ID_BYTES], int32_t n_ranks,
                           int32_t rank);
int32_t llkv_gpu_comm_destroy(llkv_gpu_ctx* ctx);

#ifdef __cplusplus
}
#endif
#endif /* LLKV_GPU_H */

//! `extern "C"` bindings to `include/llkv_gpu.h`, 1:1.  Authored, not compiled here (no Rust toolchain in the image):
//! the same symbols are exercised through Python ctypes (`rust-llkv_b200/llkv_b200/gpu.py`) by the test-suite, and
//! `tests/test_host_logic.py` checks that the shared library exports every symbol declared below.
//!
//! Field layouts mirror the C structs exactly (`#[repr(C)]`); enum values are the `LLKV_*` constants of the header.
#![allow(non_camel_case_types)]

use core::ffi::{c_char, c_void};

#[repr(C)]
#[derive(Clone, Copy)]
pub struct llkv_literal {
    pub kind: i32,
    pub precision: u8,
    pub scale: i8,
    pub _pad: [u8; 2],
    pub lo: u64,
    pub hi: u64,
}

#[repr(C)]
#[derive(Clone, Copy)]
pub struct llkv_scalar_node {
    pub tag: i32,
    pub op: i32,
    pub left: i32,
    pub right: i32,
    pub field_id: u64,
    pub literal: llkv_literal,
    pub cast_type: i32,
    pub cast_precision: u8,
    pub cast_scale: i8,
    pub _pad: [u8; 2],
}

#[repr(C)]
#[derive(Clone, Copy)]
pub struct llkv_eval_op {
    pub tag: i32,
    pub operator_tag: i32,
    pub field_id: u64,
    pub lower_kind: i32,
    pub upper_kind: i32,
    pub lit_begin: i32,
    pub lit_count: i32,
    pub expr_left: i32,
    pub expr_right: i32,
    pub cmp_op: i32,
    pub negated: i32,
    pub child_count: i32,
    pub literal_bool: i32,
}

#[repr(C)]
#[derive(Clone, Copy)]
pub struct llkv_agg_spec {
    pub kind: i32,
    pub expr_root: i32,
    pub data_type: i32,
    pub precision: u8,
    pub scale: i8,
    pub distinct: u8,
    pub _pad: u8,
}

/// One ORDER BY key over the finalized rows (`OrderByPlan`, llkv-plan/src/plans.rs:1205-1225).
#[repr(C)]
#[derive(Clone, Copy)]
pub struct llkv_order_key {
    pub is_aggregate: i32,
    pub index: i32,
    pub descending: i32,
    pub nulls_first: i32,
}

/// One HAVING term: output column `cmp_op` literal.
#[repr(C)]
#[derive(Clone, Copy)]
pub struct llkv_having_term {
    pub is_aggregate: i32,
    pub index: i32,
    pub cmp_op: i32,
    pub _pad: i32,
    pub literal: llkv_literal,
}

#[repr(C)]
#[derive(Clone, Copy)]
pub struct llkv_agg_value {
    pub lo: u64,
    pub hi: u64,
    pub type_: i32,
    pub precision: u8,
    pub scale: i8,
    pub valid: u8,
    pub _pad: u8,
}

#[repr(C)]
#[derive(Clone, Copy)]
pub struct llkv_group_key {
    pub bits: u64,
    pub type_: i32,
    pub valid: u8,
    /// 1 = `bits` is a code of the key column's dictionary (`llkv_gpu_column_dict_entry`)
    pub dict: u8,
    pub _pad: [u8; 2],
}

/// `ScanOptions` (`llkv-column-map/src/store/scan/options.rs:13-37`) for `llkv_gpu_column_scan`.
#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct llkv_scan_options {
    pub sorted: i32,
    pub reverse: i32,
    pub with_row_ids: i32,
    pub include_nulls: i32,
    pub nulls_first: i32,
    pub has_lower: i32,
    pub lower_inclusive: i32,
    pub has_upper: i32,
    pub upper_inclusive: i32,
    pub _pad: i32,
    pub lower_bits: u64,
    pub upper_bits: u64,
    pub offset: u64,
    pub limit: u64,
}

/// One column as `llkv_gpu_debug_plan` sees it: type and statistics, no data.
#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct llkv_debug_column {
    pub logical_field_id: u64,
    pub prim_type: i32,
    pub precision: u8,
    pub scale: i8,
    pub has_minmax: u8,
    pub dec_fits_i64: u8,
    pub min_value: i64,
    pub max_value: i64,
    pub n_rows: u64,
    pub max_strlen: u8,
    pub nullable: u8,
    pub _pad: [u8; 6],
}

/// ChunkMetadata (llkv-column-map/src/store/descriptor.rs:23-32).
#[repr(C)]
#[derive(Clone, Copy, Default, Debug)]
pub struct llkv_chunk_metadata {
    pub chunk_pk: u64,
    pub value_order_perm_pk: u64,
    pub row_count: u64,
    pub serialized_bytes: u64,
    pub min_val_u64: u64,
    pub max_val_u64: u64,
    pub null_count: u64,
    pub distinct_count: u64,
}

/// ColumnDescriptor, fixed part (descriptor.rs:87-98).
#[repr(C)]
#[derive(Clone, Copy, Default, Debug)]
pub struct llkv_column_descriptor {
    pub field_id: u64,
    pub head_page_pk: u64,
    pub tail_page_pk: u64,
    pub total_row_count: u64,
    pub total_chunk_count: u64,
    pub data_type_code: u32,
    pub index_meta_len: u32,
}

/// std::ops::Bound over raw value bits (kind: LLKV_BOUND_INCLUDED 0, LLKV_BOUND_EXCLUDED 1, LLKV_BOUND_UNBOUNDED 2).
#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct llkv_range_bound {
    pub kind: i32,
    pub _pad: i32,
    pub value_bits: u64,
}

#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct llkv_run_info {
    pub rows: u64,
    pub kernel_launches: u32,
    pub used_wide_path: u32,
    pub algorithmic_bytes_per_row: u32,
    pub physical_bytes_per_row: u32,
    pub grid: u32,
    pub block: u32,
    pub rows_per_tile: u32,
    pub stages: u32,
    pub smem_bytes: u32,
    pub fast_groups: u32,
    pub last_kernel_ms: f32,
    pub used_fast_kernel: u32,
    pub used_jit_kernel: u32,
    pub partitions: u32,
    pub tiles_pruned: u32,
    pub graph_replays: u32,
    pub merged_p2p: u32,
    pub last_merge_ms: f32,
    pub packed_tuples: u32,
    pub published_steps: u32,
}

#[repr(C)]
pub struct llkv_gpu_ctx {
    _private: [u8; 0],
}
#[repr(C)]
pub struct llkv_gpu_column {
    _private: [u8; 0],
}
#[repr(C)]
pub struct llkv_gpu_program {
    _private: [u8; 0],
}
#[repr(C)]
pub struct llkv_gpu_agg {
    _private: [u8; 0],
}

pub const LLKV_GPU_ABI_VERSION: i32 = 1;
pub const LLKV_GPU_UNIQUE_ID_BYTES: usize = 128;

extern "C" {
    pub fn llkv_gpu_abi_version() -> i32;
    pub fn llkv_gpu_last_error(buf: *mut c_char, cap: usize) -> usize;
    pub fn llkv_gpu_device_count() -> i32;

    pub fn llkv_gpu_ctx_create(device_ordinal: i32, n_streams: i32, pinned_bytes: u64, out: *mut *mut llkv_gpu_ctx) -> i32;
    pub fn llkv_gpu_ctx_destroy(ctx: *mut llkv_gpu_ctx);
    pub fn llkv_gpu_ctx_synchronize(ctx: *mut llkv_gpu_ctx) -> i32;
    pub fn llkv_gpu_ctx_stream(ctx: *mut llkv_gpu_ctx, out_stream: *mut *mut c_void) -> i32;
    pub fn llkv_gpu_ctx_set_timing(ctx: *mut llkv_gpu_ctx, enabled: i32) -> i32;
    pub fn llkv_gpu_ctx_set_tuning(ctx: *mut llkv_gpu_ctx, ctas_per_sm: i32, block_threads: i32, stages: i32, rows_per_thread: i32, force_wide: i32) -> i32;
    pub fn llkv_gpu_ctx_set_jit(ctx: *mut llkv_gpu_ctx, mode: i32) -> i32;
    pub fn llkv_gpu_ctx_set_partitioning(ctx: *mut llkv_gpu_ctx, mode: i32) -> i32;
    pub fn llkv_gpu_ctx_set_pruning(ctx: *mut llkv_gpu_ctx, mode: i32) -> i32;
    pub fn llkv_gpu_host_alloc(bytes: u64, out: *mut *mut c_void) -> i32;
    pub fn llkv_gpu_host_free(p: *mut c_void) -> i32;
    pub fn llkv_gpu_host_register(p: *const c_void, bytes: u64) -> i32;
    pub fn llkv_gpu_host_unregister(p: *const c_void) -> i32;
    /// Host workers narrowing Decimal128 chunks from page-locked sources before the DMA: -1 default, 0 off.
    pub fn llkv_gpu_ctx_set_upload_threads(ctx: *mut llkv_gpu_ctx, n_threads: i32) -> i32;
    /// Share (percent) of a hybrid Decimal128 upload that takes the copy engine and is narrowed on the device; -1 = automatic.
    pub fn llkv_gpu_ctx_set_dma_share(ctx: *mut llkv_gpu_ctx, percent: i32) -> i32;
    /// llkv_gpu_agg_execute replays a captured CUDA graph once a step repeats unchanged: 1 (default) / 0.
    pub fn llkv_gpu_ctx_set_graphs(ctx: *mut llkv_gpu_ctx, mode: i32) -> i32;

    /// Compiles a plan against column statistics only (no device): the lean program's listing, optionally its specialised
    /// cubin.  For tooling and CPU-side tests.
    pub fn llkv_gpu_debug_plan(cols: *const llkv_debug_column, n_cols: i32, prog: *const llkv_gpu_program, created_by_col: i32,
                               deleted_by_col: i32, txn_id: u64, snapshot_id: u64, specs: *const llkv_agg_spec, n_aggs: i32,
                               nodes: *const llkv_scalar_node, n_nodes: i32, group_key_fields: *const u64, n_keys: i32,
                               expr_mode: i32, cardinality_hint: u64, block_threads: i32, rows_per_thread: i32, stages: i32,
                               ctas_per_sm: i32, jit: i32, cubin_path: *const c_char, out_text: *mut c_char, out_cap: u64) -> i32;

    pub fn llkv_gpu_descriptor_parse(bytes: *const c_void, len: u64, out: *mut llkv_column_descriptor) -> i32;
    pub fn llkv_gpu_descriptor_page_parse(bytes: *const c_void, len: u64, next_page_pk: *mut u64, out: *mut llkv_chunk_metadata, capacity: u64, n_entries: *mut u64) -> i32;
    pub fn llkv_gpu_sortable_u64(prim_type: i32, value_bits: u64) -> u64;
    pub fn llkv_gpu_chunk_stats(prim_type: i32, values: *const c_void, n_rows: u64, validity: *const u8, out: *mut llkv_chunk_metadata) -> i32;
    pub fn llkv_gpu_chunk_overlaps(prim_type: i32, chunk_min_u64: u64, chunk_max_u64: u64, lower: *const llkv_range_bound, upper: *const llkv_range_bound) -> i32;

    pub fn llkv_gpu_column_register(ctx: *mut llkv_gpu_ctx, logical_field_id: u64, prim_type: i32, precision: u8, scale: i8, out: *mut *mut llkv_gpu_column) -> i32;
    pub fn llkv_gpu_column_reserve(col: *mut llkv_gpu_column, n_rows: u64) -> i32;
    pub fn llkv_gpu_column_append_chunk(col: *mut llkv_gpu_column, chunk_pk: u64, values: *const c_void, n_rows: u64, validity: *const u8, row_ids: *const u64, row_id_base: u64, aux: *const c_void) -> i32;
    pub fn llkv_gpu_column_append_blob(col: *mut llkv_gpu_column, chunk_pk: u64, blob: *const c_void, blob_len: u64, row_ids: *const u64, row_id_base: u64) -> i32;
    /// Issues and waits for the copies earlier appends left pending: page-locked sources may be reused afterwards.
    pub fn llkv_gpu_column_flush(col: *mut llkv_gpu_column) -> i32;
    pub fn llkv_gpu_column_seal(col: *mut llkv_gpu_column) -> i32;
    pub fn llkv_gpu_column_h2d_bytes(col: *const llkv_gpu_column, out_bytes: *mut u64) -> i32;
    /// `ColumnStore::delete_rows`: the rows become gaps of the resident image.
    pub fn llkv_gpu_column_delete_rows(col: *mut llkv_gpu_column, row_ids: *const u64, n: u64) -> i32;
    pub fn llkv_gpu_column_present_rows(col: *mut llkv_gpu_column, out_rows: *mut u64) -> i32;
    /// `ColumnStore::scan(field, ScanOptions, visitor)`: sorted on the device, paginated, with null runs.
    pub fn llkv_gpu_column_scan(col: *mut llkv_gpu_column, anchor: *mut llkv_gpu_column, options: *const llkv_scan_options, chunk_rows: u64,
                                visit: Option<unsafe extern "C" fn(user: *mut c_void, prim_type: i32, values: *const c_void, row_ids: *const u64, n_rows: u64) -> i32>,
                                user: *mut c_void) -> i32;
    /// Entries of the dictionary of a Utf8 column that holds strings longer than 7 bytes (0: packed short strings).
    pub fn llkv_gpu_column_dict_size(col: *mut llkv_gpu_column, out_entries: *mut u64) -> i32;
    /// The string behind a `llkv_group_key` whose `dict` is 1.
    pub fn llkv_gpu_column_dict_entry(col: *mut llkv_gpu_column, code: u64, out_bytes: *mut *const u8, out_len: *mut u64) -> i32;
    /// `SortIndexOps::stage_build_for_chunk` for every chunk of the resident column, on the device.
    pub fn llkv_gpu_column_build_sort_index(col: *mut llkv_gpu_column, chunk_rows: u64) -> i32;
    /// One chunk's permutation as the blob the pager stores under `value_order_perm_pk`.
    pub fn llkv_gpu_column_sort_index_blob(col: *mut llkv_gpu_column, chunk_index: u64, out_blob: *mut c_void, cap: u64, out_len: *mut u64) -> i32;
    /// `gather_rows` with `GatherNullPolicy::IncludeNulls`: values in request order, `out_valid[i] == 0` for absent rows.
    pub fn llkv_gpu_column_gather(col: *mut llkv_gpu_column, row_ids: *const u64, n: u64, out_values: *mut c_void, out_bytes: u64, out_valid: *mut u8) -> i32;
    pub fn llkv_gpu_column_rows(col: *const llkv_gpu_column, out_rows: *mut u64) -> i32;
    pub fn llkv_gpu_column_read(col: *mut llkv_gpu_column, row_begin: u64, n_rows: u64, out: *mut c_void, out_bytes: u64) -> i32;
    /// `ColumnStore::scan` with an unsorted visitor: one callback per chunk, values (+ row ids) borrowed for the call.
    pub fn llkv_gpu_column_visit(col: *mut llkv_gpu_column, chunk_rows: u64, with_row_ids: i32,
                                 visit: Option<unsafe extern "C" fn(user: *mut c_void, prim_type: i32, values: *const c_void, row_ids: *const u64, n_rows: u64) -> i32>,
                                 user: *mut c_void) -> i32;
    pub fn llkv_gpu_column_clear(col: *mut llkv_gpu_column) -> i32;
    pub fn llkv_gpu_column_destroy(col: *mut llkv_gpu_column) -> i32;

    pub fn llkv_gpu_program_compile(ctx: *mut llkv_gpu_ctx, ops: *const llkv_eval_op, n_ops: i32, literals: *const llkv_literal, n_literals: i32, nodes: *const llkv_scalar_node, n_nodes: i32, list_roots: *const i32, n_list_roots: i32, out: *mut *mut llkv_gpu_program) -> i32;
    pub fn llkv_gpu_program_destroy(prog: *mut llkv_gpu_program);

    pub fn llkv_gpu_mvcc_set(ctx: *mut llkv_gpu_ctx, table_id: u64, created_by: *mut llkv_gpu_column, deleted_by: *mut llkv_gpu_column, txn_id: u64, snapshot_id: u64, noncommitted: *const u64, n_noncommitted: i32) -> i32;
    pub fn llkv_gpu_mvcc_clear(ctx: *mut llkv_gpu_ctx, table_id: u64) -> i32;

    pub fn llkv_gpu_filter_bitmap(ctx: *mut llkv_gpu_ctx, table_id: u64, prog: *const llkv_gpu_program, apply_mvcc: i32, row_begin: u64, row_end: u64, out_words: *mut u64, n_words: u64, out_count: *mut u64) -> i32;

    pub fn llkv_gpu_agg_create(ctx: *mut llkv_gpu_ctx, table_id: u64, specs: *const llkv_agg_spec, n_aggs: i32, nodes: *const llkv_scalar_node, n_nodes: i32, group_key_fields: *const u64, n_keys: i32, expr_mode: i32, cardinality_hint: u64, out: *mut *mut llkv_gpu_agg) -> i32;
    pub fn llkv_gpu_agg_reset(agg: *mut llkv_gpu_agg) -> i32;
    pub fn llkv_gpu_agg_run(agg: *mut llkv_gpu_agg, prog: *const llkv_gpu_program, apply_mvcc: i32, row_begin: u64, row_end: u64) -> i32;
    pub fn llkv_gpu_agg_merge(agg: *mut llkv_gpu_agg) -> i32;
    /// reset + run + (merge) in one call; replayed as one CUDA graph once the step repeats unchanged.
    pub fn llkv_gpu_agg_execute(agg: *mut llkv_gpu_agg, prog: *const llkv_gpu_program, apply_mvcc: i32, row_begin: u64, row_end: u64, merge: i32) -> i32;
    pub fn llkv_gpu_agg_group_count(agg: *mut llkv_gpu_agg, out_groups: *mut u64) -> i32;
    pub fn llkv_gpu_agg_finalize(agg: *mut llkv_gpu_agg, out_values: *mut llkv_agg_value, out_keys: *mut llkv_group_key, group_capacity: u64, out_groups: *mut u64) -> i32;
    /// HAVING / ORDER BY / OFFSET / LIMIT applied by every later `llkv_gpu_agg_finalize`.
    pub fn llkv_gpu_agg_set_output(agg: *mut llkv_gpu_agg, having: *const llkv_having_term, n_having: i32, order: *const llkv_order_key, n_order: i32, offset: u64, limit: u64) -> i32;
    pub fn llkv_gpu_agg_run_info(agg: *const llkv_gpu_agg, out: *mut llkv_run_info) -> i32;
    pub fn llkv_gpu_agg_destroy(agg: *mut llkv_gpu_agg);

    pub fn llkv_gpu_comm_unique_id(out_id: *mut u8) -> i32;
    pub fn llkv_gpu_comm_init(ctx: *mut llkv_gpu_ctx, id: *const u8, n_ranks: i32, rank: i32) -> i32;
    pub fn llkv_gpu_comm_destroy(ctx: *mut llkv_gpu_ctx) -> i32;
}

/// `llkv_result::Error` from a status code + the thread's last message (llkv-result/src/error.rs:31-176).
pub fn last_error_message() -> String {
    let mut buf = vec![0u8; 1024];
    let n = unsafe { llkv_gpu_last_error(buf.as_mut_ptr() as *mut c_char, buf.len()) };
    buf.truncate(n.min(buf.len().saturating_sub(1)));
    String::from_utf8_lossy(&buf).into_owned()
}

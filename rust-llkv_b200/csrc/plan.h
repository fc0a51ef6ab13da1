// plan.h — the compiled scan plan shared by the host compiler (compiler.cpp) and the device interpreter
// (scan_kernel.cu).  One Plan = one fused pass: stage column tiles -> predicate program -> MVCC rule ->
// projection arithmetic -> aggregate update, all in registers/shared memory, every column read once.
#pragma once
#ifdef __CUDACC_RTC__  // runtime compilation (jit.cpp): no host headers
typedef unsigned char uint8_t;
typedef unsigned short uint16_t;
typedef unsigned int uint32_t;
typedef unsigned long long uint64_t;
typedef int int32_t;
typedef long long int64_t;
typedef unsigned long size_t;
#else
#include <stdint.h>
#endif

namespace llkv {

constexpr int kMaxCols = 24;
constexpr int kMaxInstr = 320;
constexpr int kMaxFastInstr = 96;      // lean-kernel program (lean_kernel.cuh)
constexpr int kMaxLits = 96;
constexpr int kMaxNoncommitted = 32;
constexpr int kMaxKeys = 8;
constexpr int kMaxWords = 96;          // accumulator words per group row
constexpr int kMaxStackDepth = 12;     // value stack (2 cached in registers + spill slots in shared memory)
constexpr uint32_t kPadRows = 4096;    // column allocations are padded to this many rows (bulk copies never run off the end)
constexpr unsigned long long kEmptyKey = ~0ull;

// ---- opcodes of the per-row stack machine -------------------------------------------------------------
// Value classes: I = signed integer <= 64 bit (sign-extended), U = unsigned 64, F = f64 bits, D = Decimal128
// (i128; i64 in the narrow interpreter), B = predicate result (bit0 = rows bit T, NULL flag = not in domain).
enum Op : uint16_t {
  OP_END = 0,
  OP_PUSH_COL,   // a = column index, b = LoadKind
  OP_PUSH_LIT,   // c = literal index, b = 1 -> NULL literal
  OP_PICK,       // a = depth below top (0 = dup)
  OP_POP,
  OP_NIP,        // drop the entry below the top
  // arrow-arith checked integer ops (llkv-compute/src/kernels.rs:112-137)
  OP_ADD_I, OP_SUB_I, OP_MUL_I, OP_DIV_I, OP_MOD_I,
  OP_ADD_F, OP_SUB_F, OP_MUL_F, OP_DIV_F, OP_MOD_F,
  // Decimal128: b = 1 -> exact mode (DecimalValue::new precision <= 38 check, scalar/decimal.rs:128-170)
  OP_ADD_D, OP_SUB_D, OP_MUL_D,
  // casts (arrow-cast, safe mode: failure -> NULL)
  OP_CAST_I_F, OP_CAST_U_F,
  OP_CAST_D_F,     // c = literal index holding 10^scale as f64
  OP_CAST_I_D,     // a = scale (multiply by 10^a), b = precision, c = 1: the integer is unsigned
  OP_CAST_D_UP,    // a = k, b = precision: x * 10^k
  OP_CAST_D_DOWN,  // a = k, b = precision: x / 10^k rounded half away from zero
  OP_CAST_F_I,
  OP_CAST_I_I,     // a = bits
  OP_CAST_U_I, OP_CAST_I_U, OP_CAST_I_B,
  OP_RESCALE_DX,   // a = k: exact-mode rescale up, overflow -> error (scalar/decimal.rs:30-48)
  // compare -> B (arrow-ord: floats by total order).  a = CompareOp
  OP_CMP_I, OP_CMP_U, OP_CMP_F, OP_CMP_D,
  // typed predicates against literals (llkv-expr/src/typed_predicate.rs:75-142). a = lower_kind | upper_kind<<2 | eq<<4,
  // c = literal index (lower, then upper)
  OP_PRED_I, OP_PRED_U, OP_PRED_F, OP_PRED_D,
  OP_IN_BITS,    // b = count, c = first literal (I/U/short-string/bool: bit equality)
  OP_IN_F, OP_IN_D,
  OP_PRED_STR,   // packed short string against a pattern: a = 0 ends-with / 1 contains / 2 starts-with, | 4 = ASCII case-insensitive;
                 // b = pattern length (<= 7), c = literal (the packed pattern, lower-cased already when case-insensitive)
  OP_PRED_ISNULL, OP_PRED_NOTNULL, OP_PRED_ALL,  // leaf IsNull / IsNotNull / Range(Unbounded,Unbounded): domain = field present
  OP_ISNULL,     // Expr::IsNull{expr,negated}: a = negated; domain = all rows
  OP_INLIST_FOLD, // pops item-compare result into the (matched, saw_null) accumulator below it: internal to PushInList
  OP_INLIST_END,  // a = negated; also folds the NULL flag of the IN target below the accumulator and drops the target
  OP_AND, OP_OR, OP_NOT,
  OP_BOOL_LIT,   // a = value
  OP_FILTER,     // pop B: active &= T.  a bit0 = the warp may stop when no row is active (nothing later can raise an error)
  OP_SELECT_DONE, // end of the selection phase: from here on errors count for selected rows only
  OP_RAISE,      // a = FLAG_* bit index: raised when any row is still active (errors the reference raises at update time)
  OP_MVCC,       // a = created_by column, b = deleted_by column
  OP_GROUP,      // a = number of keys on the stack (packed per Plan::key_*)
  // aggregates. a bit0 = keep the value on the stack; b = fast (per-thread) word; c = global word offset
  OP_AGG_COUNT_STAR, OP_AGG_COUNT,
  OP_AGG_SUM_I, OP_AGG_SUM_D, OP_AGG_FSUM,
  OP_AGG_MIN_I, OP_AGG_MAX_I, OP_AGG_MIN_U, OP_AGG_MAX_U, OP_AGG_MIN_F, OP_AGG_MAX_F, OP_AGG_MIN_D, OP_AGG_MAX_D,
  OP_AGG_FIRSTROW, // MIN over the row index (first-appearance order of groups)
  OP_AGG_FIRSTVALID, // MIN over the row index of non-NULL values (keeps the value)
  OP_AGG_FIRSTNAN,   // MIN over the row index of NaN values (keeps the value): MinFloat64/MaxFloat64 leading-NaN rule
  OP_EMIT_BITMAP,
  OP_COUNT_
};

// ---- opcodes of the lean kernel (lean_kernel.cuh): the hot subset of the machine above as an accumulator machine,
// lowered by the compiler's range analysis for plans whose values provably fit 64 bits.  One i64 (or f64 bits)
// accumulator per row lives in registers; other operands come straight from column tiles, literals or temporaries
// (registers in a specialised build, a tile-sized shared-memory array otherwise).  NULLs are static: an operand is NULL
// exactly where one of the columns it reads is (FInstr::h names them); no overflow checks that the analysis proved dead.
enum FastOp : uint16_t {
  FO_END = 0,
  FO_LEAF,        // a = column, b = LoadKind, c = literal index of (lo, hi): active &= lo <= v <= hi (signed unless LK_U*/LK_STR8)
  FO_MVCC,        // a = created_by column, b = deleted_by column
  FO_SELECT_DONE, // warp leaves the tile when no row is active
  FO_GROUP,       // keys come from Plan::key_col[] (packed as Plan::key_*): CTA-local slot per row
  FO_LD_COL,      // acc = column.            a = column, b = LoadKind
  FO_LD_LIT,      // acc = literal.           c = literal index
  FO_LD_TMP,      // acc = tmp[a]
  FO_ST_TMP,      // tmp[a] = acc
  FO_OP_COL,      // acc = acc op column.     a = FastBin | FB_REV (column op acc), b = LoadKind, c = column
  FO_OP_LIT,      // acc = acc op literal.    a = FastBin | FB_REV, c = literal index
  FO_OP_TMP,      // acc = acc op tmp[b].     a = FastBin | FB_REV
  FO_DIVR,        // a = k, b = 0 signed / 1 non-negative / 2 non-negative and < 2^32 with k <= 9 (value and divisor in 32
                  // bits): acc / 10^k rounded half away from zero
  FO_MULP,        // a = k: acc * 10^k (proven not to overflow)
  FO_I2F,         // i64 -> f64
  FO_D2F,         // c = literal holding 10^scale as f64: (f64)acc / 10^scale
  // aggregates over acc: b = per-warp word, c = global word
  FO_COUNT_STAR, FO_COUNT, FO_FIRSTROW,
  FO_SUM,         // a & 3 = value class: 1 -> 0 <= v < 2^16 (u32 per-thread accumulator), 2 -> |v| < 2^47 (i64 per-thread
                  // accumulator stays exact over 2^15 rows per thread and launch), 0 -> not proven (checked per value);
                  // a bit7 = 4-limb global layout
  FO_FSUM, FO_MIN_I, FO_MAX_I, FO_MIN_F, FO_MAX_F, FO_FIRSTVALID, FO_FIRSTNAN,
  FO_VALID,       // a = column, b = 0: active &= row is valid (not NULL) in the column / 1: active &= row is NULL in it
                  // c = 1: pushed onto the predicate-mask stack instead (b = 2: Range(Unbounded, Unbounded), true on every row)
  // Predicate trees (OR / NOT, llkv-scan/src/predicate.rs:32-193,665-777) on a small stack of (rows, not-in-domain) bit masks,
  // one bit per row of the thread.  FO_LEAF with e = 1 pushes (valid & in range, ~valid) instead of ANDing into the selection.
  FO_MASK_AND, FO_MASK_OR,  // rows: and / or; not-in-domain: or / and (domains intersect / unite, llkv-compute/src/program.rs:500-512)
  FO_MASK_NOT,    // rows = domain - rows
  FO_MASK_LIT,    // a = 0 / 1: push a constant, determined on every row
  FO_MASK_FILTER, // pop: active &= rows
  FO_CMP,         // general comparison of two scalar expressions (compute_compare, llkv-compute/src/kernels.rs:269-297): push
                  // (acc cmp operand) onto the predicate-mask stack.  a = LLKV_CMP_* | kind << 4 (0 signed, 1 unsigned, 2 f64
                  // by total order); b = operand source (0 column c, 1 literal c, 2 tmp c) | FastLoad << 8; h = plan columns
                  // whose NULLs make the comparison NULL (neither selected nor in the domain of a NOT)
  FO_ISNULL,      // Expr::IsNull { expr, negated } over a scalar expression: push (expr IS [NOT] NULL, determined on every row).
                  // a = negated; h = plan columns whose NULLs make the expression NULL
  FO_COUNT_
};
#if defined(__CUDACC__) || defined(__CUDACC_RTC__)
#define LLKV_HD __host__ __device__
#else
#define LLKV_HD
#endif
// Hash of a wide GROUP BY key (single_wide_key == 2): chained over the keys in order, NULL keys by a constant
LLKV_HD constexpr unsigned long long key_hash_init() { return 0x243F6A8885A308D3ull; }
LLKV_HD constexpr unsigned long long key_hash_step(unsigned long long h, unsigned long long field, bool isnull) {
  h = (h ^ (isnull ? 0xD6E8FEB86659FD93ull : field)) * 0x9E3779B97F4A7C15ull;
  h ^= h >> 29;
  h *= 0xBF58476D1CE4E5B9ull;
  h ^= h >> 32;
  return h;
}
LLKV_HD constexpr unsigned long long key_hash_done(unsigned long long h) { return h == ~0ull ? 1ull : h; }  // (~0 = the table's empty marker)
// aggregates whose update needs the row's operand value (the others need the row id or nothing)
LLKV_HD constexpr bool lean_takes_operand(uint32_t op) {
  return op == FO_SUM || op == FO_FSUM || op == FO_MIN_I || op == FO_MAX_I || op == FO_MIN_F || op == FO_MAX_F;
}
enum FastBin : uint8_t {
  FB_ADD = 0, FB_SUB, FB_MUL,   // 64-bit, proven not to overflow
  FB_MUL32,                      // both operands proven to fit i32
  FB_ADD_CK, FB_SUB_CK, FB_MUL_CK,  // checked: overflow raises FLAG_NARROW_FAIL (the 128-bit interpreter decides what it means)
  FB_ADD_F, FB_SUB_F, FB_MUL_F,
  FB_REV = 0x80                  // operands swapped: (other) op acc
};
constexpr int kFastTmps = 3;     // tile-sized temporaries of the lean kernel

enum KeyKind : uint8_t { KK_INT = 0, KK_STR = 1 };
enum LoadKind : uint8_t { LK_I8, LK_I16, LK_I32, LK_I64, LK_U8, LK_U16, LK_U32, LK_U64, LK_F32, LK_F64, LK_D128, LK_STR8,
                          LK_D64,    // Decimal128 column kept as i64 in HBM: every value is a sign-extended i64 (narrowed at seal or on the host)
                          LK_D32 };  // ... kept as i32: every value is a sign-extended i32

// classes of accumulator words: how a word is initialised, merged across CTAs / launches / ranks
enum WordClass : uint8_t {
  WC_SUM = 0, WC_MIN = 1, WC_MAX = 2, WC_FSUM = 3,
  WC_MIN128 = 4, WC_MAX128 = 5,          // high word (order-preserving) of a 128-bit min/max pair; the next word is the low half
  WC_PAIR_LO_MIN = 6, WC_PAIR_LO_MAX = 7
};

// how a per-thread fast word is folded into the global words at the end of the kernel
enum FastKind : uint8_t {
  FK_COUNT = 0,   // u64 count            -> 1 WC_SUM word
  FK_SUM_I64,     // i64 narrow sum       -> L0, L1, NEG64       (value = L0 + L1*2^32 - NEG64*2^64)
  FK_SUM_I128,    // i64 narrow sum       -> L0..L3, NEG128      (value = sum L_k 2^(32k) - NEG128*2^128)
  FK_FSUM,        // f64 sum              -> 1 WC_FSUM word
  FK_MIN, FK_MAX, // order-preserving u64 -> 1 WC_MIN / WC_MAX word
  FK_MIN128_HI, FK_MAX128_HI, // two fast words (hi, lo) -> two global words, merged with a 128-bit CAS
  FK_SKIP         // second word of a 128-bit pair
};

struct Instr {
  uint16_t op;
  uint8_t a, b;
  uint32_t c;
};

struct FInstr {  // lean-kernel instruction, pre-decoded (two 16-byte shared-memory loads, no field unpacking)
  uint32_t op, a, b, c;
  uint32_t d, e, f;  // fused operand pre-load: d = 0 none / 1 acc = literal e / 2 acc = column e of FastLoad f / 3 acc = tmp e
  uint32_t g;        // FO_LEAF: 1 = unsigned comparison, 2 = floats by their ordered integer image, 3 = IN list of f literals; FO_SUM: operand width in bits when proven in [0, 2^32), else 0
  uint32_t h;        // aggregates: bit c = the operand is NULL where plan column c is NULL (the row is then skipped)
};
// physical layouts the lean kernel reads (everything else stays on the general interpreter)
enum FastLoad : uint32_t {
  LKF_4 = 0, LKF_8 = 1, LKF_16 = 2, LKF_1 = 3, LKF_S1 = 4,  // i32 / 8 bytes / low half of 16 / u8 / one-byte string as a packed key
  LKF_1S = 5, LKF_2 = 6, LKF_2U = 7, LKF_4U = 8,            // i8 / i16 / u16 / u32
  LKF_4F = 9                                                // f32, widened to the f64 the arithmetic works in
};

struct Lit {
  unsigned long long lo, hi;
};

struct ColDesc {
  const void* base;              // device values buffer (Arrow layout, little endian)
  const unsigned char* validity; // device validity bitmap (LSB first) or null
  uint32_t elem_bytes;           // 1,2,4,8,16
  uint32_t smem_off;             // byte offset of this column's tile inside a stage
  uint32_t vsmem_off;            // byte offset of the validity tile inside a stage
  uint32_t _pad;
};

struct FastWord {
  uint8_t kind;       // FastKind
  uint8_t lean_width; // lean kernel: bytes of the per-thread accumulator (4 or 8; 0 = 8), set by the lean lowering
  uint8_t lean_rowrel;// lean kernel: the word holds a row index, kept relative to the launch's first tile
  uint8_t _pad;
  uint32_t gword;     // first global word it folds into
};

struct Plan {
  // ---- program
  uint32_t n_instr, n_cols, n_lits, max_depth;
  Instr code[kMaxInstr];
  Lit lits[kMaxLits];
  ColDesc cols[kMaxCols];
  // ---- MVCC snapshot (llkv-transaction/src/mvcc.rs:282-334,414-419)
  unsigned long long txn_id, snapshot_id;
  uint32_t n_noncommitted, _pad0;
  unsigned long long noncommitted[kMaxNoncommitted];
  // ---- group keys: each key value is reduced to key_bits[k] bits (+1 null bit when key_nullable) and packed
  uint32_t n_keys;
  uint32_t single_wide_key;       // 1: one 64-bit key, K = value, NULL key -> dedicated slot
                                  // 2: keys that do not pack into 64 bits: K = key_hash_* over the keys' 64-bit images and
                                  // NULL flags; the values come back from the columns at the group's first row and a
                                  // verification pass proves that no two different keys met in one K (FLAG_KEY_COLLISION)
  uint8_t key_bits[kMaxKeys];
  uint8_t key_nullable[kMaxKeys];
  uint8_t key_kind[kMaxKeys];     // KeyKind
  uint8_t key_strlen[kMaxKeys];   // KK_STR: longest string in the column (<= 7)
  unsigned long long key_min[kMaxKeys];  // KK_INT: subtracted before packing (column minimum)
  // ---- accumulators
  uint32_t n_fast_words;          // per-thread words per CTA-local group
  uint32_t n_gwords;              // words per global group row
  FastWord fast[kMaxWords];
  uint8_t gword_class[kMaxWords]; // WordClass per global word
  // ---- launch geometry
  unsigned long long row_begin, row_end;
  unsigned long long first_tile, n_tiles;  // tiles are tile_rows-aligned from row 0
  uint32_t tile_rows;             // blockDim.x * R
  uint32_t stages;                // >= 2 when staged
  uint32_t staged;                // 1: cp.async.bulk tiles into shared memory; 0: direct global loads
  uint32_t stage_bytes;           // stride between stages in shared memory
  uint32_t tx_bytes;              // bytes one tile's bulk copies deliver (mbarrier expect_tx)
  uint32_t fast_groups;           // CTA-local group slots with per-thread accumulators (power of two, 0 = none)
  uint32_t bitmap_mode;           // 1: OP_EMIT_BITMAP present -> never skip inactive warps
  // ---- lean-kernel program (valid when n_finstr != 0)
  uint32_t n_finstr;
  uint32_t fast_tmps;             // tile-sized temporaries the lean program uses (<= kFastTmps)
  FInstr fcode[kMaxFastInstr];
  uint8_t key_col[kMaxKeys];      // plan column index of each GROUP BY key
  uint8_t key_load[kMaxKeys];     // its LoadKind
  // shared-memory layout (byte offsets from the dynamic smem base; all 128-byte aligned)
  uint32_t smem_bar_off, smem_stage_off, smem_acc_off, smem_spill_off, smem_tbl_off, smem_total;
  // ---- global state
  unsigned long long* gkeys;      // [gcap] open addressing, kEmptyKey = free; group rows gcap (key == kEmptyKey) and gcap+1 (NULL key)
  unsigned long long* gwords;     // [(gcap+2) * n_gwords]
  unsigned long long gcap;        // power of two (1 for ungrouped: row 0)
  uint32_t* flags;                // device status word (FLAG_*)
  unsigned long long* out_bitmap; // bitmap_mode: bit i = row_begin + i  (32-bit words written)
  unsigned long long* out_count;  // bitmap_mode: number of selected rows
  unsigned long long row_origin;  // row id of the columns' position 0: first-row words hold row ids, so shards of one table merge into
                                  // the table's first-appearance order
  const unsigned char* exists_bits;  // row-id-sparse tables: bit i = a row with id row_origin + i exists (null: every position is a row)
};

// ---- the lean kernel's view of a plan (lean_kernel.cuh): passed by value as a __grid_constant__ kernel parameter, so the
// program, literals and layout are read through the constant cache / uniform registers and cost no shared memory.
// LeanShape is everything structural (program, layout, geometry): the runtime compiler (jit.cpp) specialises the kernel on
// it, so a specialised kernel reads only the dynamic half (pointers, literals, row range, snapshot) from the parameter.
constexpr int kLeanMaxWords = 48;
constexpr uint32_t kLeanRowsPerThreadLog2 = 15;  // a thread folds at most 2^15 rows per launch (keeps narrow accumulators exact)
struct LeanCol {
  uint32_t elem_bytes;
  uint32_t smem_off;   // byte offset of this column's tile inside a stage
  uint32_t has_valid;  // the column has a validity bitmap: tile_rows / 8 bytes of it are staged with every tile
  uint32_t vsmem_off;  // ... at this byte offset inside a stage
};
struct LeanWord {
  uint32_t kind;    // FastKind
  uint32_t width;   // 4 or 8 bytes per thread
  uint32_t rowrel;  // row index relative to first_tile * tile_rows
  uint32_t off;     // byte offset of this word's [consumer thread] block inside a slot
  uint32_t gword;   // first global word it folds into
};
struct LeanShape {
  FInstr code[kMaxFastInstr];
  LeanCol cols[kMaxCols];
  LeanWord words[kLeanMaxWords];
  uint32_t key_bits[kMaxKeys], key_kind[kMaxKeys], key_strlen[kMaxKeys], key_col[kMaxKeys], key_load[kMaxKeys];
  uint32_t key_nullable[kMaxKeys];  // packed keys: the field is followed by a null bit (a NULL key value is its own group)
  uint32_t n_code, n_cols, n_words, n_gwords, n_keys, single_wide_key;
  uint32_t direct_global;  // high-cardinality GROUP BY: no CTA-local slots, every selected row updates the global table
  uint32_t nc;           // consumer threads per CTA
  uint32_t rows_per_thread;
  uint32_t fg;           // CTA-local group slots (power of two; 1 when ungrouped)
  uint32_t slot_stride;  // bytes of one slot's accumulators (all consumer threads)
  uint32_t tile_rows, stages, stage_bytes, tx_bytes;
  uint32_t smem_bar_off, smem_stage_off, smem_acc_off, smem_tmp_off, smem_tbl_off, smem_total;
  // Partitioned high-cardinality GROUP BY (specialised builds only): instead of updating the global table row by row
  // (random DRAM sectors), the scan writes (key, row id, aggregate operands) tuples into hash partitions whose slice of the
  // table fits in L2; partition_apply_kernel then folds one partition after the other.
  uint32_t partition;      // 1: tuples out, no accumulation in this kernel
  uint32_t n_fields;       // 64-bit fields per tuple: key, row id, one per aggregate that takes an operand
  uint32_t smem_part_off;  // counters [3][kMaxPartitions + 1] u32, then the tile's tuples [n_fields][tile_rows] u64
  uint32_t use_tile_list;  // 1: the launch walks LeanPlan::tile_list (zone-map pruning); part of the shape so that the
                           // specialised dense kernel carries no trace of it
  // partition == 2, "packed" tuples: key, launch-relative row and the SUM operands of a row fit one 64-bit word
  // (pack_key_bits | pack_row_bits | pack_op_bits[0] | ...).  The CTA collects the tuples of many tiles in a batch buffer and
  // scatters a batch at a time into up to kMaxPackedPartitions partitions small enough for partition_fold_kernel to
  // aggregate in shared memory.  smem_part_off: u32 fill, pad, u32 cnt[parts], u32 base[parts], u64 buf[pack_batch].
  uint32_t pack_key_bits, pack_row_bits, pack_batch, pack_parts;
  uint32_t pack_op_bits[8];
  // row-id-sparse tables: bit i of LeanPlan::exists_bits = a row with id (origin + i) exists; staged like a validity tile
  uint32_t has_exists, exists_smem_off;
};
constexpr int kMaxPartitions = 256;
constexpr int kMaxPackedPartitions = 4096;
struct LeanPlan {
  LeanShape s;
  long long lits[kMaxLits];
  const void* col_base[kMaxCols];
  const unsigned char* col_valid[kMaxCols];  // validity bitmaps (LSB first) of the columns with LeanCol::has_valid
  const unsigned char* exists_bits;
  unsigned long long noncommitted[kMaxNoncommitted];
  unsigned long long key_min[kMaxKeys];
  unsigned long long txn_id, snapshot_id;
  unsigned long long row_begin, row_end, first_tile, n_tiles;
  unsigned long long* gkeys;
  unsigned long long* gwords;
  unsigned long long gcap;
  uint32_t* flags;
  unsigned long long row_origin;  // row id of position 0 (see Plan::row_origin)
  uint32_t n_noncommitted, _pad;
  // partitioned GROUP BY: partition q's field f of tuple j is part_out[(q * n_fields + f) * part_cap + j]; part_cursor[q]
  // counts the tuples reserved so far (tuples past part_cap are applied to the table directly by the scan)
  unsigned long long* part_out;
  uint32_t* part_cursor;
  unsigned long long part_cap;
  uint32_t part_bits, part_shift;  // partition = (mix64(key) & (gcap - 1)) >> part_shift, 2^part_bits partitions
  uint32_t part_dense, _pad2;      // packed tuples: 1 = partition = key >> part_shift (dense integer keys: a partition is a key range)
  // zone-map pruning: when set, the launch visits tiles tile_list[0 .. n_tiles) (ascending, >= first_tile) instead of
  // first_tile .. first_tile + n_tiles: the host dropped the tiles whose zones no conjunct range leaf can match
  const uint32_t* tile_list;
};
constexpr uint32_t kZoneRows = 4096;  // rows per zone-map entry (= the reference's chunk of Decimal128 / Date32 rows, slicing.rs:155-166)

// one aggregate of a partitioned plan as partition_apply_kernel sees it
struct PartOp {
  uint32_t op, flags, gword, _pad;
};
constexpr int kMaxPartOperands = 8;  // operand fields per tuple (tuple = key, row id, operands)
struct PartPlan {
  const unsigned long long* tuples;
  const uint32_t* cursor;
  unsigned long long part_cap;
  unsigned long long* gkeys;
  unsigned long long* gwords;
  unsigned long long gcap;
  uint32_t* flags;
  uint32_t n_parts, n_fields, n_keys, n_gwords, n_nops, n_vops, chunk, chunks_per_part;
  PartOp nops[kLeanMaxWords];       // aggregates without an operand (COUNT, first row)
  PartOp vops[kMaxPartOperands];    // aggregates with one: vops[j] reads tuple field 2 + j
};

// pass 2 of the packed form (partition_fold_kernel): one CTA aggregates a whole partition in shared memory and writes each
// group of it to the global table once
struct FoldPlan {
  const unsigned long long* tuples;  // partition q: tuples[q * part_cap ..]
  const uint32_t* cursor;
  unsigned long long part_cap;
  unsigned long long* gkeys;
  unsigned long long* gwords;
  unsigned long long gcap;
  uint32_t* flags;
  unsigned long long row_base;       // row id of launch-relative row 0
  uint32_t n_parts, n_gwords, n_keys;
  uint32_t key_bits, row_bits;
  uint32_t dense, part_shift;        // dense: slot = key & (slots - 1), key = q << part_shift | slot; else a hash table in shared memory
  uint32_t slots;                    // shared-memory slots per partition (power of two)
  uint32_t n_ops, n_counts;
  uint32_t op_bits[8], op_gword[8], op_wide[8];  // SUM operands: bits in the tuple, first global word, 1 = 4-limb global layout
  uint32_t count_gword[kLeanMaxWords];           // words that count rows (COUNT(*), COUNT(col) of a non-null column)
  uint32_t first_gword;              // word holding the group's first row id (MIN), ~0u = none
};

enum : uint32_t {
  FLAG_NARROW_FAIL = 1u << 0,      // the 64-bit interpreter met a value that needs 128 bits: rerun wide
  FLAG_ARITH_OVERFLOW = 1u << 1,   // arrow-arith checked op overflowed on a selected row
  FLAG_DIV_ZERO = 1u << 2,
  FLAG_EXACT_OVERFLOW = 1u << 3,   // exact-mode decimal op overflowed / exceeded 38 digits
  FLAG_TABLE_FULL = 1u << 4,       // global group table is full
  FLAG_BAD_PLAN = 1u << 5,
  FLAG_TYPE_ERROR = 1u << 6,       // OP_RAISE: aggregate argument of a type the accumulator rejects, met on a selected row
  FLAG_MERGE_TIMEOUT = 1u << 7,    // multi-GPU merge: a peer's partial state never arrived
  FLAG_MERGE_OVERSIZE = 1u << 8,   // multi-GPU merge over peer mailboxes: some rank's group table outgrew a mailbox slot
  FLAG_MERGE_RETRY = 1u << 9,      // ... some rank's scan has to be repeated first (64-bit overflow, table full): every rank merges again
  FLAG_MERGE_PEER_FAILED = 1u << 10, // ... some rank's scan ended with an error: no merged result on any rank
  FLAG_KEY_COLLISION = 1u << 11     // hashed wide GROUP BY keys: two different keys share a 64-bit hash
};

}  // namespace llkv

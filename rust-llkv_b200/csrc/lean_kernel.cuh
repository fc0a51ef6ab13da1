// lean_kernel.cuh — body of the lean scan -> filter -> MVCC -> project -> aggregate kernel for sm_100a.
//
// Runs the FastOp program the compiler lowers (compiler.cpp: lower_fast) when range analysis over the columns' min/max
// statistics proves that every value fits 64 bits: typed leaves, IN lists, general comparisons and IS NULL over scalar
// expressions, AND / OR / NOT trees with domains, validity bitmaps (NULL-skipping aggregates, nullable GROUP BY keys),
// MVCC, projection arithmetic, aggregates.  Everything else runs on the general interpreter (scan_kernel.cu); both
// produce identical accumulator states.
//
// The same source is compiled twice:
//   * ahead of time (lean_kernel.cu, nvcc): Cfg = LeanDynCfg, the program and layout are read from the __grid_constant__
//     kernel parameter and interpreted (one dispatch per instruction and tile);
//   * at run time (jit.cpp, NVRTC) for plans that run repeatedly: Cfg = LeanJitCfg, the program and layout (LeanShape) are
//     a compile-time constant, `step()` is instantiated once per program position with a constexpr instruction, so the
//     dispatch, the operand decoding and every layout offset fold away and the compiler sees straight-line code.
//
// Shape of one CTA: NC consumer threads + one producer warp.
//   * The producer's elected lane keeps `stages` row tiles in flight with cp.async.bulk (TMA 1-D bulk copies, one per
//     column per tile) and full/empty mbarriers per stage; consumers never wait on HBM and there is no __syncthreads
//     in the tile loop.
//   * Each consumer thread owns R rows of the tile (row = r * NC + thread, so a warp's shared-memory reads of 4/8 B
//     elements are conflict free).  Typed predicate leaves compare straight out of the tile into a bit mask; the
//     projection arithmetic is an accumulator machine: one i64 per row in registers, the other operand read from a
//     column tile, a literal or a tile-sized temporary in shared memory.
//   * Aggregates are thread-private: every consumer thread owns one accumulator per (CTA-local group slot, word) in
//     shared memory, laid out [slot][word][thread] so a warp's read-modify-write is conflict free and needs no atomics
//     (64-bit shared-memory atomics are CAS loops on this architecture).  Words whose per-thread total provably fits
//     32 bits (counts, row indices, small sums) are 4 bytes wide.
//   * At the end the threads' accumulators are reduced per (slot, word) with warp shuffles and folded into the global
//     group table with one atomic per word.
//
// Variants selected by the shape (constants in a specialised build):
//   * direct_global — high-cardinality GROUP BY: no CTA-local slots, every selected row looks up its row of the global
//     table (the thread's R probes advance together, round by round) and updates it with one RED per word;
//   * partition (specialised builds only) — the same plans when the table outgrows L2: instead of updating the table the
//     CTA writes the tile's (key, row id, operands) tuples into hash partitions (LeanTile::scatter); partition_kernel.cu
//     folds them partition by partition, inside L2;
//   * use_tile_list — zone-map pruning: the launch walks LeanPlan::tile_list (the tiles whose zones some conjunct range
//     leaf can match) instead of the dense tile range.
#pragma once
#include "device_util.cuh"
#include "plan.h"

namespace llkv {

#define LLKV_FULL 0xffffffffu
// has_slow as a branch condition (inside LeanTile::step): SLOW is false in the copy of a specialised program that runs
// after a GROUP instruction found a CTA-local slot for every row of the warp
#define LLKV_SLOW_HERE (SLOW && has_slow)

__device__ __forceinline__ double lean_f64(i64 v) { return __longlong_as_double(v); }
__device__ __forceinline__ i64 lean_bits(double d) { return __double_as_longlong(d); }

// Row of the global group table for key K (inserting it if new).  Bit 63 of the result reports a full table (the row is
// then the spare one and the run is repeated with a larger table): no pointer to caller state, so callers' per-row
// registers never get their address taken.
constexpr u64 kSlotTableFull = 1ull << 63;
static __device__ __noinline__ u64 lean_global_slot_raw(u64* gkeys, u64 gcap, uint32_t n_keys, u64 K) {
  if (n_keys == 0) return 0;
  if (K == kEmptyKey) return gcap;
  const u64 mask = gcap - 1;
  u64 h = mix64(K) & mask;
  for (u64 i = 0; i <= mask; ++i) {
    u64 cur = gkeys[h];
    if (cur == K) return h;
    if (cur == kEmptyKey) {
      const u64 old = atomicCAS(&gkeys[h], kEmptyKey, K);
      if (old == kEmptyKey || old == K) return h;
    }
    h = (h + 1) & mask;
  }
  return gcap | kSlotTableFull;  // parked on the spare row; the flag makes the run fail
}
__device__ __forceinline__ u64 lean_global_slot(u64* gkeys, u64 gcap, uint32_t n_keys, u64 K, uint32_t& errbits) {
  const u64 gs = lean_global_slot_raw(gkeys, gcap, n_keys, K);
  if (gs & kSlotTableFull) errbits |= FLAG_TABLE_FULL;
  return gs & ~kSlotTableFull;
}

// rows without a CTA-local group slot (more groups than slots) and values too large for the per-thread i64 partials go
// straight to the global table, one atomic per word: kept out of line
static __device__ __noinline__ void lean_slow_accumulate(u64* w, uint32_t op, uint32_t flags, i64 v, u64 row) {
  switch (op) {
    case FO_COUNT_STAR: case FO_COUNT: atomicAdd(w, 1ull); break;
    case FO_FIRSTROW: case FO_FIRSTVALID: case FO_FIRSTNAN: atomicMin(w, row); break;
    case FO_SUM:
      if (flags & 0x80) gadd_sum_i128(w, (i128)v);
      else gadd_sum_i64(w, (i128)v);
      break;
    case FO_FSUM: atomicAdd(reinterpret_cast<double*>(w), lean_f64(v)); break;
    case FO_MIN_I:
      if (flags & 0x80) gmin128(w, enc_i64(v >> 63), (u64)v, false);  // Decimal128 state: (hi encoded, lo) pair
      else atomicMin(w, enc_i64(v));
      break;
    case FO_MAX_I:
      if (flags & 0x80) gmin128(w, enc_i64(v >> 63), (u64)v, true);
      else atomicMax(w, enc_i64(v));
      break;
    case FO_MIN_F: atomicMin(w, enc_f64(lean_f64(v))); break;
    default: atomicMax(w, enc_f64(lean_f64(v))); break;
  }
}

// one aggregate's update from a tuple field of a partitioned plan: MIN/MAX operands travel in their order-preserving
// encoding (what emit() parks), everything else as the raw value
__device__ __forceinline__ void lean_apply_field(u64* w, uint32_t op, uint32_t flags, u64 field, u64 row) {
  const bool enc = op == FO_MIN_I || op == FO_MAX_I;
  lean_slow_accumulate(w, op, flags, enc ? (i64)(field ^ 0x8000000000000000ull) : (i64)field, row);
}

// packed GROUP BY key of row `idx` of the staged tile (slow path; the hot path computes keys in LeanTile::row_keys)
static __device__ __noinline__ u64 lean_row_key(const LeanPlan& p, const LeanShape& S, const unsigned char* sb, uint32_t idx) {
  u64 K = 0;
  int shift = 0;
  for (uint32_t k = 0; k < S.n_keys; ++k) {
    const unsigned char* base = sb + S.cols[S.key_col[k]].smem_off;
    const uint32_t kind = S.key_load[k];
    i64 v;
    if (kind == LKF_S1) v = (i64)(((u64)base[idx] << 56) | 1ull);
    else if (kind == LKF_1) v = base[idx];
    else if (kind == LKF_1S) v = reinterpret_cast<const signed char*>(base)[idx];
    else if (kind == LKF_2) v = reinterpret_cast<const short*>(base)[idx];
    else if (kind == LKF_2U) v = reinterpret_cast<const unsigned short*>(base)[idx];
    else if (kind == LKF_4U) v = reinterpret_cast<const unsigned int*>(base)[idx];
    else if (kind == LKF_4) v = reinterpret_cast<const int*>(base)[idx];
    else if (kind == LKF_16) v = reinterpret_cast<const i64*>(base)[2 * idx];
    else v = reinterpret_cast<const i64*>(base)[idx];
    const int bits = (int)S.key_bits[k];
    u64 f;
    if (S.key_kind[k] == KK_STR) {
      const int L = (int)S.key_strlen[k];
      f = (L ? (((u64)v >> (64 - 8 * L)) << 3) : 0ull) | ((u64)v & 7ull);
    } else {
      f = (u64)v - p.key_min[k];
    }
    if (S.single_wide_key == 2) K = key_hash_step(k == 0 ? key_hash_init() : K, (u64)v, false);
    else if (S.single_wide_key) K = (u64)v;
    else {
      bool is_null = false;
      if (S.key_nullable[k] && S.cols[S.key_col[k]].has_valid) {
        const uint32_t* w = reinterpret_cast<const uint32_t*>(sb + S.cols[S.key_col[k]].vsmem_off);
        is_null = !((w[idx >> 5] >> (idx & 31)) & 1u);
      }
      if (!is_null) K |= (bits == 64 ? f : (f & ((1ull << bits) - 1))) << shift;
      if (S.key_nullable[k]) K |= (u64)is_null << (shift + bits);
    }
    shift += bits + (S.single_wide_key == 0 && S.key_nullable[k] ? 1 : 0);
  }
  return S.single_wide_key == 2 ? key_hash_done(K) : K;
}

__device__ __forceinline__ void mbar_wait_parked(void* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  while (!mbar_try_wait_hint(bar, parity, 20000u)) {
  }
}

__device__ __forceinline__ uint32_t hash_key32(u64 K) {
  const uint32_t x = (uint32_t)K ^ (uint32_t)(K >> 32) * 0x9e3779b1u;
  return (x * 0x85ebca6bu) >> 8;
}

__host__ __device__ constexpr bool lean_is_aggregate(uint32_t op) { return op >= FO_COUNT_STAR && op <= FO_FIRSTNAN; }
// index of the aggregate instruction at `pc` among the program's aggregate instructions (specialised builds)
template <class Cfg>
__host__ __device__ constexpr int lean_stash_index(int pc) {
  int k = 0;
  for (int i = 0; i < pc; ++i)
    if (lean_is_aggregate(Cfg::code(i).op)) ++k;
  return k;
}

// partitioned plans: tuple field of the aggregate at `pc` (0 = key, 1 = row id, then one per operand-taking aggregate)
template <class Cfg>
__host__ __device__ constexpr int lean_field_index(int pc) {
  int k = 2;
  for (int i = 0; i < pc; ++i)
    if (lean_takes_operand(Cfg::code(i).op)) ++k;
  return k;
}
__device__ __forceinline__ void lean_consumer_barrier(int nc) { asm volatile("bar.sync 1, %0;" ::"r"(nc) : "memory"); }

// interpreted: the shape comes with the kernel parameter
struct LeanDynCfg {
  static constexpr bool kStatic = false;
  static constexpr bool kDefer = false;
  static constexpr bool kPartition = false;
  static constexpr bool kPacked = false;
  static constexpr bool kSplitSlow = false;
  static constexpr int kStash = 1;
  static constexpr int kTmps = 1;
  static __host__ __device__ constexpr FInstr code(int) { return FInstr{}; }
  static __device__ __forceinline__ const LeanShape& shape(const LeanPlan& p) { return p.s; }
};

// Per-tile execution state of one consumer thread.  Everything lives in registers: step() is force-inlined into the
// dispatch loop (interpreted) or into the unrolled program (specialised).
template <int R, class Cfg>
struct LeanTile {
  const LeanPlan& p;
  const LeanShape& S;
  const int tid, NC;
  const uint32_t T;
  unsigned char* const my4;  // this thread's 4-byte accumulators: my4 + word.off + soff[r]
  unsigned char* const my8;
  i64* const tmp_base;
  u64* const tbl;
  const bool grouped;
  // per tile
  const unsigned char* sb = nullptr;
  u64 row0 = 0;
  uint32_t rel0 = 0;
  i64 acc[R];
  uint32_t soff[R];  // byte offset of the row's slot inside the accumulator area
  uint32_t gsl[R];   // rows in negm: their row of the global table (capacity < 2^32)
  unsigned actm = 0;  // bit r: row r of this thread is selected
  unsigned negm = 0;  // bit r: selected row without a CTA-local group slot (goes to the global table directly)
  bool has_slow = false;  // warp-uniform: some lane has a row in negm
  uint32_t errbits = 0;
  // specialised + grouped: operands / row masks of the tile's aggregate instructions, applied by flush()
  u64 stash_v[Cfg::kStash][R];
  unsigned stash_m[Cfg::kStash];
  i64 treg[Cfg::kTmps][R];  // specialised: the program's temporaries (a thread only ever reads its own rows' entries)
  u64 pk[Cfg::kPartition ? R : 1];  // partitioned plans: the rows' packed keys, kept from GROUP to scatter()
  unsigned char* const part_smem;
  uint32_t batch_tiles = 0;         // packed form: tiles appended to the batch buffer since the last flush
  // predicate trees (OR / NOT): a small stack of (rows, not-in-domain) masks, one bit per row of this thread
  unsigned mt[8], mn[8];
  int msp = 0;

  __device__ __forceinline__ LeanTile(const LeanPlan& plan, const LeanShape& shape, unsigned char* smem, int tid_, int nc)
      : p(plan), S(shape), tid(tid_), NC(nc), T(shape.tile_rows), my4(smem + shape.smem_acc_off + tid_ * 4),
        my8(smem + shape.smem_acc_off + tid_ * 8), tmp_base(reinterpret_cast<i64*>(smem + shape.smem_tmp_off)),
        tbl(reinterpret_cast<u64*>(smem + shape.smem_tbl_off)), grouped(shape.n_keys != 0), part_smem(smem + shape.smem_part_off) {}

  // one column's R values as sign/zero-extended i64.  The lean kernel knows four physical layouts.
  __device__ __forceinline__ void load_col(uint32_t col, uint32_t kind, i64 (&out)[R]) const {
    const unsigned char* base = sb + S.cols[col].smem_off;
    if (kind == LKF_8) {
#pragma unroll
      for (int r = 0; r < R; ++r) out[r] = reinterpret_cast<const i64*>(base)[r * NC + tid];
    } else if (kind == LKF_4) {
#pragma unroll
      for (int r = 0; r < R; ++r) out[r] = reinterpret_cast<const int*>(base)[r * NC + tid];
    } else if (kind == LKF_16) {  // Decimal128 proven to hold sign-extended i64 values: the low half is the value
#pragma unroll
      for (int r = 0; r < R; ++r) out[r] = reinterpret_cast<const i64*>(base)[2 * (r * NC + tid)];
    } else if (kind == LKF_1) {
#pragma unroll
      for (int r = 0; r < R; ++r) out[r] = base[r * NC + tid];
    } else if (kind == LKF_1S) {
#pragma unroll
      for (int r = 0; r < R; ++r) out[r] = reinterpret_cast<const signed char*>(base)[r * NC + tid];
    } else if (kind == LKF_2) {
#pragma unroll
      for (int r = 0; r < R; ++r) out[r] = reinterpret_cast<const short*>(base)[r * NC + tid];
    } else if (kind == LKF_2U) {
#pragma unroll
      for (int r = 0; r < R; ++r) out[r] = reinterpret_cast<const unsigned short*>(base)[r * NC + tid];
    } else if (kind == LKF_4U) {
#pragma unroll
      for (int r = 0; r < R; ++r) out[r] = reinterpret_cast<const unsigned int*>(base)[r * NC + tid];
    } else if (kind == LKF_4F) {
#pragma unroll
      for (int r = 0; r < R; ++r) out[r] = lean_bits((double)reinterpret_cast<const float*>(base)[r * NC + tid]);
    } else {  // LKF_S1: one-byte strings as packed keys
#pragma unroll
      for (int r = 0; r < R; ++r) out[r] = (i64)(((u64)base[r * NC + tid] << 56) | 1ull);
    }
  }

  // validity of this thread's R rows in one column's staged bitmap tile: row r * NC + tid is bit (tid & 31) of 32-bit word
  // r * (NC / 32) + tid / 32, the same word for the whole warp (one broadcast read per row slot)
  __device__ __forceinline__ unsigned bits_of(const unsigned char* tile) const {
    const uint32_t* w = reinterpret_cast<const uint32_t*>(tile) + (tid >> 5);
    unsigned m = 0;
#pragma unroll
    for (int r = 0; r < R; ++r) m |= ((w[r * (NC >> 5)] >> (tid & 31)) & 1u) << r;
    return m;
  }
  __device__ __forceinline__ unsigned col_valid(uint32_t col) const { return bits_of(sb + S.cols[col].vsmem_off); }
  // rows on which every column of `cols` (bit c = plan column c) is valid
  __device__ __forceinline__ unsigned valid_mask(uint32_t cols) const {
    unsigned m = (1u << R) - 1u;
#pragma unroll
    for (uint32_t c = 0; c < (uint32_t)kMaxCols; ++c)
      if ((cols >> c) & 1u) m &= col_valid(c);
    return m;
  }

  // acc = acc op other  (rev: other op acc)
  __device__ __forceinline__ void binop(uint32_t opr, const i64 (&o)[R]) {
    const bool rev = (opr & FB_REV) != 0;
    switch (opr & 0x7f) {
      case FB_ADD:
#pragma unroll
        for (int r = 0; r < R; ++r) acc[r] += o[r];
        break;
      case FB_SUB:
#pragma unroll
        for (int r = 0; r < R; ++r) acc[r] = rev ? o[r] - acc[r] : acc[r] - o[r];
        break;
      case FB_MUL:
#pragma unroll
        for (int r = 0; r < R; ++r) acc[r] *= o[r];
        break;
      case FB_MUL32:  // both operands proven to fit i32: one mul.wide.s32 (the optimiser otherwise widens to a 64 x 64 product)
#pragma unroll
        for (int r = 0; r < R; ++r) {
          i64 prod;
          asm("mul.wide.s32 %0, %1, %2;" : "=l"(prod) : "r"((int)acc[r]), "r"((int)o[r]));
          acc[r] = prod;
        }
        break;
      case FB_ADD_CK: case FB_SUB_CK: case FB_MUL_CK:
#pragma unroll
        for (int r = 0; r < R; ++r) {
          const i64 a = rev ? o[r] : acc[r], b = rev ? acc[r] : o[r];
          i64 c;
          const uint32_t k = opr & 0x7f;
          const bool ok = k == FB_ADD_CK ? add_ck(a, b, c) : k == FB_SUB_CK ? sub_ck(a, b, c) : mul_ck(a, b, c);
          if (!ok && ((actm >> r) & 1u)) errbits |= FLAG_NARROW_FAIL;
          acc[r] = c;
        }
        break;
      case FB_ADD_F:
#pragma unroll
        for (int r = 0; r < R; ++r) acc[r] = lean_bits(lean_f64(acc[r]) + lean_f64(o[r]));
        break;
      case FB_SUB_F:
#pragma unroll
        for (int r = 0; r < R; ++r) acc[r] = lean_bits(rev ? lean_f64(o[r]) - lean_f64(acc[r]) : lean_f64(acc[r]) - lean_f64(o[r]));
        break;
      default:
#pragma unroll
        for (int r = 0; r < R; ++r) acc[r] = lean_bits(lean_f64(acc[r]) * lean_f64(o[r]));
        break;
    }
  }

  // packed GROUP BY keys of this thread's R rows (key-major: each key column's constants are read once)
  __device__ __forceinline__ void row_keys(u64 (&keys)[R]) const {
#pragma unroll
    for (int r = 0; r < R; ++r) keys[r] = 0;
    int shift = 0;
#pragma unroll
    for (uint32_t k = 0; k < (uint32_t)kMaxKeys; ++k) {
      if (k < S.n_keys) {
        i64 v[R];
        load_col(S.key_col[k], S.key_load[k], v);
        const int bits = (int)S.key_bits[k];
        const u64 kmin = p.key_min[k];
        const bool is_str = S.key_kind[k] == KK_STR;
        const int L = (int)S.key_strlen[k];
        const u64 mask = bits == 64 ? ~0ull : ((1ull << bits) - 1);
        // nullable packed key: field 0 and the null bit set where the value is NULL
        const bool nullable = S.single_wide_key == 0 && S.key_nullable[k] != 0;
        const unsigned valid = nullable && S.cols[S.key_col[k]].has_valid ? col_valid(S.key_col[k]) : (1u << R) - 1u;
#pragma unroll
        for (int r = 0; r < R; ++r) {
          const u64 f = is_str ? ((L ? (((u64)v[r] >> (64 - 8 * L)) << 3) : 0ull) | ((u64)v[r] & 7ull)) : (u64)v[r] - kmin;
          if (S.single_wide_key == 2) keys[r] = key_hash_step(k == 0 ? key_hash_init() : keys[r], (u64)v[r], false);
          else if (S.single_wide_key) keys[r] = (u64)v[r];
          else if (nullable) keys[r] |= ((valid >> r) & 1u) ? (f & mask) << shift : 1ull << (shift + bits);
          else keys[r] |= (f & mask) << shift;
        }
        shift += bits + (nullable ? 1 : 0);
      }
    }
    if (S.single_wide_key == 2) {
#pragma unroll
      for (int r = 0; r < R; ++r) keys[r] = key_hash_done(keys[r]);
    }
  }

  // Rows that go to the global table one atomic at a time: rows without a CTA-local slot (their global row was looked up
  // once, at GROUP: high-cardinality plans send nearly every row this way) and values outside the proven range (rare:
  // the global row is looked up here).
  __device__ __forceinline__ void slow_rows(uint32_t op, uint32_t flags, unsigned rows, uint32_t gword) {
    if (__any_sync(LLKV_FULL, rows != 0)) {
#pragma unroll
      for (int r = 0; r < R; ++r)  // unrolled: acc[] must never be indexed dynamically
        if ((rows >> r) & 1u) {
          u64 gs = gsl[r];
          if (!((negm >> r) & 1u)) gs = lean_global_slot(p.gkeys, p.gcap, S.n_keys, lean_row_key(p, S, sb, (uint32_t)(r * NC + tid)), errbits);
          lean_slow_accumulate(&p.gwords[gs * S.n_gwords + gword], op, flags, acc[r], row0 + (u64)r * NC + tid);
        }
    }
  }

  // `rel_row0`: first row of the tile relative to the launch's first tile (a launch covers < 2^32 rows, so the per-tile
  // bookkeeping is 32-bit; the absolute row is only formed where an aggregate needs it)
  __device__ __forceinline__ void begin_tile(const unsigned char* stage, uint32_t rel_row0, u64 base_row, uint32_t begin_rel, uint32_t end_rel) {
    sb = stage;
    row0 = p.row_origin + base_row + rel_row0;  // a row id: only first-row words and the per-row global path use it
    rel0 = rel_row0 + (uint32_t)tid;  // launch-relative index of this thread's row r = 0
    negm = 0;
    has_slow = false;
    msp = 0;
    if (rel_row0 >= begin_rel && rel_row0 + T <= end_rel) {
      actm = (1u << R) - 1u;
    } else {
      actm = 0;
#pragma unroll
      for (int r = 0; r < R; ++r) {
        const uint32_t row = rel0 + (uint32_t)(r * NC);
        if (row >= begin_rel && row < end_rel) actm |= 1u << r;
      }
    }
    if (S.has_exists) actm &= bits_of(sb + S.exists_smem_off);  // row ids nobody holds (deleted rows, gaps) are not rows
#pragma unroll
    for (int r = 0; r < R; ++r) {
      acc[r] = 0;
      soff[r] = 0;
      gsl[r] = 0;
    }
  }

  // executes one instruction for this thread's R rows; false = the warp is done with the tile
  // specialised builds instantiate only the case of the instruction at PC (the others are discarded at compile time:
  // a quarter of the NVRTC time); the interpreting build keeps them all
  template <int PC>
  static __host__ __device__ constexpr bool live(uint32_t op) {
    if constexpr (Cfg::kStatic && PC >= 0) return Cfg::code(PC).op == op;
    else return true;
  }
  template <int PC, bool SLOW = true>
  __device__ __forceinline__ bool step(const FInstr& in) {
    // optional operand pre-load fused into the instruction: acc = literal / column / temporary
    if (in.d == 2) load_col(in.e, in.f, acc);
    else if (in.d == 1) {
      const i64 v = p.lits[in.e];
#pragma unroll
      for (int r = 0; r < R; ++r) acc[r] = v;
    } else if (in.d == 3) {
      if constexpr (Cfg::kStatic && PC >= 0) {
        constexpr uint32_t slot = Cfg::code(PC).e;
#pragma unroll
        for (int r = 0; r < R; ++r) acc[r] = treg[slot][r];
      } else {
        const i64* t = tmp_base + (size_t)in.e * T;
#pragma unroll
        for (int r = 0; r < R; ++r) acc[r] = t[r * NC + tid];
      }
    }
    const unsigned ng = SLOW ? negm : 0u;  // (no row of the warp is in negm when the SLOW = false copy runs)
    switch (in.op) {
      case FO_LEAF: if constexpr (live<PC>(FO_LEAF)) {
        const i64 lo = p.lits[in.c], hi = p.lits[in.c + 1];
        const unsigned char* base = sb + S.cols[in.a].smem_off;
        unsigned m = 0;
        if (in.g == 3) {  // IN list of in.f entries: equality of the 64-bit images
          i64 v[R];
          load_col(in.a, in.b, v);
          for (uint32_t k = 0; k < in.f; ++k) {
            const i64 L = p.lits[in.c + k];
#pragma unroll
            for (int r = 0; r < R; ++r) m |= (unsigned)(v[r] == L) << r;
          }
        } else if (in.g == 1 ? (u64)hi < (u64)lo : hi < lo) {
          // empty range: nothing matches
        } else if (in.g == 2) {  // floats through their order-preserving integer image (NaNs lie outside [k(-inf), k(+inf)])
          if (in.b == LKF_4) {
            const uint32_t l = (uint32_t)(int)lo, span = (uint32_t)(int)hi - l;
#pragma unroll
            for (int r = 0; r < R; ++r) {
              const int b = reinterpret_cast<const int*>(base)[r * NC + tid];
              m |= (unsigned)(((uint32_t)(b ^ ((b >> 31) & 0x7fffffff)) - l) <= span) << r;
            }
          } else {
            const u64 span = (u64)hi - (u64)lo;
#pragma unroll
            for (int r = 0; r < R; ++r) {
              const i64 b = reinterpret_cast<const i64*>(base)[r * NC + tid];
              m |= (unsigned)(((u64)(b ^ ((b >> 63) & 0x7fffffffffffffffll)) - (u64)lo) <= span) << r;
            }
          }
        } else if (in.b == LKF_4) {
          // lo <= v <= hi as one unsigned compare of (v - lo)
          const uint32_t l = (uint32_t)(int)lo, span = (uint32_t)(int)hi - l;
#pragma unroll
          for (int r = 0; r < R; ++r) {
            const uint32_t v = reinterpret_cast<const uint32_t*>(base)[r * NC + tid];
            m |= (unsigned)((v - l) <= span) << r;
          }
        } else if ((in.b == LKF_8 || in.b == LKF_16) && in.g == 0) {
          const u64 span = (u64)hi - (u64)lo;
          const int stride = in.b == LKF_16 ? 2 : 1;
#pragma unroll
          for (int r = 0; r < R; ++r) {
            const u64 v = reinterpret_cast<const u64*>(base)[stride * (r * NC + tid)];
            m |= (unsigned)((v - (u64)lo) <= span) << r;
          }
        } else {  // unsigned 8-byte / 1-byte kinds
          i64 v[R];
          load_col(in.a, in.b, v);
          const u64 span = (u64)hi - (u64)lo;
#pragma unroll
          for (int r = 0; r < R; ++r) m |= (unsigned)(((u64)v[r] - (u64)lo) <= span) << r;
        }
        if (in.e) {  // inside an OR / NOT tree: (valid & in range, not valid)
          const unsigned all = (1u << R) - 1u;
          const unsigned v = S.cols[in.a].has_valid ? col_valid(in.a) : all;
          mt[msp] = m & v;
          mn[msp] = ~v & all;
          ++msp;
        } else {
          actm &= m;
        }
        return true;
      }
      case FO_MVCC: if constexpr (live<PC>(FO_MVCC)) {
        // RowVersion::is_visible_for (llkv-transaction/src/mvcc.rs:282-334), branch free.  TxnIdManager::status: MAX -> None
        // (not committed), 1 -> Committed, listed ids -> Active/Aborted, anything else -> Committed.  The host keeps 1 out
        // of the non-committed list.
        const u64* cbase = reinterpret_cast<const u64*>(sb + S.cols[in.a].smem_off);
        const u64* dbase = reinterpret_cast<const u64*>(sb + S.cols[in.b].smem_off);
        const u64 txn = p.txn_id, snap = p.snapshot_id;
        const bool own_enabled = txn != 1ull;
        u64 cb[R], db[R];
#pragma unroll
        for (int r = 0; r < R; ++r) {
          cb[r] = cbase[r * NC + tid];
          db[r] = dbase[r * NC + tid];
        }
        // NULL created_by -> TXN_ID_AUTO_COMMIT, NULL deleted_by -> TXN_ID_NONE (llkv-transaction/src/helpers.rs:214-223)
        if (S.cols[in.a].has_valid) {
          const unsigned v = col_valid(in.a);
#pragma unroll
          for (int r = 0; r < R; ++r)
            if (!((v >> r) & 1u)) cb[r] = 1ull;
        }
        if (S.cols[in.b].has_valid) {
          const unsigned v = col_valid(in.b);
#pragma unroll
          for (int r = 0; r < R; ++r)
            if (!((v >> r) & 1u)) db[r] = ~0ull;
        }
        unsigned m = 0;
        if (snap != ~0ull && txn != ~0ull) {
          // creator passes iff cb <= snap (which excludes MAX) and cb is not listed; the deletion does not hide the row
          // iff db > snap (which includes MAX = never deleted) or db is listed.  Rows this transaction created / deleted
          // follow rules (1) and (5).
          // Fast path per pair of row slots of the warp: rows written by auto-commit and never deleted (created_by = 1,
          // deleted_by = MAX: all of a bulk-loaded table) are visible to every snapshot >= 1; when all 32 lanes hold
          // such rows the rule is skipped.  Otherwise the pair goes through the rule together, without branches: the
          // list loop is kept rolled (the host lists only ids <= snapshot, usually none or one).
#pragma unroll
          for (int r0 = 0; r0 < R; r0 += 2) {
            const int r1 = r0 + 1 < R ? r0 + 1 : r0;
            const bool trivial = cb[r0] == 1ull && db[r0] == ~0ull && cb[r1] == 1ull && db[r1] == ~0ull;
            if (__all_sync(LLKV_FULL, trivial)) {
              m |= (snap >= 1ull ? (r1 != r0 ? 3u : 1u) : 0u) << r0;
              continue;
            }
            bool cl0 = false, dl0 = false, cl1 = false, dl1 = false;  // created_by / deleted_by is a non-committed transaction
#pragma unroll 1
            for (uint32_t k = 0; k < p.n_noncommitted; ++k) {
              const u64 id = p.noncommitted[k];
              cl0 |= cb[r0] == id;
              dl0 |= db[r0] == id;
              cl1 |= cb[r1] == id;
              dl1 |= db[r1] == id;
            }
            {
              const bool own_c = own_enabled && cb[r0] == txn, own_d = own_enabled && db[r0] == txn;
              const bool c_ok = cb[r0] <= snap && !cl0, d_ok = db[r0] > snap || dl0;
              m |= (unsigned)(!own_d && (own_c || (c_ok && d_ok))) << r0;
            }
            if (r1 != r0) {
              const bool own_c = own_enabled && cb[r1] == txn, own_d = own_enabled && db[r1] == txn;
              const bool c_ok = cb[r1] <= snap && !cl1, d_ok = db[r1] > snap || dl1;
              m |= (unsigned)(!own_d && (own_c || (c_ok && d_ok))) << r1;
            }
          }
        } else {  // degenerate snapshot ids: the rule as written
#pragma unroll
          for (int r = 0; r < R; ++r) {
            bool c_comm = cb[r] != ~0ull, d_comm = true;
            for (uint32_t k = 0; k < p.n_noncommitted; ++k) {
              const u64 id = p.noncommitted[k];
              c_comm = c_comm && id != cb[r];
              d_comm = d_comm && id != db[r];
            }
            const bool own_c = own_enabled && cb[r] == txn;
            const bool own_d = own_enabled && db[r] == txn;
            const bool others = c_comm && cb[r] <= snap && (db[r] == ~0ull || (!own_d && (!d_comm || db[r] > snap)));
            const bool vis = own_c ? !own_d : others;
            m |= (unsigned)vis << r;
          }
        }
        actm &= m;
        return true;
      }
      case FO_SELECT_DONE: return __any_sync(LLKV_FULL, actm != 0);
      case FO_GROUP: if constexpr (live<PC>(FO_GROUP)) {
        u64 keys[R];
        row_keys(keys);
        const uint32_t FG = S.fg;
        negm = 0;
        if constexpr (Cfg::kPartition) {  // the rows leave this kernel as tuples: scatter()
#pragma unroll
          for (int r = 0; r < R; ++r) pk[r] = keys[r];
          has_slow = false;
          return true;
        }
        if (S.direct_global) {  // high cardinality: a CTA-local table would hold a vanishing share of the keys
          negm = actm;
          has_slow = __any_sync(LLKV_FULL, negm != 0);
          if (has_slow) {
            // The thread's R probes run together, one step of every unresolved row per round (warp-convergent under
            // __any_sync): R table reads in flight per thread instead of R dependent round trips.
            const uint32_t mask = (uint32_t)p.gcap - 1u;  // (the table has < 2^32 rows: gsl[] is 32-bit)
            u64 cur[R];
            unsigned need = 0;
#pragma unroll
            for (int r = 0; r < R; ++r) {
              const bool probe = ((negm >> r) & 1u) && keys[r] != kEmptyKey;
              gsl[r] = probe ? ((uint32_t)mix64(keys[r]) & mask) : (uint32_t)p.gcap;  // the reserved key value has its own row
              cur[r] = probe ? __ldcg(&p.gkeys[gsl[r]]) : 0ull;
              need |= (unsigned)probe << r;
            }
            uint32_t rounds = 0;
            while (__any_sync(LLKV_FULL, need != 0)) {
#pragma unroll
              for (int r = 0; r < R; ++r) {
                if (!((need >> r) & 1u)) continue;
                bool done = cur[r] == keys[r];
                if (!done && cur[r] == kEmptyKey) {
                  const u64 old = atomicCAS(&p.gkeys[gsl[r]], kEmptyKey, keys[r]);
                  done = old == kEmptyKey || old == keys[r];
                }
                if (done) need &= ~(1u << r);
                else {
                  gsl[r] = (gsl[r] + 1u) & mask;
                  cur[r] = __ldcg(&p.gkeys[gsl[r]]);
                }
              }
              if (++rounds > mask && need) {  // every slot seen: the table is full (the run is repeated with a larger one)
                errbits |= FLAG_TABLE_FULL;
#pragma unroll
                for (int r = 0; r < R; ++r)
                  if ((need >> r) & 1u) gsl[r] = (uint32_t)p.gcap;
                need = 0;
              }
            }
          }
          return true;
        }
        unsigned miss = 0;
        if (FG == 4) {
          // Four slots (GROUP BY of at most four expected groups, TPC-H Q1): fully associative, no hashing.  The four
          // keys are two broadcast 16-byte reads; the slot is the index of the matching key.  Half the accumulator
          // footprint of an eight-slot table, which is what bounds the resident warps of a grouped plan.
          const ulonglong2 k01 = *reinterpret_cast<const ulonglong2*>(&tbl[0]);
          const ulonglong2 k23 = *reinterpret_cast<const ulonglong2*>(&tbl[2]);
          // packed keys of at most 31 bits: the low halves decide (a free entry's low half is all ones, no such key has it)
          uint32_t kb_total = 0;
#pragma unroll
          for (uint32_t k = 0; k < (uint32_t)kMaxKeys; ++k)
            if (k < S.n_keys) kb_total += S.key_bits[k] + (S.key_nullable[k] ? 1u : 0u);
          const bool narrow = S.single_wide_key == 0 && kb_total <= 31;
#pragma unroll
          for (int r = 0; r < R; ++r) {
            const u64 K = keys[r];
            bool h0, h1, h2, h3;
            if (narrow) {
              const uint32_t k32 = (uint32_t)K;
              h0 = k32 == (uint32_t)k01.x, h1 = k32 == (uint32_t)k01.y, h2 = k32 == (uint32_t)k23.x, h3 = k32 == (uint32_t)k23.y;
            } else {
              h0 = K == k01.x, h1 = K == k01.y, h2 = K == k23.x, h3 = K == k23.y;
            }
            const uint32_t sl = h0 ? 0u : h1 ? 1u : h2 ? 2u : 3u;
            soff[r] = sl * S.slot_stride;
            if (!((h0 || h1 || h2 || h3) && (narrow || K != kEmptyKey)) && ((actm >> r) & 1u)) miss |= 1u << r;
          }
        } else {
          // Probe without branches: the key's home pair of slots (two adjacent entries, one 16-byte read).  Probe order
          // is home slot, its pair neighbour, then the following pairs, so after the first tiles a key of a
          // low-cardinality GROUP BY is found here even when two keys share a home slot.
#pragma unroll
          for (int r = 0; r < R; ++r) {
            const uint32_t h = hash_key32(keys[r]) & (FG - 1);
            const ulonglong2 pair = *reinterpret_cast<const ulonglong2*>(&tbl[h & ~1u]);
            const u64 k_home = (h & 1u) ? pair.y : pair.x, k_other = (h & 1u) ? pair.x : pair.y;
            const bool hit_home = k_home == keys[r], hit_other = k_other == keys[r];
            const uint32_t sl = hit_home ? h : (h ^ 1u);
            soff[r] = sl * S.slot_stride;
            if (!((hit_home || hit_other) && keys[r] != kEmptyKey) && ((actm >> r) & 1u)) miss |= 1u << r;
          }
        }
        if (__any_sync(LLKV_FULL, miss != 0)) {  // new key, longer collision chain, table full or the reserved key value
#pragma unroll
          for (int r = 0; r < R; ++r) {
            if ((miss >> r) & 1u) {
              const u64 K = keys[r];
              int sl = -1;
              if (K != kEmptyKey) {
                const uint32_t h0 = FG == 4 ? 0u : (hash_key32(K) & (FG - 1));  // four slots: filled in index order
#pragma unroll 1
                for (uint32_t i = 0; i < FG; ++i) {
                  const uint32_t h = ((((h0 >> 1) + (i >> 1)) << 1) | ((h0 ^ i) & 1u)) & (FG - 1);
                  const u64 cur = tbl[h];
                  if (cur == K) { sl = (int)h; break; }
                  if (cur == kEmptyKey) {
                    const u64 old = atomicCAS(&tbl[h], kEmptyKey, K);
                    if (old == kEmptyKey || old == K) { sl = (int)h; break; }
                  }
                }
              }
              soff[r] = sl >= 0 ? (uint32_t)sl * S.slot_stride : 0u;
              if (sl < 0) negm |= 1u << r;
            }
          }
        }
        has_slow = __any_sync(LLKV_FULL, negm != 0);
        if (has_slow) {  // one global-table lookup per row, shared by every aggregate of the plan
#pragma unroll
          for (int r = 0; r < R; ++r)
            if ((negm >> r) & 1u) gsl[r] = (uint32_t)lean_global_slot(p.gkeys, p.gcap, S.n_keys, keys[r], errbits);
        }
        return true;
      }

      case FO_LD_COL: case FO_LD_LIT: case FO_LD_TMP: return true;  // the pre-load above is the whole instruction
      case FO_ST_TMP: if constexpr (live<PC>(FO_ST_TMP)) {
        if constexpr (Cfg::kStatic && PC >= 0) {
          constexpr uint32_t slot = Cfg::code(PC).a;
#pragma unroll
          for (int r = 0; r < R; ++r) treg[slot][r] = acc[r];
        } else {
          i64* t = tmp_base + (size_t)in.a * T;
#pragma unroll
          for (int r = 0; r < R; ++r) t[r * NC + tid] = acc[r];
        }
        return true;
      }
      case FO_OP_COL: if constexpr (live<PC>(FO_OP_COL)) {
        i64 v[R];
        load_col(in.c, in.b, v);
        binop(in.a, v);
        return true;
      }
      case FO_OP_LIT: if constexpr (live<PC>(FO_OP_LIT)) {
        i64 v[R];
        const i64 l = p.lits[in.c];
#pragma unroll
        for (int r = 0; r < R; ++r) v[r] = l;
        binop(in.a, v);
        return true;
      }
      case FO_OP_TMP: if constexpr (live<PC>(FO_OP_TMP)) {
        i64 v[R];
        if constexpr (Cfg::kStatic && PC >= 0) {
          constexpr uint32_t slot = Cfg::code(PC).b;
#pragma unroll
          for (int r = 0; r < R; ++r) v[r] = treg[slot][r];
        } else {
          const i64* t = tmp_base + (size_t)in.b * T;
#pragma unroll
          for (int r = 0; r < R; ++r) v[r] = t[r * NC + tid];
        }
        binop(in.a, v);
        return true;
      }
      case FO_DIVR: if constexpr (live<PC>(FO_DIVR)) {
        if (in.b == 2) {  // 0 <= x < 2^32
          const unsigned d = (unsigned)kPow10U64[in.a], half = d / 2;
#pragma unroll
          for (int r = 0; r < R; ++r) {
            const unsigned x = (unsigned)acc[r];
            const unsigned q = x / d;
            acc[r] = (i64)(q + ((x - q * d) >= half ? 1u : 0u));
          }
        } else if (in.b == 1) {  // x >= 0
          const u64 d = kPow10U64[in.a], half = d / 2;
#pragma unroll
          for (int r = 0; r < R; ++r) {
            const u64 x = (u64)acc[r];
            const u64 q = x / d;
            acc[r] = (i64)(q + ((x - q * d) >= half ? 1ull : 0ull));
          }
        } else {
#pragma unroll
          for (int r = 0; r < R; ++r) acc[r] = div_pow10_round<i64>(acc[r], (int)in.a);
        }
        return true;
      }
      case FO_MULP: if constexpr (live<PC>(FO_MULP)) {
        const i64 m = pow10_i64((int)in.a);
#pragma unroll
        for (int r = 0; r < R; ++r) acc[r] *= m;
        return true;
      }
      case FO_I2F:
#pragma unroll
        for (int r = 0; r < R; ++r) acc[r] = lean_bits(__ll2double_rn(acc[r]));
        return true;
      case FO_D2F: if constexpr (live<PC>(FO_D2F)) {
        const double den = __longlong_as_double(p.lits[in.c]);
#pragma unroll
        for (int r = 0; r < R; ++r) acc[r] = lean_bits(__ll2double_rn(acc[r]) / den);
        return true;
      }

      // ------------------------------------------------------------ aggregates: one private accumulator per thread,
      // CTA-local slot and word.  Ungrouped plans fold the thread's R rows in registers first.  Grouped plans update
      // per row (emit): at once when interpreted, deferred to the end of the tile when specialised (see flush()).
      case FO_COUNT_STAR: case FO_COUNT: if constexpr (live<PC>(FO_COUNT_STAR) || live<PC>(FO_COUNT)) {
        const unsigned lv = in.h ? (actm & valid_mask(in.h)) : actm;  // rows whose operand is not NULL
        if (LLKV_SLOW_HERE) slow_rows(in.op, in.a, ng & lv, in.c);
        const unsigned okm = lv & ~ng;
        const LeanWord lw = S.words[in.b];
        if (!grouped) {
          const unsigned c = __popc(okm);
          if (lw.width == 4) *reinterpret_cast<uint32_t*>(my4 + lw.off) += c;
          else *reinterpret_cast<u64*>(my8 + lw.off) += c;
        } else {
          u64 none[R];
#pragma unroll
          for (int r = 0; r < R; ++r) none[r] = 0;
          emit<PC>(in, okm, none);
        }
        return true;
      }
      case FO_FIRSTROW: case FO_FIRSTVALID: case FO_FIRSTNAN: if constexpr (live<PC>(FO_FIRSTROW) || live<PC>(FO_FIRSTVALID) || live<PC>(FO_FIRSTNAN)) {
        unsigned setm = in.h ? (actm & valid_mask(in.h)) : actm;
        if (in.op == FO_FIRSTNAN) {
#pragma unroll
          for (int r = 0; r < R; ++r) {
            const double d = lean_f64(acc[r]);
            if (d == d) setm &= ~(1u << r);
          }
        }
        if (LLKV_SLOW_HERE) slow_rows(in.op, in.a, setm & ng, in.c);
        setm &= ~ng;
        u64 none[R];
#pragma unroll
        for (int r = 0; r < R; ++r) none[r] = 0;
        emit<PC>(in, setm, none);  // also the ungrouped case: soff[] is zero
        return true;
      }
      case FO_SUM: if constexpr (live<PC>(FO_SUM)) {
        const uint32_t cls = in.a & 3;  // 0: check each value
        const unsigned lv = in.h ? (actm & valid_mask(in.h)) : actm;  // rows whose operand is not NULL
        unsigned fastm = lv & ~ng;
        if (cls == 0 && !Cfg::kPartition) {  // (tuples carry the full value; the table update is exact for any i64)
          unsigned bigm = 0;
#pragma unroll
          for (int r = 0; r < R; ++r)
            if (!(acc[r] < ((i64)1 << 47) && acc[r] > -((i64)1 << 47))) bigm |= 1u << r;
          bigm &= lv;
          slow_rows(FO_SUM, in.a, bigm | (ng & lv), in.c);
          fastm &= ~bigm;
        } else if (LLKV_SLOW_HERE) {
          slow_rows(FO_SUM, in.a, ng & lv, in.c);
        }
        const LeanWord lw = S.words[in.b];
        if (!grouped) {
          i64 x = 0;
#pragma unroll
          for (int r = 0; r < R; ++r)
            if ((fastm >> r) & 1u) x += acc[r];
          if (lw.width == 4) *reinterpret_cast<uint32_t*>(my4 + lw.off) += (uint32_t)x;
          else *reinterpret_cast<u64*>(my8 + lw.off) += (u64)x;
        } else {
          u64 v[R];
#pragma unroll
          for (int r = 0; r < R; ++r) v[r] = (u64)acc[r];
          emit<PC>(in, fastm, v);
        }
        return true;
      }
      case FO_FSUM: if constexpr (live<PC>(FO_FSUM)) {
        const unsigned lv = in.h ? (actm & valid_mask(in.h)) : actm;
        if (LLKV_SLOW_HERE) slow_rows(FO_FSUM, in.a, ng & lv, in.c);
        const unsigned okm = lv & ~ng;
        const LeanWord lw = S.words[in.b];
        if (!grouped) {
          double x = 0.0;
#pragma unroll
          for (int r = 0; r < R; ++r)
            if ((okm >> r) & 1u) x += lean_f64(acc[r]);
          double* a = reinterpret_cast<double*>(my8 + lw.off);
          *a += x;
        } else {
          u64 v[R];
#pragma unroll
          for (int r = 0; r < R; ++r) v[r] = (u64)acc[r];
          emit<PC>(in, okm, v);
        }
        return true;
      }
      case FO_MIN_I: case FO_MAX_I: case FO_MIN_F: case FO_MAX_F: if constexpr (live<PC>(FO_MIN_I) || live<PC>(FO_MAX_I) || live<PC>(FO_MIN_F) || live<PC>(FO_MAX_F)) {
        const bool is_f = in.op == FO_MIN_F || in.op == FO_MAX_F;
        unsigned setm = in.h ? (actm & valid_mask(in.h)) : actm;
        u64 e[R];
#pragma unroll
        for (int r = 0; r < R; ++r) {
          if (is_f) {
            const double d = lean_f64(acc[r]);
            if (d != d) setm &= ~(1u << r);  // NaN never replaces a number (llkv-aggregate/src/lib.rs:1309-1331)
            e[r] = enc_f64(d);
          } else e[r] = enc_i64(acc[r]);
        }
        if (LLKV_SLOW_HERE) slow_rows(in.op, in.a, setm & ng, in.c);
        setm &= ~ng;
        emit<PC>(in, setm, e);  // also the ungrouped case: soff[] is zero
        return true;
      }
      case FO_VALID: if constexpr (live<PC>(FO_VALID)) {
        const unsigned all = (1u << R) - 1u;
        const unsigned v = S.cols[in.a].has_valid ? col_valid(in.a) : all;
        if (in.c) {  // IS NOT NULL / IS NULL / Range(Unbounded, Unbounded) inside a tree; the domain is the valid rows
          mt[msp] = in.b == 0 ? v : in.b == 1 ? (~v & all) : all;
          mn[msp] = ~v & all;
          ++msp;
        } else {
          actm &= in.b ? ~v : v;
        }
        return true;
      }
      case FO_CMP: if constexpr (live<PC>(FO_CMP)) {
        // compute_compare (llkv-compute/src/kernels.rs:269-297) on the 64-bit images; a NULL on either side is NULL
        i64 v[R];
        const uint32_t src = in.b & 0xffu;
        if (src == 0) load_col(in.c, in.b >> 8, v);
        else if (src == 1) {
          const i64 l = p.lits[in.c];
#pragma unroll
          for (int r = 0; r < R; ++r) v[r] = l;
        } else {
          if constexpr (Cfg::kStatic && PC >= 0) {
            constexpr uint32_t slot = Cfg::code(PC).c;
#pragma unroll
            for (int r = 0; r < R; ++r) v[r] = treg[slot < (uint32_t)Cfg::kTmps ? slot : 0][r];
          } else {
            const i64* t = tmp_base + (size_t)in.c * T;
#pragma unroll
            for (int r = 0; r < R; ++r) v[r] = t[r * NC + tid];
          }
        }
        const uint32_t cmp = in.a & 0xfu, kind = in.a >> 4;
        unsigned m = 0;
#pragma unroll
        for (int r = 0; r < R; ++r) {
          bool lt, eq;
          if (kind == 1) {
            lt = (u64)acc[r] < (u64)v[r];
            eq = acc[r] == v[r];
          } else if (kind == 2) {
            const i64 a = f64_total_key(lean_f64(acc[r])), b = f64_total_key(lean_f64(v[r]));
            lt = a < b;
            eq = a == b;
          } else {
            lt = acc[r] < v[r];
            eq = acc[r] == v[r];
          }
          const bool res = cmp == 0 ? eq : cmp == 1 ? !eq : cmp == 2 ? lt : cmp == 3 ? (lt || eq) : cmp == 4 ? !(lt || eq) : !lt;
          m |= (unsigned)res << r;
        }
        const unsigned all = (1u << R) - 1u;
        const unsigned valid = in.h ? valid_mask(in.h) : all;
        mt[msp] = m & valid;
        mn[msp] = ~valid & all;
        ++msp;
        return true;
      }
      case FO_ISNULL: if constexpr (live<PC>(FO_ISNULL)) {
        const unsigned all = (1u << R) - 1u;
        const unsigned valid = in.h ? valid_mask(in.h) : all;
        mt[msp] = (in.a ? valid : ~valid) & all;
        mn[msp] = 0;
        ++msp;
        return true;
      }
      case FO_MASK_AND: case FO_MASK_OR: if constexpr (live<PC>(FO_MASK_AND) || live<PC>(FO_MASK_OR)) {
        // rows: bitmap AND / OR; domain: intersect / unite (llkv-compute/src/program.rs:500-512)
        const unsigned t1 = mt[msp - 2], t0 = mt[msp - 1], n1 = mn[msp - 2], n0 = mn[msp - 1];
        mt[msp - 2] = in.op == FO_MASK_AND ? (t1 & t0) : (t1 | t0);
        mn[msp - 2] = in.op == FO_MASK_AND ? (n1 | n0) : (n1 & n0);
        --msp;
        return true;
      }
      case FO_MASK_NOT:  // domain - rows (llkv-scan/src/predicate.rs:167-186)
        mt[msp - 1] = ~mn[msp - 1] & ~mt[msp - 1] & ((1u << R) - 1u);
        return true;
      case FO_MASK_LIT:
        mt[msp] = in.a ? (1u << R) - 1u : 0u;
        mn[msp] = 0;
        ++msp;
        return true;
      case FO_MASK_FILTER:
        actm &= mt[--msp];
        return true;
      case FO_END:
        if constexpr (Cfg::kStatic && PC >= 0 && !Cfg::kPartition) flush();
        return false;
      default: errbits |= FLAG_BAD_PLAN; return false;
    }
  }

  // One row's update of one accumulator word (`in` is the aggregate instruction, `v` its operand for this row).
  __device__ __forceinline__ void apply_row(const FInstr& in, bool on, u64 v, int r) {
    if (!on) return;
    const LeanWord lw = S.words[in.b];
    switch (in.op) {
      case FO_COUNT_STAR: case FO_COUNT:
        if (lw.width == 4) *reinterpret_cast<uint32_t*>(my4 + lw.off + soff[r]) += 1u;
        else *reinterpret_cast<u64*>(my8 + lw.off + soff[r]) += 1ull;
        break;
      case FO_FIRSTROW: case FO_FIRSTVALID: case FO_FIRSTNAN:
        if (lw.width == 4) {  // launch-relative row index
          uint32_t* a = reinterpret_cast<uint32_t*>(my4 + lw.off + soff[r]);
          const uint32_t cand = rel0 + (uint32_t)(r * NC), cur = *a;
          *a = cand < cur ? cand : cur;
        } else {
          u64* a = reinterpret_cast<u64*>(my8 + lw.off + soff[r]);
          const u64 cand = row0 + (u64)(r * NC + tid), cur = *a;
          *a = cand < cur ? cand : cur;
        }
        break;
      case FO_SUM:
        if (lw.width == 4) *reinterpret_cast<uint32_t*>(my4 + lw.off + soff[r]) += (uint32_t)v;
        else *reinterpret_cast<u64*>(my8 + lw.off + soff[r]) += v;
        break;
      case FO_FSUM: {
        double* a = reinterpret_cast<double*>(my8 + lw.off + soff[r]);
        *a += lean_f64((i64)v);
        break;
      }
      default: {  // FO_MIN_* / FO_MAX_* on order-preserving encodings
        const bool is_min = in.op == FO_MIN_I || in.op == FO_MIN_F;
        u64* a = reinterpret_cast<u64*>(my8 + lw.off + soff[r]);
        const u64 cur = *a;
        *a = (is_min ? v < cur : v > cur) ? v : cur;
        break;
      }
    }
  }

  // Interpreted: the update happens at once, aggregate by aggregate.  Specialised + grouped: operands and row masks are
  // parked in registers (one entry per aggregate instruction, indexed at compile time) and applied by flush() row by
  // row: the words of one row are provably distinct addresses, so their loads and stores overlap instead of forming one
  // read-modify-write chain per aggregate (two rows of a thread may share a slot, which serialises them).
  template <int PC>
  __device__ __forceinline__ void emit(const FInstr& in, unsigned mask, const u64 (&v)[R]) {
    if constexpr (Cfg::kStatic && PC >= 0 && Cfg::kDefer) {
      constexpr int k = lean_stash_index<Cfg>(PC);
      stash_m[k] = mask;
#pragma unroll
      for (int r = 0; r < R; ++r) stash_v[k][r] = v[r];
    } else {
#pragma unroll
      for (int r = 0; r < R; ++r) apply_row(in, (mask >> r) & 1u, v[r], r);
    }
  }

  template <int PC>
  __device__ __forceinline__ void flush_row(int r) {
    if constexpr (Cfg::kStatic) {
      constexpr FInstr in = Cfg::code(PC);
      if constexpr (lean_is_aggregate(in.op)) {
        constexpr int k = lean_stash_index<Cfg>(PC);
        apply_row(in, (stash_m[k] >> r) & 1u, stash_v[k][r], r);
      }
      if constexpr (in.op != FO_END && PC + 1 < kMaxFastInstr) flush_row<PC + 1>(r);
    }
  }
  __device__ __forceinline__ void flush() {
    if constexpr (Cfg::kStatic) {
      if constexpr (Cfg::kDefer) {
#pragma unroll
        for (int r = 0; r < R; ++r) flush_row<0>(r);
      }
    }
  }

  // ---------------------------------------------------------------------------------- partitioned GROUP BY (pass 1)
  // Every consumer thread calls scatter() once per tile (also warps that left the program early: their actm is 0).
  // The tile's selected rows become tuples (key, row id, operands), are counting-sorted by hash partition in shared
  // memory and leave as one run per partition and field; space in a partition is reserved with one atomic per
  // partition and tile, so each partition's stream grows sequentially and full lines reach DRAM.
  __device__ __forceinline__ uint32_t part_of(u64 K) const {
    return K == kEmptyKey ? 0u : (uint32_t)((mix64(K) & (p.gcap - 1)) >> p.part_shift);
  }
  template <int PC>
  __device__ __forceinline__ void stage_row(u64* stage, uint32_t idx, int r) {
    if constexpr (Cfg::kStatic) {
      constexpr FInstr in = Cfg::code(PC);
      if constexpr (lean_takes_operand(in.op)) stage[(uint32_t)lean_field_index<Cfg>(PC) * T + idx] = stash_v[lean_stash_index<Cfg>(PC)][r];
      if constexpr (in.op != FO_END && PC + 1 < kMaxFastInstr) stage_row<PC + 1>(stage, idx, r);
    }
  }
  // a tuple that found its partition full: applied to the table here (the per-row path of direct_global plans)
  template <int PC>
  __device__ __forceinline__ void apply_tuple(const u64* stage, uint32_t i, u64 gs, u64 row) {
    if constexpr (Cfg::kStatic) {
      constexpr FInstr in = Cfg::code(PC);
      if constexpr (lean_is_aggregate(in.op)) {
        u64 v = 0;
        if constexpr (lean_takes_operand(in.op)) v = stage[(uint32_t)lean_field_index<Cfg>(PC) * T + i];
        lean_apply_field(&p.gwords[gs * S.n_gwords + in.c], in.op, in.a, v, row);
      }
      if constexpr (in.op != FO_END && PC + 1 < kMaxFastInstr) apply_tuple<PC + 1>(stage, i, gs, row);
    }
  }
  // ---------------------------------------------------------------------------------- packed tuples (partition == 2)
  // One 64-bit word per selected row: key | launch-relative row | SUM operands.  The CTA appends the tuples of
  // pack_batch / tile_rows tiles to a batch buffer in shared memory (no barrier: one shared-memory atomic per warp and tile),
  // then scatters the batch: count per partition, one global atomic per non-empty partition reserves the space, every
  // tuple goes to its place with a streaming store.  Partitions are small enough (a few thousand groups) for
  // partition_fold_kernel to aggregate each of them in shared memory, so no row of the scan ever updates the table in
  // global memory; the batch makes the runs per partition long enough for L2 to assemble full lines.
  __device__ __forceinline__ uint32_t part_of_packed(u64 t) const {
    const u64 K = t & ((1ull << S.pack_key_bits) - 1);
    return p.part_dense ? (uint32_t)(K >> p.part_shift) : (uint32_t)((mix64(K) & (p.gcap - 1)) >> p.part_shift);
  }
  template <int PC>
  __device__ __forceinline__ u64 pack_ops(int r, uint32_t shift) const {
    if constexpr (Cfg::kStatic) {
      constexpr FInstr in = Cfg::code(PC);
      u64 v = 0;
      uint32_t next = shift;
      if constexpr (lean_takes_operand(in.op)) {
        v = stash_v[lean_stash_index<Cfg>(PC)][r] << shift;
        next = shift + S.pack_op_bits[lean_field_index<Cfg>(PC) - 2];
      }
      if constexpr (in.op != FO_END && PC + 1 < kMaxFastInstr) v |= pack_ops<PC + 1>(r, next);
      return v;
    } else {
      return 0;
    }
  }
  // a tuple that found its partition full (skewed keys): applied to the table here, word by word
  template <int PC>
  __device__ __forceinline__ void apply_packed(u64 t, u64 gs, u64 row, uint32_t shift) {
    if constexpr (Cfg::kStatic) {
      constexpr FInstr in = Cfg::code(PC);
      uint32_t next = shift;
      if constexpr (lean_is_aggregate(in.op)) {
        u64 v = 0;
        if constexpr (lean_takes_operand(in.op)) {
          const uint32_t bits = S.pack_op_bits[lean_field_index<Cfg>(PC) - 2];
          v = (t >> shift) & ((1ull << bits) - 1);
          next = shift + bits;
        }
        lean_slow_accumulate(&p.gwords[gs * S.n_gwords + in.c], in.op, in.a, (i64)v, row);
      }
      if constexpr (in.op != FO_END && PC + 1 < kMaxFastInstr) apply_packed<PC + 1>(t, gs, row, next);
    }
  }
  // Shared-memory layout of the packed form (smem_part_off): u32 fill, u32 pad, u32 off[parts], u32 gdelta[parts],
  // u64 buf[pack_batch], u16 order[pack_batch].
  __device__ __forceinline__ void flush_packed() {
    if constexpr (Cfg::kPacked) {
      uint32_t* const s_fill = reinterpret_cast<uint32_t*>(part_smem);
      const uint32_t P = S.pack_parts;
      uint32_t* const off = s_fill + 2;     // per partition: count, then first sorted position, then one past its last
      uint32_t* const gdelta = off + P;     // reserved position in the partition's global stream minus its first sorted position
      const u64* const buf = reinterpret_cast<const u64*>(gdelta + P);
      unsigned short* const order = reinterpret_cast<unsigned short*>(const_cast<u64*>(buf) + S.pack_batch);
      uint32_t* const s_scan = reinterpret_cast<uint32_t*>(order + S.pack_batch);  // one partial sum per consumer warp
      lean_consumer_barrier(NC);  // every append of the batch is in the buffer
      const uint32_t n = *s_fill;
      for (uint32_t q = (uint32_t)tid; q < P; q += (uint32_t)NC) off[q] = 0;
      lean_consumer_barrier(NC);
      if (tid == 0) *s_fill = 0;
      for (uint32_t i = (uint32_t)tid; i < n; i += (uint32_t)NC) atomicAdd(&off[part_of_packed(buf[i])], 1u);
      lean_consumer_barrier(NC);
      // exclusive prefix of the counts (every thread owns a contiguous share of the partitions) + one global atomic per
      // non-empty partition reserving the batch's share of its stream
      {
        const uint32_t per = (P + (uint32_t)NC - 1) / (uint32_t)NC;
        const uint32_t lo = (uint32_t)tid * per, hi = lo + per < P ? lo + per : P;
        uint32_t sum = 0;
        for (uint32_t q = lo; q < hi; ++q) sum += off[q];
        const int lane = tid & 31, wid = tid >> 5;
        uint32_t inc = sum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const uint32_t y = __shfl_up_sync(LLKV_FULL, inc, o);
          if (lane >= o) inc += y;
        }
        if (lane == 31) s_scan[wid] = inc;
        lean_consumer_barrier(NC);
        uint32_t wbase = 0;
        for (int w = 0; w < wid; ++w) wbase += s_scan[w];
        uint32_t run = wbase + inc - sum;
        for (uint32_t q = lo; q < hi; ++q) {
          const uint32_t c = off[q];
          const uint32_t g = c ? atomicAdd(&p.part_cursor[q], c) : 0u;
          off[q] = run;
          gdelta[q] = g - run;
          run += c;
        }
      }
      lean_consumer_barrier(NC);
      // sorted order: position -> index of the tuple in the buffer
      for (uint32_t i = (uint32_t)tid; i < n; i += (uint32_t)NC) order[atomicAdd(&off[part_of_packed(buf[i])], 1u)] = (unsigned short)i;
      lean_consumer_barrier(NC);
      // consecutive threads write consecutive tuples of a partition: whole sectors, few pages per warp
      const u64 cap = p.part_cap;
      const uint32_t kb = S.pack_key_bits, rb = S.pack_row_bits;
      for (uint32_t j = (uint32_t)tid; j < n; j += (uint32_t)NC) {
        const u64 t = buf[order[j]];
        const uint32_t q = part_of_packed(t);
        const u64 pos = (u64)(uint32_t)(gdelta[q] + j);
        if (pos < cap) {
          __stcs(&p.part_out[(u64)q * cap + pos], t);  // read once, by the next kernel
        } else {
          const u64 K = t & ((1ull << kb) - 1);
          const u64 gs = lean_global_slot(p.gkeys, p.gcap, S.n_keys, K, errbits);
          const u64 row = p.row_origin + p.first_tile * (u64)T + ((t >> kb) & ((1ull << rb) - 1));
          apply_packed<0>(t, gs, row, kb + rb);
        }
      }
      lean_consumer_barrier(NC);  // the buffer is free for the next batch
    }
  }
  __device__ __forceinline__ void scatter_packed() {
    if constexpr (Cfg::kPacked) {
      uint32_t* const s_fill = reinterpret_cast<uint32_t*>(part_smem);
      u64* const buf = reinterpret_cast<u64*>(s_fill + 2 + 2u * S.pack_parts);
      const int lane = tid & 31;
      const uint32_t c = (uint32_t)__popc(actm);
      uint32_t inc = c;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const uint32_t y = __shfl_up_sync(LLKV_FULL, inc, o);
        if (lane >= o) inc += y;
      }
      uint32_t wbase = 0;
      if (lane == 31 && inc) wbase = atomicAdd(s_fill, inc);
      wbase = __shfl_sync(LLKV_FULL, wbase, 31);
      uint32_t at = wbase + inc - c;
      const uint32_t kb = S.pack_key_bits, rb = S.pack_row_bits;
#pragma unroll
      for (int r = 0; r < R; ++r)
        if ((actm >> r) & 1u) buf[at++] = pk[r] | ((u64)(rel0 + (uint32_t)(r * NC)) << kb) | pack_ops<0>(r, kb + rb);
      if (++batch_tiles == S.pack_batch / T) {  // the next tile might not fit: every consumer thread counts the same tiles
        flush_packed();
        batch_tiles = 0;
      }
    }
  }

  __device__ __forceinline__ void scatter() {
    if constexpr (Cfg::kPacked) {
      scatter_packed();
    } else if constexpr (Cfg::kPartition) {
      uint32_t* const s_cnt = reinterpret_cast<uint32_t*>(part_smem);
      uint32_t* const s_off = s_cnt + (kMaxPartitions + 1);
      uint32_t* const s_gb = s_off + (kMaxPartitions + 1);
      u64* const stage = reinterpret_cast<u64*>(s_gb + (kMaxPartitions + 1) + 1);
      const uint32_t P = 1u << p.part_bits;
      uint32_t part[R], pos[R];
#pragma unroll
      for (int r = 0; r < R; ++r) {
        part[r] = part_of(pk[r]);
        pos[r] = 0;
        if ((actm >> r) & 1u) pos[r] = atomicAdd(&s_cnt[part[r]], 1u);
      }
      lean_consumer_barrier(NC);
      for (uint32_t q = (uint32_t)tid; q < P; q += (uint32_t)NC) {
        const uint32_t c = s_cnt[q];
        s_gb[q] = c ? atomicAdd(&p.part_cursor[q], c) : 0u;
      }
      if (tid < 32) {  // exclusive prefix of the counts: each lane sums a contiguous share, then a warp scan
        const uint32_t per = (P + 31u) >> 5;
        const uint32_t lo = (uint32_t)tid * per;
        uint32_t sum = 0;
        for (uint32_t q = lo; q < lo + per && q < P; ++q) sum += s_cnt[q];
        uint32_t inc = sum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const uint32_t y = __shfl_up_sync(LLKV_FULL, inc, o);
          if (tid >= o) inc += y;
        }
        uint32_t run = inc - sum;
        for (uint32_t q = lo; q < lo + per && q < P; ++q) {
          s_off[q] = run;
          run += s_cnt[q];
        }
        if (tid == 31) s_off[P] = inc;  // tuples of the tile
      }
      lean_consumer_barrier(NC);
#pragma unroll
      for (int r = 0; r < R; ++r)
        if ((actm >> r) & 1u) {
          const uint32_t idx = s_off[part[r]] + pos[r];
          stage[idx] = pk[r];
          stage[T + idx] = row0 + (u64)(r * NC + tid);
          stage_row<0>(stage, idx, r);
        }
      lean_consumer_barrier(NC);
      const uint32_t total = s_off[P];
      const u64 cap = p.part_cap;
      const uint32_t NF = S.n_fields;
      for (uint32_t i = (uint32_t)tid; i < total; i += (uint32_t)NC) {
        const u64 K = stage[i];
        const uint32_t q = part_of(K);
        const u64 j = (u64)s_gb[q] + (i - s_off[q]);
        if (j < cap) {
          u64* out = p.part_out + (u64)q * NF * cap + j;
          for (uint32_t f = 0; f < NF; ++f) __stcs(&out[(u64)f * cap], stage[f * T + i]);  // read once, by the next kernel
        } else {
          const u64 gs = lean_global_slot(p.gkeys, p.gcap, S.n_keys, K, errbits);
          apply_tuple<0>(stage, i, gs, stage[T + i]);
        }
      }
      for (uint32_t q = (uint32_t)tid; q < P; q += (uint32_t)NC) s_cnt[q] = 0;
      lean_consumer_barrier(NC);
    }
  }

  // specialised: one instantiation of step() per program position, the instruction is a compile-time constant
  // Grouped plans with CTA-local slots (kSplitSlow): the instructions after GROUP exist twice.  A warp whose rows all
  // found a slot (every tile of a low-cardinality GROUP BY after the first few) runs the copy without the per-aggregate
  // "rows for the global table?" branches: one branch per tile instead of one taken branch over cold code per aggregate.
  template <int PC, bool SLOW = true>
  __device__ __forceinline__ void run_static() {
    if constexpr (Cfg::kStatic) {
      constexpr FInstr in = Cfg::code(PC);
      if (!step<PC, SLOW>(in)) return;
      if constexpr (in.op != FO_END && PC + 1 < kMaxFastInstr) {
        if constexpr (in.op == FO_GROUP && Cfg::kSplitSlow) {
          if (has_slow) run_static<PC + 1, true>();
          else run_static<PC + 1, false>();
        } else {
          run_static<PC + 1, SLOW>();
        }
      }
    }
  }
  // interpreted: the next instruction is fetched early so the constant-cache latency overlaps this instruction's work
  __device__ __forceinline__ void run_dynamic() {
    uint32_t pc = 0;
    FInstr in = S.code[0];
    while (true) {
      const FInstr nxt = S.code[pc + 1];
      if (!step<-1>(in)) break;
      in = nxt;
      ++pc;
    }
  }
};

// The publishing epilogue (LeanPlan::publish): every CTA has folded into the table; the one that draws the last ticket
// copies the status word and the table to page-locked host memory and re-arms the state for the next step, so a repeated
// step is this one kernel.  `s_flag`: a shared word the fold no longer reads.  A global ticket and a plain shared store
// (no shared atomics).
__device__ __forceinline__ void lean_publish(const LeanPlan& p, const LeanShape& S, u64* s_flag) {
  const uint32_t tid = threadIdx.x;
  __threadfence();  // this thread's table updates and status bits, before its CTA's ticket
  __syncthreads();
  if (tid == 0) *s_flag = atomicAdd(p.ticket, 1u) == gridDim.x - 1 ? 1ull : 0ull;
  __syncthreads();
  if (!*s_flag) return;
  __threadfence();
  const uint32_t n_words = (uint32_t)(p.gcap + 2) * S.n_gwords, n_keys = S.n_keys ? (uint32_t)p.gcap : 0u;
  u64* const out = p.publish;
  if (tid == 0) out[0] = __ldcg(p.flags);
  for (uint32_t i = tid; i < n_words; i += blockDim.x) out[1 + i] = __ldcg(&p.gwords[i]);
  for (uint32_t i = tid; i < n_keys; i += blockDim.x) out[1 + n_words + i] = __ldcg(&p.gkeys[i]);
  __threadfence_system();
  __syncthreads();  // every read of the state is done before it is re-armed
  for (uint32_t i = tid; i < n_words; i += blockDim.x) p.gwords[i] = gword_initial(p.gclass[i % S.n_gwords]);
  for (uint32_t i = tid; i < n_keys; i += blockDim.x) p.gkeys[i] = kEmptyKey;
  if (tid == 0) {
    *p.flags = 0;
    *p.ticket = 0;
  }
}

template <int R, class Cfg>
__device__ __forceinline__ void lean_body(const LeanPlan& p) {
  extern __shared__ __align__(128) unsigned char smem[];
  const LeanShape& S = Cfg::shape(p);
  const int tid = threadIdx.x;
  const int NC = (int)S.nc;  // consumer threads (blockDim.x - 32)
  const int lane = tid & 31;
  const int warp = tid >> 5;
  const int n_cwarps = NC >> 5;
  const bool is_producer = warp == n_cwarps;

  u64* const full_bar = reinterpret_cast<u64*>(smem + S.smem_bar_off);
  u64* const empty_bar = full_bar + S.stages;
  unsigned char* const stage0 = smem + S.smem_stage_off;
  unsigned char* const accb = smem + S.smem_acc_off;               // [slot][word][consumer thread]
  u64* const tbl = reinterpret_cast<u64*>(smem + S.smem_tbl_off);  // CTA-local group keys, then the slots' global rows
  u64* const gslot_s = tbl + S.fg;

  const uint32_t FG = S.fg;
  const uint32_t NW = S.n_words;
  const uint32_t ST = S.stages;
  const bool grouped = S.n_keys != 0;

  // accumulator init: MIN-class words start at all ones
  if (tid < NC) {
    for (uint32_t g = 0; g < FG; ++g)
      for (uint32_t w = 0; w < NW; ++w) {
        const LeanWord lw = S.words[w];
        unsigned char* blk = accb + g * S.slot_stride + lw.off;
        const bool min_class = lw.kind == FK_MIN || lw.kind == FK_MIN128_HI;
        if (lw.width == 4) reinterpret_cast<uint32_t*>(blk)[tid] = min_class ? 0xffffffffu : 0u;
        else if (lw.width == 8) reinterpret_cast<u64*>(blk)[tid] = min_class ? ~0ull : 0ull;
      }
  }
  for (uint32_t g = tid; g < FG; g += blockDim.x) tbl[g] = grouped ? kEmptyKey : 0ull;
  if constexpr (Cfg::kPacked) {
    uint32_t* const s_fill = reinterpret_cast<uint32_t*>(smem + S.smem_part_off);
    for (uint32_t q = tid; q < 2u + 2u * S.pack_parts; q += blockDim.x) s_fill[q] = 0;
  } else if constexpr (Cfg::kPartition) {
    uint32_t* const s_cnt = reinterpret_cast<uint32_t*>(smem + S.smem_part_off);
    for (uint32_t q = tid; q < 3u * (kMaxPartitions + 1) + 1u; q += blockDim.x) s_cnt[q] = 0;
  }
  if (tid == 0) {
    for (uint32_t s = 0; s < ST; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], (uint32_t)n_cwarps);
    }
    mbar_fence_init();
  }
  __syncthreads();

  const uint32_t T = S.tile_rows;
  const uint32_t n_tiles = (uint32_t)p.n_tiles;  // < 2^32 / T per launch (the host splits longer scans)
  const uint32_t my_tiles = (n_tiles > blockIdx.x) ? (n_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
  const u64 base_row = p.first_tile * (u64)T;
  uint32_t errbits = 0;

  if (is_producer) {
    // ---------------------------------------------------------------- producer: TMA bulk copies, `stages` tiles in flight
    if (lane == 0) {
      uint32_t s = 0, round = 0;
      for (uint32_t li = 0, rt = blockIdx.x; li < my_tiles; ++li, rt += gridDim.x) {
        const u64 tile = S.use_tile_list ? (u64)p.tile_list[rt] : p.first_tile + rt;  // (read before the wait: off the critical path)
        if (round) mbar_wait_parked(&empty_bar[s], (round - 1) & 1);
        unsigned char* sbuf = stage0 + (size_t)s * S.stage_bytes;
        mbar_arrive_expect_tx(&full_bar[s], S.tx_bytes);
#pragma unroll
        for (uint32_t c = 0; c < (uint32_t)kMaxCols; ++c) {
          if (c < S.n_cols) {
            const uint32_t bytes = T * S.cols[c].elem_bytes;
            bulk_g2s(sbuf + S.cols[c].smem_off, reinterpret_cast<const unsigned char*>(p.col_base[c]) + tile * (u64)bytes, bytes, &full_bar[s]);
            if (S.cols[c].has_valid) bulk_g2s(sbuf + S.cols[c].vsmem_off, p.col_valid[c] + tile * (u64)(T >> 3), T >> 3, &full_bar[s]);
          }
        }
        if (S.has_exists) bulk_g2s(sbuf + S.exists_smem_off, p.exists_bits + tile * (u64)(T >> 3), T >> 3, &full_bar[s]);
        if (++s == ST) {
          s = 0;
          ++round;
        }
      }
    }
  } else {
    // ---------------------------------------------------------------- consumers
    LeanTile<R, Cfg> t(p, S, smem, tid, NC);
    const uint32_t begin_rel = (uint32_t)(p.row_begin - base_row);
    const u64 end64 = p.row_end - base_row;
    const uint32_t end_rel = end64 > 0xffffffffull ? 0xffffffffu : (uint32_t)end64;
    uint32_t s = 0, round = 0;
    for (uint32_t li = 0, rt = blockIdx.x; li < my_tiles; ++li, rt += gridDim.x) {
      const uint32_t rel_tile = S.use_tile_list ? p.tile_list[rt] - (uint32_t)p.first_tile : rt;  // (requested before the wait)
      mbar_wait_parked(&full_bar[s], round & 1);
      t.begin_tile(stage0 + (size_t)s * S.stage_bytes, rel_tile * T, base_row, begin_rel, end_rel);
      if constexpr (Cfg::kStatic) t.template run_static<0>();
      else t.run_dynamic();
      if constexpr (Cfg::kPartition) t.scatter();
      __syncwarp();
      if (lane == 0) mbar_arrive(&empty_bar[s]);  // this warp is done with the stage
      if (++s == ST) {
        s = 0;
        ++round;
      }
    }
    if constexpr (Cfg::kPacked) t.flush_packed();  // what the last tiles left in the batch buffer
    errbits = t.errbits;
  }

  // ---------------------------------------------------------------- fold the threads' accumulators into the global group table
  __syncthreads();
  const int n_warps = (NC >> 5) + 1;
  for (uint32_t g = tid; g < FG; g += blockDim.x) {
    const u64 K = tbl[g];
    u64 gs = ~0ull;
    if (!grouped) gs = 0;
    else if (K != kEmptyKey) gs = lean_global_slot(p.gkeys, p.gcap, S.n_keys, K, errbits);
    gslot_s[g] = gs;
  }
  __syncthreads();
  for (uint32_t i = (uint32_t)warp; i < FG * NW; i += (uint32_t)n_warps) {
    const uint32_t g = i / NW, w = i % NW;
    const u64 gs = gslot_s[g];
    if (gs == ~0ull) continue;
    const LeanWord lw = S.words[w];
    if (lw.kind == FK_SKIP) continue;
    const unsigned char* blk = accb + g * S.slot_stride + lw.off;
    u64* grow = &p.gwords[gs * S.n_gwords];
    switch (lw.kind) {
      case FK_COUNT: {
        u64 s = 0;
        for (int t = lane; t < NC; t += 32) s += lw.width == 4 ? (u64)reinterpret_cast<const uint32_t*>(blk)[t] : reinterpret_cast<const u64*>(blk)[t];
        for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(LLKV_FULL, s, o);
        if (lane == 0 && s) atomicAdd(&grow[lw.gword], s);
        break;
      }
      case FK_SUM_I64: case FK_SUM_I128: {
        i128 t128 = 0;
        for (int t = lane; t < NC; t += 32)
          t128 += lw.width == 4 ? (i128)reinterpret_cast<const uint32_t*>(blk)[t] : (i128)reinterpret_cast<const i64*>(blk)[t];
        for (int o = 16; o; o >>= 1) {
          const u64 olo = __shfl_xor_sync(LLKV_FULL, (u64)t128, o);
          const u64 ohi = __shfl_xor_sync(LLKV_FULL, (u64)((u128)t128 >> 64), o);
          t128 += (i128)(((u128)ohi << 64) | (u128)olo);
        }
        if (lane == 0 && t128 != 0) {
          if (lw.kind == FK_SUM_I64) gadd_sum_i64(&grow[lw.gword], t128);
          else gadd_sum_i128(&grow[lw.gword], t128);
        }
        break;
      }
      case FK_FSUM: {
        double s = 0.0;
        for (int t = lane; t < NC; t += 32) s += reinterpret_cast<const double*>(blk)[t];
        for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(LLKV_FULL, s, o);
        if (lane == 0) atomicAdd(reinterpret_cast<double*>(&grow[lw.gword]), s);
        break;
      }
      case FK_MIN: {
        u64 s = ~0ull;
        for (int t = lane; t < NC; t += 32) {
          u64 v;
          if (lw.width == 4) {
            const uint32_t x = reinterpret_cast<const uint32_t*>(blk)[t];
            v = x == 0xffffffffu ? ~0ull : (lw.rowrel ? p.row_origin + base_row + x : (u64)x);
          } else v = reinterpret_cast<const u64*>(blk)[t];
          s = v < s ? v : s;
        }
        for (int o = 16; o; o >>= 1) {
          const u64 y = __shfl_xor_sync(LLKV_FULL, s, o);
          s = y < s ? y : s;
        }
        if (lane == 0 && s != ~0ull) atomicMin(&grow[lw.gword], s);
        break;
      }
      case FK_MAX: {
        u64 s = 0ull;
        for (int t = lane; t < NC; t += 32) {
          const u64 v = reinterpret_cast<const u64*>(blk)[t];
          s = v > s ? v : s;
        }
        for (int o = 16; o; o >>= 1) {
          const u64 y = __shfl_xor_sync(LLKV_FULL, s, o);
          s = y > s ? y : s;
        }
        if (lane == 0) atomicMax(&grow[lw.gword], s);
        break;
      }
      case FK_MIN128_HI: case FK_MAX128_HI: {  // thread state: one order-preserving u64 of an i64-ranged Decimal128
        const bool is_max = lw.kind == FK_MAX128_HI;
        u64 s = is_max ? 0ull : ~0ull;
        for (int t = lane; t < NC; t += 32) {
          const u64 v = reinterpret_cast<const u64*>(blk)[t];
          s = is_max ? (v > s ? v : s) : (v < s ? v : s);
        }
        for (int o = 16; o; o >>= 1) {
          const u64 y = __shfl_xor_sync(LLKV_FULL, s, o);
          s = is_max ? (y > s ? y : s) : (y < s ? y : s);
        }
        if (lane == 0 && s != (is_max ? 0ull : ~0ull)) {
          const i64 v = (i64)(s ^ 0x8000000000000000ull);
          gmin128(&grow[lw.gword], enc_i64(v >> 63), (u64)v, is_max);
        }
        break;
      }
      default: errbits |= FLAG_BAD_PLAN; break;
    }
  }
  if (errbits) atomicOr(p.flags, errbits);
  if constexpr (!Cfg::kPartition) {
    if (p.publish) lean_publish(p, S, gslot_s);
  }
}

}  // namespace llkv

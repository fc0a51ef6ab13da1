// scan_kernel.cu — the fused scan -> predicate -> MVCC -> projection -> aggregate kernel for sm_100a.
//
// One persistent CTA per SM slot walks row tiles of tile_rows = blockDim.x * R rows.  Thread 0 keeps
// (stages-1) tiles in flight with cp.async.bulk (TMA 1-D bulk copies, one per column per tile) completing on
// an mbarrier per stage; all threads then run the Plan's stack program over their R rows of the tile with the
// two top-of-stack entries in registers.  Aggregates go to per-thread accumulators in shared memory
// (CTA-local group slots), folded into the global group table once per CTA at the end.  No column byte is read
// from HBM more than once; nothing is materialised.
//
// Two instantiations of the interpreter exist: NARROW (values in 64 bits — Decimal128 columns whose values
// fit in i64; any value or intermediate that does not fit raises FLAG_NARROW_FAIL and the host reruns the pass)
// and WIDE (full i128 arithmetic).  Results are identical whenever the narrow pass does not raise the flag.
//
// Replaces, for one pass: the typed filter loops (llkv-column-map/src/store/scan/filter.rs:605-958), the
// predicate interpreter (llkv-scan/src/predicate.rs:32-193), the MVCC row loop
// (llkv-transaction/src/helpers.rs:178-245), row gather + ScalarEvaluator (llkv-scan/src/row_stream.rs:451-623,
// llkv-compute/src/eval.rs:565-750) and AggregateAccumulator::update (llkv-aggregate/src/lib.rs:759-1477).
#include "device_util.cuh"
#include "plan.h"

namespace llkv {

template <bool WIDE>
struct VT {
  typedef i64 type;
};
template <>
struct VT<true> {
  typedef i128 type;
};

__device__ __forceinline__ double as_f64(i64 v) { return __longlong_as_double(v); }
__device__ __forceinline__ double as_f64(i128 v) { return __longlong_as_double((i64)v); }
__device__ __forceinline__ i64 f64_bits(double d) { return __double_as_longlong(d); }

// ------------------------------------------------------------------ the interpreter
template <bool WIDE, int R>
__global__ void __launch_bounds__(512) scan_kernel(const Plan* __restrict__ gplan) {
  typedef typename VT<WIDE>::type V;
  extern __shared__ __align__(128) unsigned char smem[];
  const int tid = threadIdx.x;
  const int NT = blockDim.x;
  const int lane = tid & 31;
  const int warp = tid >> 5;

  // ---- stage the plan in shared memory
  Plan& p = *reinterpret_cast<Plan*>(smem);
  {
    const uint32_t n4 = sizeof(Plan) / 4;
    const uint32_t* src = reinterpret_cast<const uint32_t*>(gplan);
    uint32_t* dst = reinterpret_cast<uint32_t*>(smem);
    for (uint32_t i = tid; i < n4; i += NT) dst[i] = src[i];
  }
  __syncthreads();

  u64* const bars = reinterpret_cast<u64*>(smem + p.smem_bar_off);
  unsigned char* const stage0 = smem + p.smem_stage_off;
  u64* const acc = reinterpret_cast<u64*>(smem + p.smem_acc_off);
  V* const spill = reinterpret_cast<V*>(smem + p.smem_spill_off);
  u64* const tbl = reinterpret_cast<u64*>(smem + p.smem_tbl_off);

  const uint32_t FG = p.fast_groups;
  const uint32_t NFW = p.n_fast_words;
  // ---- init per-thread accumulators, CTA group table, barriers
  for (uint32_t g = 0; g < FG; ++g)
    for (uint32_t w = 0; w < NFW; ++w) {
      const uint8_t k = p.fast[w].kind;
      u64 init = 0;
      if (k == FK_MIN || k == FK_MIN128_HI) init = ~0ull;
      if (k == FK_SKIP && w > 0 && p.fast[w - 1].kind == FK_MIN128_HI) init = ~0ull;
      acc[(g * NFW + w) * NT + tid] = init;
    }
  for (uint32_t g = tid; g < FG; g += NT) tbl[g] = (p.n_keys == 0) ? 0ull : kEmptyKey;
  if (tid == 0 && p.staged) {
    for (uint32_t s = 0; s < p.stages; ++s) mbar_init(&bars[s], 1);
    mbar_fence_init();
  }
  __syncthreads();

  const u64 n_tiles = p.n_tiles;
  const uint32_t T = p.tile_rows;
  uint32_t errbits = 0;
  u64 sel_count = 0;

  // tiles owned by this CTA: first_tile + blockIdx.x + i*gridDim.x
  const u64 my_tiles = (n_tiles > blockIdx.x) ? (n_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;

  auto issue_tile = [&](u64 local_i) {
    const u64 tile = p.first_tile + blockIdx.x + local_i * gridDim.x;
    const uint32_t s = (uint32_t)(local_i % p.stages);
    unsigned char* sb = stage0 + (size_t)s * p.stage_bytes;
    mbar_arrive_expect_tx(&bars[s], p.tx_bytes);  // tx_bytes counts exactly the bytes copied below
    for (uint32_t c = 0; c < p.n_cols; ++c) {
      const ColDesc& cd = p.cols[c];
      const uint32_t bytes = T * cd.elem_bytes;
      bulk_g2s(sb + cd.smem_off, reinterpret_cast<const unsigned char*>(cd.base) + tile * (u64)bytes, bytes, &bars[s]);
      if (cd.validity) bulk_g2s(sb + cd.vsmem_off, cd.validity + tile * (u64)(T / 8), T / 8, &bars[s]);
    }
  };

  if (p.staged && tid == 0) {
    for (u64 i = 0; i + 1 < p.stages && i < my_tiles; ++i) issue_tile(i);
  }

  for (u64 li = 0; li < my_tiles; ++li) {
    const u64 tile = p.first_tile + blockIdx.x + li * gridDim.x;
    const u64 row0 = tile * (u64)T;
    const unsigned char* sb = stage0;
    if (p.staged) {
      const uint32_t s = (uint32_t)(li % p.stages);
      if (tid == 0 && li + p.stages - 1 < my_tiles) issue_tile(li + p.stages - 1);
      mbar_wait(&bars[s], (uint32_t)((li / p.stages) & 1));
      sb = stage0 + (size_t)s * p.stage_bytes;
    }

    // ---- per-row state
    V t0[R], t1[R];
    uint32_t nm[R];     // NULL flag per absolute stack position
    bool act[R];
    int slot[R];        // CTA-local group slot, -1 = use the global path
    u64 gkey[R];
    bool gnull[R];
    i64 gs[R];          // cached global slot, -1 = not looked up yet
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const u64 row = row0 + (u64)r * NT + tid;
      act[r] = row >= p.row_begin && row < p.row_end;
      // row-id-sparse tables: positions whose row id nobody holds (deleted rows, gaps) are not rows
      if (p.exists_bits && act[r]) act[r] = (p.exists_bits[row >> 3] >> (row & 7)) & 1;
      nm[r] = 0;
      t0[r] = 0;
      t1[r] = 0;
      slot[r] = (p.n_keys == 0 && FG > 0) ? 0 : -1;
      gkey[r] = 0;
      gnull[r] = false;
      gs[r] = (p.n_keys == 0) ? 0 : -1;
    }
    int sp = 0;
    bool pred_phase = true;  // selection phase: errors count for every row of the scanned range (the reference evaluates
                             // predicate expressions over the whole domain); afterwards only for selected rows
    auto err_row = [&](int r) -> bool {
      if (!pred_phase) return act[r];
      const u64 row = row0 + (u64)r * NT + tid;
      if (!(row >= p.row_begin && row < p.row_end)) return false;
      return !p.exists_bits || ((p.exists_bits[row >> 3] >> (row & 7)) & 1);
    };

    // helpers -----------------------------------------------------------------------------------------
    auto spill_ptr = [&](int depth, int r) -> V* { return spill + ((size_t)(depth * R + r) * NT + tid); };
    auto push_prep = [&]() {  // make room: t1 -> memory, t0 -> t1
      if (sp >= 2) {
#pragma unroll
        for (int r = 0; r < R; ++r) *spill_ptr(sp - 2, r) = t1[r];
      }
#pragma unroll
      for (int r = 0; r < R; ++r) t1[r] = t0[r];
    };
    auto set_null = [&](int r, int pos, bool isnull) { nm[r] = (nm[r] & ~(1u << pos)) | ((uint32_t)isnull << pos); };
    auto is_null = [&](int r, int pos) -> bool { return (nm[r] >> pos) & 1u; };
    auto pop_refill = [&]() {  // after a binary op consumed t1: reload t1 from memory
      if (sp >= 3) {
#pragma unroll
        for (int r = 0; r < R; ++r) t1[r] = *spill_ptr(sp - 3, r);
      }
    };
    auto col_is_null = [&](const ColDesc& cd, int r) -> bool {
      if (!cd.validity) return false;
      const uint32_t rit = (uint32_t)r * NT + tid;
      if (p.staged) return !((sb[cd.vsmem_off + (rit >> 3)] >> (rit & 7)) & 1);
      const u64 row = row0 + rit;
      return !((cd.validity[row >> 3] >> (row & 7)) & 1);
    };
    auto load_u64 = [&](const ColDesc& cd, int r) -> u64 {
      const uint32_t rit = (uint32_t)r * NT + tid;
      if (p.staged) return *reinterpret_cast<const u64*>(sb + cd.smem_off + (size_t)rit * 8);
      return __ldg(reinterpret_cast<const u64*>(cd.base) + row0 + rit);
    };
    auto get_gs = [&](int r) -> u64 {
      if (gs[r] < 0) gs[r] = (i64)global_slot(p, gkey[r], gnull[r], errbits);
      return (u64)gs[r];
    };

    // ---- run the program
    for (uint32_t pc = 0; pc < p.n_instr; ++pc) {
      const Instr in = p.code[pc];
      switch (in.op) {
        case OP_END: pc = p.n_instr; break;

        case OP_PUSH_COL: {
          push_prep();
          const ColDesc& cd = p.cols[in.a];
#pragma unroll
          for (int r = 0; r < R; ++r) {
            const uint32_t rit = (uint32_t)r * NT + tid;
            const unsigned char* src = p.staged ? sb + cd.smem_off + (size_t)rit * cd.elem_bytes
                                                : reinterpret_cast<const unsigned char*>(cd.base) + (row0 + rit) * cd.elem_bytes;
            V v = 0;
            switch (in.b) {
              case LK_I8: v = *reinterpret_cast<const signed char*>(src); break;
              case LK_I16: v = *reinterpret_cast<const short*>(src); break;
              case LK_I32: v = *reinterpret_cast<const int*>(src); break;
              case LK_I64: v = *reinterpret_cast<const i64*>(src); break;
              case LK_U8: v = *reinterpret_cast<const unsigned char*>(src); break;
              case LK_U16: v = *reinterpret_cast<const unsigned short*>(src); break;
              case LK_U32: v = *reinterpret_cast<const unsigned int*>(src); break;
              case LK_U64: v = (V)(*reinterpret_cast<const i64*>(src)); break;
              case LK_F32: v = f64_bits((double)*reinterpret_cast<const float*>(src)); break;
              case LK_F64: v = *reinterpret_cast<const i64*>(src); break;
              case LK_D64: v = *reinterpret_cast<const i64*>(src); break;
              case LK_D32: v = *reinterpret_cast<const int*>(src); break;
              case LK_STR8: v = (V)(((i64)(u64)(*reinterpret_cast<const unsigned char*>(src)) << 56) | 1); break;
              case LK_D128: {
                ulonglong2 w;
                if (p.staged) w = *reinterpret_cast<const ulonglong2*>(src);
                else w = ldg_nc_v2(src);
                if (WIDE) {
                  v = (V)(((u128)w.y << 64) | (u128)w.x);
                } else {
                  v = (V)(i64)w.x;
                  if ((i64)w.y != ((i64)w.x >> 63) && err_row(r)) errbits |= FLAG_NARROW_FAIL;
                }
                break;
              }
            }
            t0[r] = v;
            set_null(r, sp, col_is_null(cd, r));
          }
          ++sp;
          break;
        }
        case OP_PUSH_LIT: {
          push_prep();
          const Lit L = p.lits[in.c];
          V v;
          if (WIDE) v = (V)(((u128)L.hi << 64) | (u128)L.lo);
          else v = (V)(i64)L.lo;
#pragma unroll
          for (int r = 0; r < R; ++r) {
            t0[r] = v;
            set_null(r, sp, in.b != 0);
          }
          ++sp;
          break;
        }
        case OP_PICK: {
          const int d = in.a;  // 0 = top
          V tmp[R];
          bool tn[R];
#pragma unroll
          for (int r = 0; r < R; ++r) {
            tmp[r] = d == 0 ? t0[r] : d == 1 ? t1[r] : *spill_ptr(sp - 1 - d, r);
            tn[r] = is_null(r, sp - 1 - d);
          }
          push_prep();
#pragma unroll
          for (int r = 0; r < R; ++r) {
            t0[r] = tmp[r];
            set_null(r, sp, tn[r]);
          }
          ++sp;
          break;
        }
        case OP_POP: {
#pragma unroll
          for (int r = 0; r < R; ++r) t0[r] = t1[r];
          pop_refill();
          --sp;
          break;
        }
        case OP_NIP: {
#pragma unroll
          for (int r = 0; r < R; ++r) set_null(r, sp - 2, is_null(r, sp - 1));
          pop_refill();
          --sp;
          break;
        }

        // ---------------------------------------------------------------- binary arithmetic: t1 (lhs) op t0 (rhs)
        case OP_ADD_I: case OP_SUB_I: case OP_MUL_I: case OP_DIV_I: case OP_MOD_I: {
#pragma unroll
          for (int r = 0; r < R; ++r) {
            const i64 a = (i64)t1[r], b = (i64)t0[r];
            bool n = is_null(r, sp - 2) || is_null(r, sp - 1);
            i64 c = 0;
            bool ok = true;
            if (in.op == OP_ADD_I) ok = add_ck(a, b, c);
            else if (in.op == OP_SUB_I) ok = sub_ck(a, b, c);
            else if (in.op == OP_MUL_I) ok = mul_ck(a, b, c);
            else if (in.op == OP_DIV_I) {
              if (b == 0) n = true;  // zeros -> NULL before div (kernels.rs:121-135)
              else if (a == (i64)0x8000000000000000ll && b == -1) ok = false;
              else c = a / b;
            } else {
              if (b == 0) { if (!n && err_row(r)) errbits |= FLAG_DIV_ZERO; }
              else c = (b == -1) ? 0 : a % b;
            }
            if (!ok && !n && err_row(r)) errbits |= in.b ? FLAG_EXACT_OVERFLOW : FLAG_ARITH_OVERFLOW;
            t0[r] = (V)c;
            set_null(r, sp - 2, n);
          }
          pop_refill();
          --sp;
          break;
        }
        case OP_ADD_F: case OP_SUB_F: case OP_MUL_F: case OP_DIV_F: case OP_MOD_F: {
#pragma unroll
          for (int r = 0; r < R; ++r) {
            const double a = as_f64(t1[r]), b = as_f64(t0[r]);
            bool n = is_null(r, sp - 2) || is_null(r, sp - 1);
            double c;
            if (in.op == OP_ADD_F) c = a + b;
            else if (in.op == OP_SUB_F) c = a - b;
            else if (in.op == OP_MUL_F) c = a * b;
            else if (in.op == OP_DIV_F) { if (b == 0.0) n = true; c = a / b; }
            else c = fmod(a, b);
            t0[r] = (V)f64_bits(c);
            set_null(r, sp - 2, n);
          }
          pop_refill();
          --sp;
          break;
        }
        case OP_ADD_D: case OP_SUB_D: case OP_MUL_D: {
#pragma unroll
          for (int r = 0; r < R; ++r) {
            const bool n = is_null(r, sp - 2) || is_null(r, sp - 1);
            V c;
            bool ok;
            if (in.op == OP_ADD_D) ok = add_ck(t1[r], t0[r], c);
            else if (in.op == OP_SUB_D) ok = sub_ck(t1[r], t0[r], c);
            else ok = mul_ck(t1[r], t0[r], c);
            if (WIDE && ok && in.b) ok = fits_precision(c, 38);  // exact mode: DecimalValue::new
            if (!ok && !n && err_row(r)) errbits |= WIDE ? (in.b ? FLAG_EXACT_OVERFLOW : FLAG_ARITH_OVERFLOW) : FLAG_NARROW_FAIL;
            t0[r] = c;
            set_null(r, sp - 2, n);
          }
          pop_refill();
          --sp;
          break;
        }

        // ---------------------------------------------------------------- casts (unary, in place)
        case OP_CAST_I_F:
#pragma unroll
          for (int r = 0; r < R; ++r) t0[r] = (V)f64_bits(__ll2double_rn((i64)t0[r]));
          break;
        case OP_CAST_U_F:
#pragma unroll
          for (int r = 0; r < R; ++r) t0[r] = (V)f64_bits(__ull2double_rn((u64)(i64)t0[r]));
          break;
        case OP_CAST_D_F: {
          const double den = __longlong_as_double((i64)p.lits[in.c].lo);
#pragma unroll
          for (int r = 0; r < R; ++r) t0[r] = (V)f64_bits(to_f64(t0[r]) / den);
          break;
        }
        case OP_CAST_I_D: case OP_CAST_D_UP: case OP_RESCALE_DX: {
#pragma unroll
          for (int r = 0; r < R; ++r) {
            V c;
            bool ok;
            if (WIDE) {
              V x = in.op == OP_CAST_I_D ? (in.c ? (V)(u64)(i64)t0[r] : (V)(i64)t0[r]) : t0[r];
              ok = mul_ck(x, (V)pow10_i128(in.a), c);
              if (ok) ok = fits_precision(c, in.op == OP_RESCALE_DX ? 38 : in.b);
              if (!ok) {
                if (in.op == OP_RESCALE_DX) { if (!is_null(r, sp - 1) && err_row(r)) errbits |= FLAG_EXACT_OVERFLOW; }
                else set_null(r, sp - 1, true);
              }
            } else {
              ok = in.a <= 18 && !(in.op == OP_CAST_I_D && in.c && (i64)t0[r] < 0) &&
                   mul_ck((i64)t0[r], pow10_i64(in.a <= 18 ? in.a : 0), c);
              if (!ok) {
                if (!is_null(r, sp - 1) && err_row(r)) errbits |= FLAG_NARROW_FAIL;
              } else if (in.op != OP_RESCALE_DX && !fits_precision(c, in.b)) {
                set_null(r, sp - 1, true);
              }
            }
            t0[r] = c;
          }
          break;
        }
        case OP_CAST_D_DOWN: {
#pragma unroll
          for (int r = 0; r < R; ++r) {
            const V c = div_pow10_round<V>(t0[r], in.a);
            if (!fits_precision(c, in.b)) set_null(r, sp - 1, true);
            t0[r] = c;
          }
          break;
        }
        case OP_CAST_F_I: {
#pragma unroll
          for (int r = 0; r < R; ++r) {
            const double f = as_f64(t0[r]);
            const bool ok = f >= -9223372036854775808.0 && f < 9223372036854775808.0;
            if (!ok) set_null(r, sp - 1, true);
            t0[r] = ok ? (V)__double2ll_rz(f) : (V)0;
          }
          break;
        }
        case OP_CAST_I_I: {
          const int bits = in.a;
#pragma unroll
          for (int r = 0; r < R; ++r) {
            const i64 v = (i64)t0[r];
            if (bits < 64 && (v < -((i64)1 << (bits - 1)) || v > ((i64)1 << (bits - 1)) - 1)) set_null(r, sp - 1, true);
          }
          break;
        }
        case OP_CAST_I_B:
#pragma unroll
          for (int r = 0; r < R; ++r) t0[r] = (V)((i64)t0[r] != 0);
          break;
        case OP_CAST_U_I:
#pragma unroll
          for (int r = 0; r < R; ++r)
            if ((i64)t0[r] < 0) set_null(r, sp - 1, true);
          break;
        case OP_CAST_I_U:
#pragma unroll
          for (int r = 0; r < R; ++r)
            if ((i64)t0[r] < 0) set_null(r, sp - 1, true);
          break;

        // ---------------------------------------------------------------- compare -> B
        case OP_CMP_I: case OP_CMP_U: case OP_CMP_F: case OP_CMP_D: {
#pragma unroll
          for (int r = 0; r < R; ++r) {
            const bool n = is_null(r, sp - 2) || is_null(r, sp - 1);
            int c;
            if (in.op == OP_CMP_I) { const i64 a = (i64)t1[r], b = (i64)t0[r]; c = a < b ? -1 : a > b; }
            else if (in.op == OP_CMP_U) { const u64 a = (u64)(i64)t1[r], b = (u64)(i64)t0[r]; c = a < b ? -1 : a > b; }
            else if (in.op == OP_CMP_F) { const i64 a = f64_total_key(as_f64(t1[r])), b = f64_total_key(as_f64(t0[r])); c = a < b ? -1 : a > b; }
            else { c = t1[r] < t0[r] ? -1 : t1[r] > t0[r]; }
            bool res;
            switch (in.a) {
              case 0: res = c == 0; break;
              case 1: res = c != 0; break;
              case 2: res = c < 0; break;
              case 3: res = c <= 0; break;
              case 4: res = c > 0; break;
              default: res = c >= 0; break;
            }
            t0[r] = (V)(res && !n);
            set_null(r, sp - 2, n);
          }
          pop_refill();
          --sp;
          break;
        }

        // ---------------------------------------------------------------- typed predicates (unary -> B)
        case OP_PRED_I: case OP_PRED_U: case OP_PRED_F: case OP_PRED_D: {
          const int lk = in.a & 3, uk = (in.a >> 2) & 3, eq = (in.a >> 4) & 1;
          const Lit L0 = p.lits[in.c];
          const Lit L1 = p.lits[in.c + ((lk != 2 && !eq) ? 1 : 0)];
#pragma unroll
          for (int r = 0; r < R; ++r) {
            const bool n = is_null(r, sp - 1);
            bool m = true;
            if (in.op == OP_PRED_I) {
              const i64 v = (i64)t0[r];
              if (eq) m = v == (i64)L0.lo;
              else {
                if (lk != 2) m = lk == 0 ? v >= (i64)L0.lo : v > (i64)L0.lo;
                if (uk != 2) m = m && (uk == 0 ? v <= (i64)L1.lo : v < (i64)L1.lo);
              }
            } else if (in.op == OP_PRED_U) {
              const u64 v = (u64)(i64)t0[r];
              if (eq) m = v == L0.lo;
              else {
                if (lk != 2) m = lk == 0 ? v >= L0.lo : v > L0.lo;
                if (uk != 2) m = m && (uk == 0 ? v <= L1.lo : v < L1.lo);
              }
            } else if (in.op == OP_PRED_F) {  // partial_cmp: NaN never matches
              const double v = as_f64(t0[r]);
              const double a = __longlong_as_double((i64)L0.lo), b = __longlong_as_double((i64)L1.lo);
              if (eq) m = v == a;
              else {
                if (lk != 2) m = lk == 0 ? v >= a : v > a;
                if (uk != 2) m = m && (uk == 0 ? v <= b : v < b);
              }
            } else {
              const V v = t0[r];
              V a, b;
              if (WIDE) { a = (V)(((u128)L0.hi << 64) | L0.lo); b = (V)(((u128)L1.hi << 64) | L1.lo); }
              else { a = (V)(i64)L0.lo; b = (V)(i64)L1.lo; }
              if (eq) m = v == a;
              else {
                if (lk != 2) m = lk == 0 ? v >= a : v > a;
                if (uk != 2) m = m && (uk == 0 ? v <= b : v < b);
              }
            }
            t0[r] = (V)(m && !n);
            // NULL flag stays: domain = field present (DomainOp::PushFieldAll)
          }
          break;
        }
        case OP_IN_BITS: case OP_IN_F: case OP_IN_D: {
#pragma unroll
          for (int r = 0; r < R; ++r) {
            const bool n = is_null(r, sp - 1);
            bool m = false;
            for (uint32_t k = 0; k < in.b; ++k) {
              const Lit L = p.lits[in.c + k];
              if (in.op == OP_IN_BITS) m = m || ((u64)(i64)t0[r] == L.lo);
              else if (in.op == OP_IN_F) m = m || (as_f64(t0[r]) == __longlong_as_double((i64)L.lo));
              else if (WIDE) m = m || (t0[r] == (V)(((u128)L.hi << 64) | L.lo));
              else m = m || ((i64)t0[r] == (i64)L.lo);
            }
            t0[r] = (V)(m && !n);
          }
          break;
        }
        case OP_PRED_STR: {
          const u64 pat = p.lits[in.c].lo;
          const unsigned L = in.b, mode = in.a & 3u;
          const u64 top = L ? (pat >> (64 - 8 * L)) : 0;
#pragma unroll
          for (int r = 0; r < R; ++r) {
            const bool n = is_null(r, sp - 1);
            u64 k = (u64)(i64)t0[r];
            const unsigned len = (unsigned)(k & 0xffu);
            if (in.a & 4u) {  // ASCII lower case of the seven string bytes (the plan proved there is no byte >= 0x80)
              const u64 b = k & ~0xffull;
              k |= (((b + 0x3f3f3f3f3f3f3f00ull) & ~(b + 0x2525252525252500ull)) & 0x8080808080808000ull) >> 2;
            }
            bool m = false;
            if (len >= L) {
              if (L == 0) m = true;
              else if (mode == 2) m = (k >> (64 - 8 * L)) == top;
              else if (mode == 0) m = ((k << (8 * (len - L))) >> (64 - 8 * L)) == top;
              else
                for (unsigned s0 = 0; s0 + L <= len; ++s0) m = m || (((k << (8 * s0)) >> (64 - 8 * L)) == top);
            }
            t0[r] = (V)(m && !n);
          }
          break;
        }
        case OP_PRED_ISNULL:
#pragma unroll
          for (int r = 0; r < R; ++r) {
            // rows = table rows - present rows; domain = present rows (table.rs:1133-1142, program.rs:467)
            t0[r] = (V)is_null(r, sp - 1);
          }
          break;
        case OP_PRED_NOTNULL:
#pragma unroll
          for (int r = 0; r < R; ++r) t0[r] = (V)!is_null(r, sp - 1);
          break;
        case OP_PRED_ALL:
#pragma unroll
          for (int r = 0; r < R; ++r) t0[r] = (V)1;
          break;
        case OP_ISNULL:
#pragma unroll
          for (int r = 0; r < R; ++r) {
            const bool n = is_null(r, sp - 1);
            t0[r] = (V)(in.a ? !n : n);
            set_null(r, sp - 1, false);
          }
          break;
        case OP_INLIST_FOLD: {  // acc(t1) <- acc | item(t0): matched |= T, saw_null |= item NULL
#pragma unroll
          for (int r = 0; r < R; ++r) {
            const bool n = is_null(r, sp - 2) || is_null(r, sp - 1);
            t0[r] = (V)(((i64)t1[r] | (i64)t0[r]) & 1);
            set_null(r, sp - 2, n);
          }
          pop_refill();
          --sp;
          break;
        }
        case OP_INLIST_END:  // stack: [target, acc] -> [result]; NULL IN (...) is NULL
#pragma unroll
          for (int r = 0; r < R; ++r) {
            const bool matched = ((i64)t0[r] & 1) != 0;
            const bool known = (matched || !is_null(r, sp - 1)) && !is_null(r, sp - 2);
            t0[r] = (V)(known && (in.a ? !matched : matched));
            set_null(r, sp - 2, !known);
          }
          pop_refill();
          --sp;
          break;
        case OP_AND: case OP_OR: {
          // rows: bitmap AND/OR; domain: Intersect / Union (llkv-compute/src/program.rs:500-512)
#pragma unroll
          for (int r = 0; r < R; ++r) {
            const bool n1 = is_null(r, sp - 2), n0 = is_null(r, sp - 1);
            const bool a = ((i64)t1[r] & 1) != 0, b = ((i64)t0[r] & 1) != 0;
            t0[r] = (V)(in.op == OP_AND ? (a && b) : (a || b));
            set_null(r, sp - 2, in.op == OP_AND ? (n1 || n0) : (n1 && n0));
          }
          pop_refill();
          --sp;
          break;
        }
        case OP_NOT:  // domain - rows (llkv-scan/src/predicate.rs:167-186)
#pragma unroll
          for (int r = 0; r < R; ++r) t0[r] = (V)(!is_null(r, sp - 1) && !((i64)t0[r] & 1));
          break;
        case OP_BOOL_LIT:
          push_prep();
#pragma unroll
          for (int r = 0; r < R; ++r) {
            t0[r] = (V)in.a;
            set_null(r, sp, false);
          }
          ++sp;
          break;
        case OP_FILTER: {
          bool any = false;
#pragma unroll
          for (int r = 0; r < R; ++r) {
            act[r] = act[r] && (((i64)t0[r] & 1) != 0);
            any = any || act[r];
            t0[r] = t1[r];
          }
          pop_refill();
          --sp;
          if ((in.a & 1) && !p.bitmap_mode && sp == 0 && !__any_sync(0xffffffffu, any)) pc = p.n_instr;  // whole warp filtered out
          break;
        }
        case OP_SELECT_DONE: {
          pred_phase = false;
          bool any = false;
#pragma unroll
          for (int r = 0; r < R; ++r) any = any || act[r];
          if (!p.bitmap_mode && sp == 0 && !__any_sync(0xffffffffu, any)) pc = p.n_instr;
          break;
        }
        case OP_RAISE: {
#pragma unroll
          for (int r = 0; r < R; ++r)
            if (act[r]) errbits |= 1u << in.a;
          break;
        }
        case OP_MVCC: {
          // RowVersion::is_visible_for (llkv-transaction/src/mvcc.rs:282-334); NULL created_by -> 1, NULL deleted_by -> MAX
          const ColDesc& cc = p.cols[in.a];
          const ColDesc& dc = p.cols[in.b];
          bool any = false;
#pragma unroll
          for (int r = 0; r < R; ++r) {
            u64 cb = load_u64(cc, r), db = load_u64(dc, r);
            if (col_is_null(cc, r)) cb = 1ull;
            if (col_is_null(dc, r)) db = ~0ull;
            bool vis;
            bool c_committed = cb != ~0ull, d_committed = db != ~0ull;
            for (uint32_t k = 0; k < p.n_noncommitted; ++k) {
              const u64 id = p.noncommitted[k];
              if (id == cb && cb != 1ull) c_committed = false;
              if (id == db && db != 1ull) d_committed = false;
            }
            if (cb == p.txn_id && p.txn_id != 1ull) vis = db != p.txn_id;
            else if (!c_committed) vis = false;
            else if (cb > p.snapshot_id) vis = false;
            else if (db == ~0ull) vis = true;
            else if (db == p.txn_id && p.txn_id != 1ull) vis = false;
            else if (!d_committed) vis = true;
            else vis = db > p.snapshot_id;
            act[r] = act[r] && vis;
            any = any || act[r];
          }
          (void)any;
          break;
        }

        // ---------------------------------------------------------------- GROUP BY key -> slot
        case OP_GROUP: {
          const int nk = in.a;
          // keys sit at stack positions sp-nk .. sp-1 (first key deepest)
#pragma unroll
          for (int r = 0; r < R; ++r) {
            u64 K = 0;
            bool knull = false;
            if (p.single_wide_key == 1) {
              K = (u64)(i64)t0[r];
              knull = is_null(r, sp - 1);
            } else if (p.single_wide_key == 2) {
              K = key_hash_init();
              for (int k = 0; k < nk; ++k) {
                const int pos = sp - nk + k;
                const int d = sp - 1 - pos;
                const u64 v = (u64)(i64)(d == 0 ? t0[r] : d == 1 ? t1[r] : *spill_ptr(pos, r));
                K = key_hash_step(K, v, is_null(r, pos));
              }
              K = key_hash_done(K);
            } else {
              int shift = 0;
              for (int k = 0; k < nk; ++k) {
                const int pos = sp - nk + k;
                const int d = sp - 1 - pos;
                const u64 v = (u64)(i64)(d == 0 ? t0[r] : d == 1 ? t1[r] : *spill_ptr(pos, r));
                const int bits = p.key_bits[k];
                const bool n = is_null(r, pos);
                u64 f;
                if (p.key_kind[k] == KK_STR) {  // packed short string: bytes from the top, length in the low 3 bits
                  const int L = p.key_strlen[k];
                  f = (L ? ((v >> (64 - 8 * L)) << 3) : 0ull) | (v & 7ull);
                } else {
                  f = v - p.key_min[k];
                }
                const u64 field = n ? 0 : (bits == 64 ? f : (f & ((1ull << bits) - 1)));
                K |= field << shift;
                shift += bits;
                if (p.key_nullable[k]) { K |= (u64)n << shift; shift += 1; }
              }
            }
            gkey[r] = K;
            gnull[r] = knull;
            gs[r] = -1;
            slot[r] = -1;
            if (act[r] && FG > 0 && !knull && K != kEmptyKey) {
              uint32_t h = (uint32_t)mix64(K) & (FG - 1);
              for (uint32_t i = 0; i < FG; ++i) {
                const u64 cur = tbl[h];
                if (cur == K) { slot[r] = (int)h; break; }
                if (cur == kEmptyKey) {
                  const u64 old = atomicCAS(&tbl[h], kEmptyKey, K);
                  if (old == kEmptyKey || old == K) { slot[r] = (int)h; break; }
                }
                h = (h + 1) & (FG - 1);
              }
            }
          }
          // drop the keys
          for (int k = 0; k < nk; ++k) {
#pragma unroll
            for (int r = 0; r < R; ++r) t0[r] = t1[r];
            pop_refill();
            --sp;
          }
          break;
        }

        // ---------------------------------------------------------------- aggregates
        case OP_AGG_COUNT_STAR: {
#pragma unroll
          for (int r = 0; r < R; ++r) {
            if (!act[r]) continue;
            if (slot[r] >= 0) acc[((uint32_t)slot[r] * NFW + in.b) * NT + tid] += 1;
            else atomicAdd(&p.gwords[get_gs(r) * p.n_gwords + in.c], 1ull);
          }
          break;
        }
        case OP_AGG_FIRSTROW: {
#pragma unroll
          for (int r = 0; r < R; ++r) {
            if (!act[r]) continue;
            const u64 row = p.row_origin + row0 + (u64)r * NT + tid;
            if (slot[r] >= 0) {
              u64* a = &acc[((uint32_t)slot[r] * NFW + in.b) * NT + tid];
              if (row < *a) *a = row;
            } else atomicMin(&p.gwords[get_gs(r) * p.n_gwords + in.c], row);
          }
          break;
        }
        case OP_AGG_FIRSTVALID: case OP_AGG_FIRSTNAN: {  // value stays on the stack
#pragma unroll
          for (int r = 0; r < R; ++r) {
            if (!act[r] || is_null(r, sp - 1)) continue;
            if (in.op == OP_AGG_FIRSTNAN) {
              const double d = as_f64(t0[r]);
              if (d == d) continue;
            }
            const u64 row = p.row_origin + row0 + (u64)r * NT + tid;
            if (slot[r] >= 0) {
              u64* a = &acc[((uint32_t)slot[r] * NFW + in.b) * NT + tid];
              if (row < *a) *a = row;
            } else atomicMin(&p.gwords[get_gs(r) * p.n_gwords + in.c], row);
          }
          break;
        }
        case OP_AGG_COUNT: case OP_AGG_SUM_I: case OP_AGG_SUM_D: case OP_AGG_FSUM:
        case OP_AGG_MIN_I: case OP_AGG_MAX_I: case OP_AGG_MIN_U: case OP_AGG_MAX_U:
        case OP_AGG_MIN_F: case OP_AGG_MAX_F: case OP_AGG_MIN_D: case OP_AGG_MAX_D: {
#pragma unroll
          for (int r = 0; r < R; ++r) {
            if (!act[r] || is_null(r, sp - 1)) continue;
            const V v = t0[r];
            u64* a = slot[r] >= 0 ? &acc[((uint32_t)slot[r] * NFW + in.b) * NT + tid] : nullptr;
            switch (in.op) {
              case OP_AGG_COUNT:
                if (a) *a += 1; else atomicAdd(&p.gwords[get_gs(r) * p.n_gwords + in.c], 1ull);
                break;
              case OP_AGG_SUM_I: case OP_AGG_SUM_D: {
                // per-thread i64 partial sums stay exact while |v| < 2^47 and a thread folds < 2^15 rows per launch
                const bool narrow = v < ((V)1 << 47) && v > -((V)1 << 47);
                if (a && narrow) *a = (u64)((i64)*a + (i64)v);
                else {
                  u64* w = &p.gwords[get_gs(r) * p.n_gwords + in.c];
                  if (in.op == OP_AGG_SUM_I) gadd_sum_i64(w, (i128)(i64)v);
                  else gadd_sum_i128(w, (i128)v);
                }
                break;
              }
              case OP_AGG_FSUM:
                if (a) *a = (u64)f64_bits(__longlong_as_double((i64)*a) + as_f64(v));
                else atomicAdd(reinterpret_cast<double*>(&p.gwords[get_gs(r) * p.n_gwords + in.c]), as_f64(v));
                break;
              case OP_AGG_MIN_I: case OP_AGG_MAX_I: case OP_AGG_MIN_U: case OP_AGG_MAX_U: case OP_AGG_MIN_F: case OP_AGG_MAX_F: {
                u64 e;
                bool is_min = in.op == OP_AGG_MIN_I || in.op == OP_AGG_MIN_U || in.op == OP_AGG_MIN_F;
                if (in.op == OP_AGG_MIN_I || in.op == OP_AGG_MAX_I) e = enc_i64((i64)v);
                else if (in.op == OP_AGG_MIN_U || in.op == OP_AGG_MAX_U) e = (u64)(i64)v;
                else {
                  const double d = as_f64(v);
                  if (d != d) break;  // NaN never replaces a number (lib.rs:1309-1331); leading-NaN case: see DESIGN.md
                  e = enc_f64(d);
                }
                if (a) { if (is_min ? e < *a : e > *a) *a = e; }
                else if (is_min) atomicMin(&p.gwords[get_gs(r) * p.n_gwords + in.c], e);
                else atomicMax(&p.gwords[get_gs(r) * p.n_gwords + in.c], e);
                break;
              }
              default: {  // MIN_D / MAX_D: (hi encoded, lo) pair
                const i128 x = (i128)v;
                const u64 hi = enc_i64((i64)(x >> 64)), lo = (u64)x;
                const bool is_max = in.op == OP_AGG_MAX_D;
                if (a) {
                  u64* a2 = a + NT;
                  const bool better = is_max ? (hi > a[0] || (hi == a[0] && lo > *a2)) : (hi < a[0] || (hi == a[0] && lo < *a2));
                  if (better) { a[0] = hi; *a2 = lo; }
                } else gmin128(&p.gwords[get_gs(r) * p.n_gwords + in.c], hi, lo, is_max);
                break;
              }
            }
          }
          if (!(in.a & 1)) {
#pragma unroll
            for (int r = 0; r < R; ++r) t0[r] = t1[r];
            pop_refill();
            --sp;
          }
          break;
        }

        case OP_EMIT_BITMAP: {
          uint32_t* out32 = reinterpret_cast<uint32_t*>(p.out_bitmap);
#pragma unroll
          for (int r = 0; r < R; ++r) {
            uint32_t m = __ballot_sync(0xffffffffu, act[r]);
            const u64 base = row0 + (u64)r * NT + (u64)warp * 32;  // first row of this warp's 32-row group
            if (lane == 0 && m) {
              sel_count += __popc(m);
              u64 bitpos;
              if (base < p.row_begin) {
                m >>= (uint32_t)(p.row_begin - base);
                bitpos = 0;
              } else bitpos = base - p.row_begin;
              const uint32_t sh = (uint32_t)(bitpos & 31);
              atomicOr(&out32[bitpos >> 5], m << sh);
              if (sh && (m >> (32 - sh))) atomicOr(&out32[(bitpos >> 5) + 1], m >> (32 - sh));
            }
          }
          break;
        }
        default: errbits |= FLAG_BAD_PLAN; pc = p.n_instr; break;
      }
    }
    if (p.staged) __syncthreads();  // everyone is done with this stage before thread 0 refills it
  }

  // ---- fold the CTA's per-thread accumulators into the global table
  __syncthreads();
  const int n_warps = NT >> 5;
  for (uint32_t g = 0; g < FG; ++g) {
    const u64 K = tbl[g];
    if (p.n_keys != 0 && K == kEmptyKey) continue;
    u64 gslot = 0;
    if (p.n_keys != 0) {
      if (lane == 0) gslot = global_slot(p, K, false, errbits);
      gslot = __shfl_sync(0xffffffffu, gslot, 0);
    }
    u64* grow = &p.gwords[gslot * p.n_gwords];
    for (uint32_t w = warp; w < NFW; w += n_warps) {
      const FastWord fw = p.fast[w];
      const u64* a = &acc[(g * NFW + w) * NT];
      switch (fw.kind) {
        case FK_COUNT: {
          u64 s = 0;
          for (int t = lane; t < NT; t += 32) s += a[t];
          for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
          if (lane == 0 && s) atomicAdd(&grow[fw.gword], s);
          break;
        }
        case FK_SUM_I64: case FK_SUM_I128: {
          i64 lo = 0, hi = 0;  // sum of low 32 bits / sum of arithmetic high parts
          for (int t = lane; t < NT; t += 32) {
            const i64 v = (i64)a[t];
            lo += (i64)((u64)v & 0xffffffffull);
            hi += v >> 32;
          }
          for (int o = 16; o; o >>= 1) {
            lo += __shfl_xor_sync(0xffffffffu, lo, o);
            hi += __shfl_xor_sync(0xffffffffu, hi, o);
          }
          if (lane == 0 && (lo | hi)) {
            const i128 t = (i128)lo + ((i128)hi << 32);
            if (fw.kind == FK_SUM_I64) gadd_sum_i64(&grow[fw.gword], t);
            else gadd_sum_i128(&grow[fw.gword], t);
          }
          break;
        }
        case FK_FSUM: {
          double s = 0.0;
          for (int t = lane; t < NT; t += 32) s += __longlong_as_double((i64)a[t]);
          for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
          if (lane == 0) atomicAdd(reinterpret_cast<double*>(&grow[fw.gword]), s);
          break;
        }
        case FK_MIN: case FK_MAX: {
          const bool is_min = fw.kind == FK_MIN;
          u64 s = is_min ? ~0ull : 0ull;
          for (int t = lane; t < NT; t += 32) s = is_min ? min(s, a[t]) : max(s, a[t]);
          for (int o = 16; o; o >>= 1) {
            const u64 x = __shfl_xor_sync(0xffffffffu, s, o);
            s = is_min ? min(s, x) : max(s, x);
          }
          if (lane == 0) { if (is_min) atomicMin(&grow[fw.gword], s); else atomicMax(&grow[fw.gword], s); }
          break;
        }
        case FK_MIN128_HI: case FK_MAX128_HI: {
          const bool is_max = fw.kind == FK_MAX128_HI;
          const u64* a2 = a + NT;
          u64 bh = is_max ? 0ull : ~0ull, bl = is_max ? 0ull : ~0ull;
          for (int t = lane; t < NT; t += 32) {
            const u64 h = a[t], l = a2[t];
            const bool better = is_max ? (h > bh || (h == bh && l > bl)) : (h < bh || (h == bh && l < bl));
            if (better) { bh = h; bl = l; }
          }
          for (int o = 16; o; o >>= 1) {
            const u64 h = __shfl_xor_sync(0xffffffffu, bh, o), l = __shfl_xor_sync(0xffffffffu, bl, o);
            const bool better = is_max ? (h > bh || (h == bh && l > bl)) : (h < bh || (h == bh && l < bl));
            if (better) { bh = h; bl = l; }
          }
          if (lane == 0) gmin128(&grow[fw.gword], bh, bl, is_max);
          break;
        }
        default: break;  // FK_SKIP
      }
    }
  }
  if (p.bitmap_mode && sel_count) atomicAdd(p.out_count, sel_count);
  if (errbits) atomicOr(p.flags, errbits);
}

// ------------------------------------------------------------------ small utility kernels
__global__ void init_table_kernel(u64* keys, u64* words, u64 rows, uint32_t n_gwords, const uint8_t* word_class_dev) {
  const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  const u64 total = rows * n_gwords;
  if (keys && i + 2 < rows) keys[i] = kEmptyKey;  // `rows` counts the two spare rows (reserved key value, NULL key), which have no key slot
  for (u64 j = i; j < total; j += (u64)gridDim.x * blockDim.x) words[j] = gword_initial(word_class_dev[j % n_gwords]);
}

// merge kernel for gathered partial tables (multi-GPU GROUP BY): rows of `src` are folded into the local table
__global__ void merge_table_kernel(const Plan* __restrict__ gplan, const u64* src_keys, const u64* src_words, u64 src_rows_cap) {
  const Plan& p = *gplan;
  const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= src_rows_cap + 2) return;
  bool occupied, knull = false;
  u64 K = kEmptyKey;
  if (p.n_keys == 0) { occupied = (i == 0); }
  else if (i < src_rows_cap) { K = src_keys[i]; occupied = K != kEmptyKey; }
  else { occupied = src_words[i * p.n_gwords] != 0; knull = (i == src_rows_cap + 1); }  // word 0 = rows folded into the group
  if (!occupied) return;
  uint32_t err = 0;
  const u64 gsl = global_slot(p, K, knull, err);
  const u64* s = &src_words[i * p.n_gwords];
  u64* d = &p.gwords[gsl * p.n_gwords];
  for (uint32_t w = 0; w < p.n_gwords; ++w) {
    switch (p.gword_class[w]) {
      case WC_SUM: if (s[w]) atomicAdd(&d[w], s[w]); break;
      case WC_FSUM: atomicAdd(reinterpret_cast<double*>(&d[w]), __longlong_as_double((i64)s[w])); break;
      case WC_MIN: atomicMin(&d[w], s[w]); break;
      case WC_MAX: atomicMax(&d[w], s[w]); break;
      case WC_MIN128: gmin128(&d[w], s[w], s[w + 1], false); break;
      case WC_MAX128: gmin128(&d[w], s[w], s[w + 1], true); break;
      default: break;
    }
  }
  if (err) atomicOr(p.flags, err);
}

// Ungrouped multi-GPU merge: the state is one row of words.  One thread per word folds the N gathered rows in rank
// order starting from the word's identity, so every rank ends with the bit-identical state (f64 sums included) and the
// whole merge is one launch after the all-gather: no table re-initialisation, no plan upload.
__global__ void merge_ungrouped_kernel(u64* dst, const u64* all_words, int n_ranks, uint32_t n_gwords, u64 rank_stride,
                                       const uint8_t* word_class_dev) {
  const uint32_t w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= n_gwords) return;
  const uint8_t c = word_class_dev[w];
  if (c == WC_PAIR_LO_MIN || c == WC_PAIR_LO_MAX) return;  // written with its high word
  if (c == WC_MIN128 || c == WC_MAX128) {
    const bool is_max = c == WC_MAX128;
    u64 bh = is_max ? 0ull : ~0ull, bl = bh;
    for (int r = 0; r < n_ranks; ++r) {
      const u64 h = all_words[(u64)r * rank_stride + w], l = all_words[(u64)r * rank_stride + w + 1];
      const bool better = is_max ? (h > bh || (h == bh && l > bl)) : (h < bh || (h == bh && l < bl));
      if (better) { bh = h; bl = l; }
    }
    dst[w] = bh;
    dst[w + 1] = bl;
    return;
  }
  u64 acc = c == WC_MIN ? ~0ull : 0ull;
  double facc = 0.0;
  for (int r = 0; r < n_ranks; ++r) {
    const u64 v = all_words[(u64)r * rank_stride + w];
    switch (c) {
      case WC_SUM: acc += v; break;
      case WC_FSUM: facc += __longlong_as_double((i64)v); break;
      case WC_MIN: acc = v < acc ? v : acc; break;
      case WC_MAX: acc = v > acc ? v : acc; break;
      default: break;
    }
  }
  dst[w] = c == WC_FSUM ? (u64)__double_as_longlong(facc) : acc;
}

// Ungrouped multi-GPU merge over NVLink peer memory, no collective library on the path: every rank stores its state row
// into a mailbox slot on every peer (plain stores into peer-mapped memory, cudaIpc), waits for the rows of all ranks in its
// own mailbox and folds them in rank order (bit-identical states on all ranks, f64 sums included).  One small kernel per
// rank and merge.
//   mailbox layout per rank: [source rank][merge parity][slot].  Two parities: a rank can be one merge ahead of a peer, never
//   two (merge e+1 needs the peer's data of e+1, which the peer's stream writes after its merge e).  A peer that never
//   arrives ends the wait after kMergeWaitNs (120 s) with FLAG_MERGE_TIMEOUT.  The limit is long on purpose: ranks reach their
//   first merge seconds apart when one of them compiles a kernel or pages the library in from a cold disk.
struct PeerMailboxes {
  u64* box[8];
};
__device__ __forceinline__ u64 ld_acquire_sys(const u64* p) {
  u64 v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_sys(u64* p, u64 v) { asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory"); }
constexpr u64 kMergeWaitNs = 120000000000ull;
__device__ __forceinline__ u64 global_timer_ns() {
  u64 t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
// The merge number (`epoch`) lives in device memory and advances with every exchange, in step on all ranks: the launch
// has no per-merge parameter, so a captured CUDA graph replays it.
//
// The exchange itself is flag-in-data (the "LL" idea of collective libraries): every 64-bit state word travels as two
// 8-byte packets (32 bits of data | the merge number), one plain store each — 8-byte stores are single-copy atomic, so a
// packet whose upper half shows the current merge number is complete by itself.  No fence, no separate flag, no release /
// acquire round: the latency of a merge is one NVLink store plus the poll (measured: ~20 us with fence + flag).
constexpr uint32_t kMergePackets = 256;  // packets per (source rank, parity) slot = kUngroupedSlotWords of the runtime
__device__ __forceinline__ void st_volatile_u64(u64* p, u64 v) { asm volatile("st.volatile.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory"); }
__device__ __forceinline__ u64 ld_volatile_u64(const u64* p) {
  u64 v;
  asm volatile("ld.volatile.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__global__ void __launch_bounds__(kMergePackets) merge_ungrouped_p2p_kernel(u64* state, PeerMailboxes peers, int n_ranks, int rank, uint32_t n_gwords,
                                                                            u64* epoch_dev, const uint8_t* word_class_dev, uint32_t* flags) {
  const uint32_t t = threadIdx.x;  // packet index: word t / 2, half t & 1
  const u64 epoch = *epoch_dev + 1;
  __shared__ uint32_t s_part[8][kMergePackets];
  __shared__ int timed_out;
  if (t == 0) timed_out = 0;
  __syncthreads();  // every thread has read the counter
  if (t == 0) *epoch_dev = epoch;
  const uint32_t e32 = (uint32_t)epoch, par = (uint32_t)(epoch & 1);
  const bool on = (t >> 1) < n_gwords;
  if (on) {
    const u64 v = state[t >> 1];
    const u64 pkt = ((u64)e32 << 32) | (uint32_t)((t & 1) ? (v >> 32) : v);
    for (int r = 0; r < n_ranks; ++r) st_volatile_u64(&peers.box[r][(uint32_t)(rank * 2 + (int)par) * kMergePackets + t], pkt);
    const u64* mine = peers.box[rank];
    const u64 t0 = global_timer_ns();
    for (int r = 0; r < n_ranks; ++r) {
      const u64* src = &mine[((uint32_t)r * 2 + par) * kMergePackets + t];
      u64 pk = ld_volatile_u64(src);
      while ((uint32_t)(pk >> 32) != e32) {
        if (global_timer_ns() - t0 > kMergeWaitNs) {
          timed_out = 1;
          break;
        }
        __nanosleep(100);
        pk = ld_volatile_u64(src);
      }
      s_part[r][t] = (uint32_t)pk;
    }
  }
  __syncthreads();
  if (timed_out) {
    if (t == 0) atomicOr(flags, FLAG_MERGE_TIMEOUT);
    return;
  }
  const uint32_t w = t;
  if (w >= n_gwords) return;
  const uint8_t c = word_class_dev[w];
  if (c == WC_PAIR_LO_MIN || c == WC_PAIR_LO_MAX) return;  // written with its high word
  auto word_of = [&](int r, uint32_t x) -> u64 { return (u64)s_part[r][2 * x] | ((u64)s_part[r][2 * x + 1] << 32); };
  if (c == WC_MIN128 || c == WC_MAX128) {
    const bool is_max = c == WC_MAX128;
    u64 bh = is_max ? 0ull : ~0ull, bl = bh;
    for (int r = 0; r < n_ranks; ++r) {
      const u64 h = word_of(r, w), l = word_of(r, w + 1);
      const bool better = is_max ? (h > bh || (h == bh && l > bl)) : (h < bh || (h == bh && l < bl));
      if (better) { bh = h; bl = l; }
    }
    state[w] = bh;
    state[w + 1] = bl;
    return;
  }
  u64 acc = c == WC_MIN ? ~0ull : 0ull;
  double facc = 0.0;
  for (int r = 0; r < n_ranks; ++r) {
    const u64 v = word_of(r, w);
    switch (c) {
      case WC_SUM: acc += v; break;
      case WC_FSUM: facc += __longlong_as_double((i64)v); break;
      case WC_MIN: acc = v < acc ? v : acc; break;
      case WC_MAX: acc = v > acc ? v : acc; break;
      default: break;
    }
  }
  state[w] = c == WC_FSUM ? (u64)__double_as_longlong(facc) : acc;
}

// Grouped multi-GPU merge over NVLink peer memory for small group tables (TPC-H Q1: 34 rows): the same mailbox protocol as
// the ungrouped merge, the message being the rank's whole table [flag = epoch | capacity | keys | words].  One CTA per rank:
//   1. store the own table into the (rank, parity) slot of every peer, fence, publish with a release flag;
//   2. wait for every rank's flag in the own mailbox;
//   3. re-initialise the own table and fold the N received tables into it in rank order — rows of one source table have
//      distinct keys, so they fold in parallel without atomics on the words, and the fixed rank order makes every rank end
//      with the bit-identical table (f64 sums included).
// No collective library, no host synchronisation, one launch.  `exchange` = 0 repeats step 3 only (the host grew the
// table after FLAG_TABLE_FULL: the received tables are still in the mailbox).  The capacity word doubles as the sender's
// status: a table that does not fit a slot (every rank reports FLAG_MERGE_OVERSIZE), a scan that has to be repeated on the
// sender first (64-bit overflow, table full: every rank leaves its table alone and reports FLAG_MERGE_RETRY, the host
// settles the scan and all ranks merge again), a scan that failed (FLAG_MERGE_PEER_FAILED everywhere).
constexpr u64 kMsgOversize = ~0ull, kMsgRerun = ~0ull - 1, kMsgFailed = ~0ull - 2;
struct GroupMergeArgs {
  u64* gkeys;
  u64* gwords;
  u64 gcap;
  const uint8_t* wclass;
  uint32_t* flags;
  PeerMailboxes peers;
  u64* epoch_dev;  // merges so far (device memory, shared with the ungrouped merge); an exchange advances it
  uint32_t n_gwords, slot_words;
  int n_ranks, rank, exchange;
};
__global__ void __launch_bounds__(512) merge_grouped_p2p_kernel(GroupMergeArgs a) {
  const uint32_t tid = threadIdx.x, NT = blockDim.x;
  const u64 epoch = *a.epoch_dev + (a.exchange ? 1 : 0);
  __syncthreads();  // every thread has read the counter
  if (tid == 0 && a.exchange) *a.epoch_dev = epoch;
  const uint32_t par = (uint32_t)(epoch & 1);
  const u64 rows = a.gcap + 2;
  const u64 n_key_words = a.gcap, n_words = rows * a.n_gwords;
  __shared__ int s_status;
  if (tid == 0) s_status = 0;
  if (a.exchange) {
    const uint32_t local = *a.flags;  // what the scan queued in front of this kernel left behind
    u64 head = a.gcap;
    if (local & ~(FLAG_NARROW_FAIL | FLAG_TABLE_FULL)) head = kMsgFailed;
    else if (local) head = kMsgRerun;
    else if (2 + n_key_words + n_words + rows > a.slot_words) head = kMsgOversize;  // (+ rows: the receiver's scratch)
    const bool fits = head == a.gcap;
    for (int r = 0; r < a.n_ranks; ++r) {
      u64* dst = a.peers.box[r] + (size_t)(a.rank * 2 + par) * a.slot_words;
      if (tid == 0) dst[1] = head;
      if (fits) {
        for (u64 i = tid; i < n_key_words; i += NT) dst[2 + i] = a.gkeys[i];
        for (u64 i = tid; i < n_words; i += NT) dst[2 + n_key_words + i] = a.gwords[i];
      }
    }
    __threadfence_system();
    __syncthreads();
    if (tid < (uint32_t)a.n_ranks) st_release_sys(a.peers.box[tid] + (size_t)(a.rank * 2 + par) * a.slot_words, epoch);
    if (tid < (uint32_t)a.n_ranks) {
      const u64* flag = a.peers.box[a.rank] + (size_t)(tid * 2 + par) * a.slot_words;
      const u64 t0 = global_timer_ns();
      while (ld_acquire_sys(flag) != epoch) {
        if (global_timer_ns() - t0 > kMergeWaitNs) {
          atomicOr(&s_status, 1);
          break;
        }
        __nanosleep(200);
      }
    }
    __syncthreads();
    __threadfence_system();
  } else {
    __syncthreads();
  }
  const u64* mine = a.peers.box[a.rank];
  if (!s_status && tid < (uint32_t)a.n_ranks) {
    const u64 head = mine[(size_t)(tid * 2 + par) * a.slot_words + 1];
    if (head == kMsgOversize) atomicOr(&s_status, 2);
    else if (head == kMsgRerun) atomicOr(&s_status, 4);
    else if (head == kMsgFailed) atomicOr(&s_status, 8);
  }
  __syncthreads();
  if (s_status) {  // the own table stays as the scan left it
    if (tid == 0)
      atomicOr(a.flags, (s_status & 1) ? FLAG_MERGE_TIMEOUT : (s_status & 8) ? FLAG_MERGE_PEER_FAILED : (s_status & 4) ? FLAG_MERGE_RETRY : FLAG_MERGE_OVERSIZE);
    return;
  }
  // fresh table
  for (u64 i = tid; i < n_key_words; i += NT) a.gkeys[i] = kEmptyKey;
  for (u64 i = tid; i < n_words; i += NT) {
    const uint8_t c = a.wclass[i % a.n_gwords];
    a.gwords[i] = (c == WC_MIN || c == WC_MIN128 || c == WC_PAIR_LO_MIN) ? ~0ull : 0ull;
  }
  __syncthreads();
  const u64 mask = a.gcap - 1;
  uint32_t err = 0;
  __shared__ uint8_t s_class[kMaxWords];
  for (uint32_t w = tid; w < a.n_gwords; w += NT) s_class[w] = a.wclass[w];
  // (a) destination row of every occupied source row of every rank, all at once: a few dependent L2 round trips in total.
  //     The rows land behind the rank's message in the mailbox slot (the sender left room for them).
  for (int r = 0; r < a.n_ranks; ++r) {
    u64* src = const_cast<u64*>(mine) + (size_t)(r * 2 + par) * a.slot_words;
    const u64 scap = src[1];
    const u64* skeys = src + 2;
    const u64* swords = src + 2 + scap;
    u64* dest = src + 2 + scap + (scap + 2) * a.n_gwords;
    for (u64 i = tid; i < scap + 2; i += NT) {
      u64 slot = ~0ull;
      if (i < scap) {
        const u64 K = skeys[i];
        if (K != kEmptyKey) {
          u64 h = mix64(K) & mask;
          for (u64 t = 0; t <= mask; ++t) {
            const u64 cur = a.gkeys[h];
            if (cur == K) { slot = h; break; }
            if (cur == kEmptyKey) {
              const u64 old = atomicCAS(&a.gkeys[h], kEmptyKey, K);
              if (old == kEmptyKey || old == K) { slot = h; break; }
            }
            h = (h + 1) & mask;
          }
          if (slot == ~0ull) err |= FLAG_TABLE_FULL;
        }
      } else if (swords[i * a.n_gwords] != 0) {  // word 0 = rows folded into the group: the spare rows (reserved key value, NULL key)
        slot = a.gcap + (i - scap);
      }
      dest[i] = slot;
    }
  }
  __syncthreads();
  // (b) the words, one thread per (source row, word), rank after rank: rows of one source table go to distinct groups, so
  //     the updates need no atomics, and the fixed rank order gives every rank the same f64 sums
  for (int r = 0; r < a.n_ranks; ++r) {
    const u64* src = mine + (size_t)(r * 2 + par) * a.slot_words;
    const u64 scap = src[1];
    const u64* swords = src + 2 + scap;
    const u64* dest = src + 2 + scap + (scap + 2) * a.n_gwords;
    const u64 items = (scap + 2) * a.n_gwords;
    for (u64 idx = tid; idx < items; idx += NT) {
      const u64 i = idx / a.n_gwords;
      const uint32_t w = (uint32_t)(idx % a.n_gwords);
      const u64 slot = dest[i];
      if (slot == ~0ull) continue;
      const uint8_t c = s_class[w];
      if (c == WC_PAIR_LO_MIN || c == WC_PAIR_LO_MAX) continue;  // written with its high word
      const u64 v = swords[idx];
      u64* d = a.gwords + slot * a.n_gwords + w;
      switch (c) {
        case WC_SUM: if (v) *d += v; break;
        case WC_FSUM: *d = (u64)__double_as_longlong(__longlong_as_double((i64)*d) + __longlong_as_double((i64)v)); break;
        case WC_MIN: if (v < *d) *d = v; break;
        case WC_MAX: if (v > *d) *d = v; break;
        default: {  // WC_MIN128 / WC_MAX128: (high, low) pair
          const bool is_max = c == WC_MAX128;
          const u64 l = swords[idx + 1], ch = d[0], cl = d[1];
          const bool better = is_max ? (v > ch || (v == ch && l > cl)) : (v < ch || (v == ch && l < cl));
          if (better) { d[0] = v; d[1] = l; }
          break;
        }
      }
    }
    __syncthreads();  // the next rank's rows may meet the same groups
  }
  if (err) atomicOr(a.flags, err);
}

// ------------------------------------------------------------------ host-callable launchers
cudaError_t launch_merge_ungrouped_p2p(u64* state, u64* const* peer_boxes, int n_ranks, int rank, uint32_t n_gwords, u64* epoch_dev,
                                       const uint8_t* word_class_dev, uint32_t* flags, cudaStream_t stream) {
  PeerMailboxes pm;
  for (int r = 0; r < 8; ++r) pm.box[r] = r < n_ranks ? peer_boxes[r] : nullptr;
  merge_ungrouped_p2p_kernel<<<1, kMergePackets, 0, stream>>>(state, pm, n_ranks, rank, n_gwords, epoch_dev, word_class_dev, flags);
  return cudaGetLastError();
}
cudaError_t launch_merge_grouped_p2p(u64* gkeys, u64* gwords, u64 gcap, uint32_t n_gwords, const uint8_t* word_class_dev, uint32_t* flags,
                                     u64* const* peer_boxes, uint32_t slot_words, int n_ranks, int rank, u64* epoch_dev, bool exchange, cudaStream_t stream) {
  GroupMergeArgs a;
  a.gkeys = gkeys;
  a.gwords = gwords;
  a.gcap = gcap;
  a.wclass = word_class_dev;
  a.flags = flags;
  for (int r = 0; r < 8; ++r) a.peers.box[r] = r < n_ranks ? peer_boxes[r] : nullptr;
  a.epoch_dev = epoch_dev;
  a.n_gwords = n_gwords;
  a.slot_words = slot_words;
  a.n_ranks = n_ranks;
  a.rank = rank;
  a.exchange = exchange ? 1 : 0;
  merge_grouped_p2p_kernel<<<1, 512, 0, stream>>>(a);
  return cudaGetLastError();
}
cudaError_t launch_merge_ungrouped(u64* dst, const u64* all_words, int n_ranks, uint32_t n_gwords, u64 rank_stride,
                                   const uint8_t* word_class_dev, cudaStream_t stream) {
  merge_ungrouped_kernel<<<(n_gwords + 127) / 128, 128, 0, stream>>>(dst, all_words, n_ranks, n_gwords, rank_stride, word_class_dev);
  return cudaGetLastError();
}

cudaError_t launch_scan(const Plan* dplan, bool wide, int rows_per_thread, uint32_t grid, uint32_t block, uint32_t smem,
                        cudaStream_t stream) {
#define LLKV_LAUNCH(W, RR)                                                                              \
  do {                                                                                                  \
    cudaError_t e = cudaFuncSetAttribute(scan_kernel<W, RR>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
    if (e != cudaSuccess) return e;                                                                     \
    scan_kernel<W, RR><<<grid, block, smem, stream>>>(dplan);                                           \
    return cudaGetLastError();                                                                          \
  } while (0)
  if (!wide) {
    if (rows_per_thread == 4) LLKV_LAUNCH(false, 4);
    if (rows_per_thread == 2) LLKV_LAUNCH(false, 2);
    LLKV_LAUNCH(false, 1);
  } else {
    if (rows_per_thread >= 2) LLKV_LAUNCH(true, 2);
    LLKV_LAUNCH(true, 1);
  }
#undef LLKV_LAUNCH
}

cudaError_t launch_init_table(u64* keys, u64* words, u64 rows, uint32_t n_gwords, const uint8_t* word_class_dev, cudaStream_t stream) {
  const u64 total = rows * n_gwords > rows ? rows * n_gwords : rows;
  u64 blocks = (total + 255) / 256;
  if (blocks > 65535ull * 16) blocks = 65535ull * 16;
  if (blocks == 0) blocks = 1;
  // every thread i < rows must exist to clear keys: grid covers max(rows, min(total, cap))
  const u64 need = (rows + 255) / 256;
  if (blocks < need) blocks = need;
  init_table_kernel<<<(unsigned)blocks, 256, 0, stream>>>(keys, words, rows, n_gwords, word_class_dev);
  return cudaGetLastError();
}

cudaError_t launch_merge_table(const Plan* dplan, const u64* src_keys, const u64* src_words, u64 src_cap, cudaStream_t stream) {
  const u64 n = src_cap + 2;
  merge_table_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(dplan, src_keys, src_words, src_cap);
  return cudaGetLastError();
}

}  // namespace llkv

// device_util.cuh — sm_100a device helpers: bulk-copy (TMA) + mbarrier PTX, 128-bit integer arithmetic with the
// overflow rules of the reference's arithmetic, order-preserving encodings, hashing.
#pragma once
#ifndef __CUDACC_RTC__
#include <cuda_runtime.h>
#include <stdint.h>
#endif

#include "plan.h"

namespace llkv {

typedef long long i64;
typedef unsigned long long u64;
typedef __int128 i128;
typedef unsigned __int128 u128;

// the value an accumulator word of class `c` (WordClass) holds before any row is folded into it
__device__ __forceinline__ u64 gword_initial(uint8_t c) {
  return (c == WC_MIN || c == WC_MIN128 || c == WC_PAIR_LO_MIN) ? ~0ull : 0ull;
}

// ------------------------------------------------------------------ mbarrier + cp.async.bulk (TMA 1-D bulk copy)
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(void* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(void* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(void* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(void* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// try_wait with a suspend-time hint: the hardware parks the thread until the phase completes or ~ns elapse
__device__ __forceinline__ bool mbar_try_wait_hint(void* bar, uint32_t parity, uint32_t ns) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity), "r"(ns)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(void* bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}
// global -> shared bulk copy completing on an mbarrier (SASS: UBLKCP).  dst/src 16-byte aligned, bytes % 16 == 0.
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, void* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// streaming 128-bit / 64-bit loads for the non-staged path
__device__ __forceinline__ ulonglong2 ldg_nc_v2(const void* p) {
  ulonglong2 r;
  asm volatile("ld.global.nc.L1::no_allocate.v2.u64 {%0, %1}, [%2];" : "=l"(r.x), "=l"(r.y) : "l"(p));
  return r;
}

// ------------------------------------------------------------------ hashing / encodings
__device__ __forceinline__ u64 mix64(u64 x) {
  x ^= x >> 33;
  x *= 0xff51afd7ed558ccdULL;
  x ^= x >> 33;
  x *= 0xc4ceb9fe1a85ec53ULL;
  x ^= x >> 33;
  return x;
}
// order-preserving u64 keys (same idea as llkv-column-map/src/codecs.rs:33-65)
__device__ __forceinline__ u64 enc_i64(i64 v) { return (u64)v ^ 0x8000000000000000ull; }
__device__ __forceinline__ u64 enc_f64(double d) {
  u64 b = (u64)__double_as_longlong(d);
  return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
// IEEE totalOrder key as a signed integer (arrow-ord float comparison)
__device__ __forceinline__ i64 f64_total_key(double d) {
  i64 b = __double_as_longlong(d);
  return b ^ (i64)((u64)(b >> 63) >> 1);
}

// ------------------------------------------------------------------ powers of ten
__constant__ u64 kPow10U64[20] = {1ull,
                                   10ull,
                                   100ull,
                                   1000ull,
                                   10000ull,
                                   100000ull,
                                   1000000ull,
                                   10000000ull,
                                   100000000ull,
                                   1000000000ull,
                                   10000000000ull,
                                   100000000000ull,
                                   1000000000000ull,
                                   10000000000000ull,
                                   100000000000000ull,
                                   1000000000000000ull,
                                   10000000000000000ull,
                                   100000000000000000ull,
                                   1000000000000000000ull,
                                   10000000000000000000ull};
// 10^0 .. 10^38 as (lo, hi)
__constant__ u64 kPow10U128[39][2] = {
    {0x0000000000000001ull, 0x0ull}, {0x000000000000000aull, 0x0ull}, {0x0000000000000064ull, 0x0ull},
    {0x00000000000003e8ull, 0x0ull}, {0x0000000000002710ull, 0x0ull}, {0x00000000000186a0ull, 0x0ull},
    {0x00000000000f4240ull, 0x0ull}, {0x0000000000989680ull, 0x0ull}, {0x0000000005f5e100ull, 0x0ull},
    {0x000000003b9aca00ull, 0x0ull}, {0x00000002540be400ull, 0x0ull}, {0x000000174876e800ull, 0x0ull},
    {0x000000e8d4a51000ull, 0x0ull}, {0x000009184e72a000ull, 0x0ull}, {0x00005af3107a4000ull, 0x0ull},
    {0x00038d7ea4c68000ull, 0x0ull}, {0x002386f26fc10000ull, 0x0ull}, {0x016345785d8a0000ull, 0x0ull},
    {0x0de0b6b3a7640000ull, 0x0ull}, {0x8ac7230489e80000ull, 0x0ull}, {0x6bc75e2d63100000ull, 0x5ull},
    {0x35c9adc5dea00000ull, 0x36ull}, {0x19e0c9bab2400000ull, 0x21eull}, {0x02c7e14af6800000ull, 0x152dull},
    {0x1bcecceda1000000ull, 0xd3c2ull}, {0x161401484a000000ull, 0x84595ull}, {0xdcc80cd2e4000000ull, 0x52b7d2ull},
    {0x9fd0803ce8000000ull, 0x33b2e3cull}, {0x3e25026110000000ull, 0x204fce5eull}, {0x6d7217caa0000000ull, 0x1431e0faeull},
    {0x4674edea40000000ull, 0xc9f2c9cd0ull}, {0xc0914b2680000000ull, 0x7e37be2022ull}, {0x85acef8100000000ull, 0x4ee2d6d415bull},
    {0x38c15b0a00000000ull, 0x314dc6448d93ull}, {0x378d8e6400000000ull, 0x1ed09bead87c0ull}, {0x2b878fe800000000ull, 0x13426172c74d82ull},
    {0xb34b9f1000000000ull, 0xc097ce7bc90715ull}, {0x00f436a000000000ull, 0x785ee10d5da46d9ull}, {0x098a224000000000ull, 0x4b3b4ca85a86c47aull}};

__device__ __forceinline__ i128 pow10_i128(int k) { return (i128)(((u128)kPow10U128[k][1] << 64) | (u128)kPow10U128[k][0]); }
__device__ __forceinline__ i64 pow10_i64(int k) { return (i64)kPow10U64[k]; }

// ------------------------------------------------------------------ checked arithmetic.  Return false on overflow.
__device__ __forceinline__ bool add_ck(i64 a, i64 b, i64& r) {
  r = (i64)((u64)a + (u64)b);
  return (((a ^ r) & (b ^ r)) >> 63) == 0;
}
__device__ __forceinline__ bool sub_ck(i64 a, i64 b, i64& r) {
  r = (i64)((u64)a - (u64)b);
  return (((a ^ b) & (a ^ r)) >> 63) == 0;
}
__device__ __forceinline__ bool mul_ck(i64 a, i64 b, i64& r) {
  r = (i64)((u64)a * (u64)b);
  return __mul64hi(a, b) == (r >> 63);
}
__device__ __forceinline__ bool add_ck(i128 a, i128 b, i128& r) {
  r = (i128)((u128)a + (u128)b);
  return (((a ^ r) & (b ^ r)) >> 127) == 0;
}
__device__ __forceinline__ bool sub_ck(i128 a, i128 b, i128& r) {
  r = (i128)((u128)a - (u128)b);
  return (((a ^ b) & (a ^ r)) >> 127) == 0;
}
static __device__ __noinline__ bool mul_ck(i128 a, i128 b, i128& out) {
  const bool neg = (a < 0) != (b < 0);
  const u128 ua = a < 0 ? (u128)0 - (u128)a : (u128)a;
  const u128 ub = b < 0 ? (u128)0 - (u128)b : (u128)b;
  const u64 a0 = (u64)ua, a1 = (u64)(ua >> 64), b0 = (u64)ub, b1 = (u64)(ub >> 64);
  out = (i128)((u128)a * (u128)b);
  if (a1 && b1) return false;
  const u128 lo = (u128)a0 * (u128)b0;
  const u128 cross = a1 ? (u128)a1 * (u128)b0 : (u128)b1 * (u128)a0;
  if ((u64)(cross >> 64)) return false;
  const u128 r = lo + (cross << 64);
  if (r < lo) return false;
  if (neg) return r <= ((u128)1 << 127);
  return (r >> 127) == 0;
}
// |v| < 10^p   (arrow is_valid_decimal_precision / DecimalValue::new digit count)
__device__ __forceinline__ bool fits_precision(i128 v, int p) {
  if (p >= 39) return true;
  const i128 lim = pow10_i128(p);
  return v < lim && v > -lim;
}
__device__ __forceinline__ bool fits_precision(i64 v, int p) {
  if (p >= 19) return true;
  const i64 lim = pow10_i64(p);
  return v < lim && v > -lim;
}

// Rust `i128 as f64`: round to nearest even
__device__ __forceinline__ double to_f64(i64 v) { return __ll2double_rn(v); }
static __device__ __noinline__ double to_f64(i128 v) {
  const bool neg = v < 0;
  const u128 a = neg ? (u128)0 - (u128)v : (u128)v;
  const u64 hi = (u64)(a >> 64), lo = (u64)a;
  double d;
  if (hi == 0) {
    d = __ull2double_rn(lo);
  } else {
    const int s = 64 - __clzll((i64)hi);  // bits above the low 64
    u64 m = (u64)(a >> s);
    const u64 lost = lo & ((s == 64) ? ~0ull : ((1ull << s) - 1));
    if (lost) m |= 1ull;  // sticky: m keeps 64 significant bits, 11 more than the mantissa, so this preserves RNE
    d = __ull2double_rn(m) * __longlong_as_double((i64)(1023 + s) << 52);
  }
  return neg ? -d : d;
}

// x / 10^k rounded half away from zero (arrow-cast decimal scale reduction; AvgDecimal128 rounding)
template <typename V>
__device__ __forceinline__ V div_pow10_round(V x, int k);
template <>
__device__ __forceinline__ i64 div_pow10_round<i64>(i64 x, int k) {
  i64 d, rem, half;
  switch (k) {  // constant divisors compile to multiply-shift
    case 1: d = x / 10; rem = x - d * 10; half = 5; break;
    case 2: d = x / 100; rem = x - d * 100; half = 50; break;
    case 3: d = x / 1000; rem = x - d * 1000; half = 500; break;
    case 4: d = x / 10000; rem = x - d * 10000; half = 5000; break;
    default: {
      const i64 div = pow10_i64(k);
      d = x / div;
      rem = x - d * div;
      half = div / 2;
    }
  }
  if (x >= 0) {
    if (rem >= half) d += 1;
  } else {
    if (rem <= -half) d -= 1;
  }
  return d;
}
template <>
__device__ __forceinline__ i128 div_pow10_round<i128>(i128 x, int k) {
  const i128 div = pow10_i128(k);
  i128 d = x / div;
  const i128 rem = x - d * div;
  const i128 half = div / 2;
  if (x >= 0) {
    if (rem >= half) d += 1;
  } else {
    if (rem <= -half) d -= 1;
  }
  return d;
}

// ------------------------------------------------------------------ global group table
static __device__ __noinline__ u64 global_slot(const Plan& p, u64 K, bool key_is_null, uint32_t& errbits) {
  if (p.n_keys == 0) return 0;
  if (key_is_null) return p.gcap + 1;
  if (K == kEmptyKey) return p.gcap;
  const u64 mask = p.gcap - 1;
  u64 h = mix64(K) & mask;
  for (u64 i = 0; i <= mask; ++i) {
    u64 cur = p.gkeys[h];
    if (cur == K) return h;
    if (cur == kEmptyKey) {
      const u64 old = atomicCAS(&p.gkeys[h], kEmptyKey, K);
      if (old == kEmptyKey || old == K) return h;
    }
    h = (h + 1) & mask;
  }
  errbits |= FLAG_TABLE_FULL;
  return p.gcap;  // parked on the spare row; the flag makes the run fail
}

// exact integer value -> limb words (see FastKind)
__device__ __forceinline__ void gadd_sum_i64(u64* w, i128 t) {
  atomicAdd(&w[0], (u64)t & 0xffffffffull);
  const u64 hi = (u64)(i64)(t >> 32);
  if (hi) atomicAdd(&w[1], hi);  // small non-negative values (most per-row updates) add nothing to the upper limb
}
__device__ __forceinline__ void gadd_sum_i128(u64* w, i128 t) {
  atomicAdd(&w[0], (u64)t & 0xffffffffull);
  atomicAdd(&w[1], (u64)(t >> 32) & 0xffffffffull);
  atomicAdd(&w[2], (u64)(t >> 64) & 0xffffffffull);
  atomicAdd(&w[3], (u64)(i64)(t >> 96));
}
__device__ __forceinline__ void cas128(ulonglong2* addr, u64 cmp_hi, u64 cmp_lo, u64 swp_hi, u64 swp_lo, u64& old_hi, u64& old_lo) {
  asm volatile(
      "{\n\t.reg .b128 cmp, swp, old;\n\t"
      "mov.b128 cmp, {%2, %3};\n\t"
      "mov.b128 swp, {%4, %5};\n\t"
      "atom.global.cas.b128 old, [%6], cmp, swp;\n\t"
      "mov.b128 {%0, %1}, old;\n\t}"
      : "=l"(old_hi), "=l"(old_lo)
      : "l"(cmp_hi), "l"(cmp_lo), "l"(swp_hi), "l"(swp_lo), "l"(addr)
      : "memory");
}
__device__ __forceinline__ void gmin128(u64* w, u64 hi_enc, u64 lo, bool is_max) {
  // 16-byte CAS loop on (hi_enc, lo): lexicographic order of (hi_enc, lo) == numeric order of the i128.
  // The current pair is read with a CAS too (cmp == swp leaves memory unchanged): two plain 8-byte loads could pair the
  // high word of one update with the low word of another, and a candidate compared against such a torn pair can be
  // dropped although it beats both real states (values of mixed sign).
  ulonglong2* addr = reinterpret_cast<ulonglong2*>(w);
  u64 cur_hi, cur_lo;
  cas128(addr, 0ull, 0ull, 0ull, 0ull, cur_hi, cur_lo);
  while (true) {
    const bool better = is_max ? (hi_enc > cur_hi || (hi_enc == cur_hi && lo > cur_lo))
                               : (hi_enc < cur_hi || (hi_enc == cur_hi && lo < cur_lo));
    if (!better) return;
    u64 old_hi, old_lo;
    cas128(addr, cur_hi, cur_lo, hi_enc, lo, old_hi, old_lo);
    if (old_hi == cur_hi && old_lo == cur_lo) return;
    cur_hi = old_hi;
    cur_lo = old_lo;
  }
}


}  // namespace llkv

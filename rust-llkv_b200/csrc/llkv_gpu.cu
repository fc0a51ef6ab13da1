// llkv_gpu.cu — the C ABI of include/llkv_gpu.h: contexts, device-resident columns (pinned staging ring ->
// cudaMemcpyAsync on copy streams), predicate programs, MVCC snapshots, the fused aggregate runs, finalize, and the
// NCCL merge of partial aggregate states.  There is no CPU fallback anywhere in this file: without a CUDA device
// llkv_gpu_ctx_create fails and every other entry point needs a context.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <deque>
#include <string_view>
#include <thread>
#include <unordered_map>
#include <vector>

#include "../../include/llkv_gpu.h"
#include "compiler.h"
#include "jit.h"
#include "plan.h"
#include "upload.h"

namespace llkv {
typedef long long i64;
typedef unsigned long long u64;
typedef __int128 i128;
typedef unsigned __int128 u128;
cudaError_t launch_scan(const Plan* dplan, bool wide, int rows_per_thread, uint32_t grid, uint32_t block, uint32_t smem,
                        cudaStream_t stream);
cudaError_t launch_lean(const LeanPlan& plan, uint32_t grid, cudaStream_t stream);
cudaError_t launch_partition_apply(const PartPlan& plan, uint32_t grid, cudaStream_t stream);
cudaError_t launch_partition_fold(const FoldPlan& plan, uint32_t grid, cudaStream_t stream);
uint32_t fold_smem_bytes(uint32_t slots, uint32_t n_ops, bool dense);
cudaError_t launch_init_table(u64* keys, u64* words, u64 rows, uint32_t n_gwords, const uint8_t* word_class_dev, cudaStream_t stream);
cudaError_t launch_merge_table(const Plan* dplan, const u64* src_keys, const u64* src_words, u64 src_cap, cudaStream_t stream);
cudaError_t launch_merge_ungrouped_p2p(u64* state, u64* const* peer_boxes, int n_ranks, int rank, uint32_t n_gwords, u64* epoch_dev,
                                       const uint8_t* word_class_dev, uint32_t* flags, cudaStream_t stream);
cudaError_t launch_merge_ungrouped(u64* dst, const u64* all_words, int n_ranks, uint32_t n_gwords, u64 rank_stride, const uint8_t* word_class_dev,
                                   cudaStream_t stream);
cudaError_t launch_merge_grouped_p2p(u64* gkeys, u64* gwords, u64 gcap, uint32_t n_gwords, const uint8_t* word_class_dev, uint32_t* flags,
                                     u64* const* peer_boxes, uint32_t slot_words, int n_ranks, int rank, u64* epoch_dev, bool exchange, cudaStream_t stream);
}  // namespace llkv
// peer mailboxes (llkv_gpu_comm_init): [n_ranks][2][256] packets for ungrouped state rows, then [n_ranks][2][kGroupSlotWords]
// words for small group tables
static constexpr uint32_t kUngroupedSlotWords = 256, kGroupSlotWords = 16384;  // (256 = scan_kernel.cu: kMergePackets)

using namespace llkv;

// ------------------------------------------------------------------------------------------------ errors
static thread_local std::string g_last_error;

static int32_t set_error(int32_t code, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_last_error = buf;
  return code;
}
int32_t llkv_set_error_message(int32_t code, const char* msg) { return set_error(code, "%s", msg); }  // for descriptor.cpp
#define CUDA_TRY(expr)                                                                                          \
  do {                                                                                                          \
    cudaError_t _e = (expr);                                                                                    \
    if (_e != cudaSuccess) return set_error(LLKV_ERR_IO, "CUDA error %s at %s:%d (%s)", cudaGetErrorString(_e), \
                                            __FILE__, __LINE__, #expr);                                         \
  } while (0)

static uint64_t fnv1a(uint64_t h, const void* data, size_t n) {
  const unsigned char* b = static_cast<const unsigned char*>(data);
  for (size_t i = 0; i < n; ++i) h = (h ^ b[i]) * 0x100000001b3ull;
  return h;
}
template <typename T>
static uint64_t fnv_pod(uint64_t h, const T& v) {
  return fnv1a(h, &v, sizeof(T));
}

// ------------------------------------------------------------------------------------------------ column kernels
struct DevStats {
  u64 min_enc, max_enc;  // order-preserving u64 image of the column's values (sign bit flipped for signed types)
  unsigned int not_i64;  // Decimal128: some value is not a sign-extended i64
  unsigned int max_strlen, min_strlen, bad_string;
  u64 data_bytes;        // Utf8: total data bytes
};

template <typename T, bool SIGNED>
__global__ void stats_kernel(const T* __restrict__ v, u64 n, DevStats* st) {
  u64 mn = ~0ull, mx = 0ull;
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
    u64 e = SIGNED ? ((u64)(i64)v[i] ^ 0x8000000000000000ull) : (u64)v[i];
    mn = e < mn ? e : mn;
    mx = e > mx ? e : mx;
  }
  for (int o = 16; o; o >>= 1) {
    const u64 a = __shfl_xor_sync(0xffffffffu, mn, o), b = __shfl_xor_sync(0xffffffffu, mx, o);
    mn = a < mn ? a : mn;
    mx = b > mx ? b : mx;
  }
  if ((threadIdx.x & 31) == 0 && mn <= mx) {
    atomicMin(&st->min_enc, mn);
    atomicMax(&st->max_enc, mx);
  }
}
__global__ void stats_dec_kernel(const ulonglong2* __restrict__ v, u64 n, DevStats* st) {
  u64 mn = ~0ull, mx = 0ull;
  unsigned int bad = 0;
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
    const ulonglong2 w = v[i];
    if ((i64)w.y != ((i64)w.x >> 63)) bad = 1;
    const u64 e = w.x ^ 0x8000000000000000ull;
    mn = e < mn ? e : mn;
    mx = e > mx ? e : mx;
  }
  for (int o = 16; o; o >>= 1) {
    const u64 a = __shfl_xor_sync(0xffffffffu, mn, o), b = __shfl_xor_sync(0xffffffffu, mx, o);
    mn = a < mn ? a : mn;
    mx = b > mx ? b : mx;
    bad |= __shfl_xor_sync(0xffffffffu, bad, o);
  }
  if ((threadIdx.x & 31) == 0) {
    if (mn <= mx) {
      atomicMin(&st->min_enc, mn);
      atomicMax(&st->max_enc, mx);
    }
    if (bad) atomicOr(&st->not_i64, 1u);
  }
}
// Zone maps: one warp per zone of kZoneRows rows, minimum and maximum as the 64-bit value a lean-kernel leaf compares
// (sign- or zero-extended; STRIDE = 2 reads the low half of a Decimal128 that holds a sign-extended i64).
template <typename T, bool SIGNED, int STRIDE>
__global__ void zone_minmax_kernel(const T* __restrict__ v, u64 n, u64* __restrict__ zones) {
  const u64 n_zones = (n + kZoneRows - 1) / kZoneRows;
  const u64 warps = ((u64)gridDim.x * blockDim.x) >> 5;
  const int lane = threadIdx.x & 31;
  for (u64 z = ((u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5; z < n_zones; z += warps) {
    const u64 lo = z * kZoneRows, hi = lo + kZoneRows < n ? lo + kZoneRows : n;
    u64 mn = ~0ull, mx = 0ull;  // in the order-preserving image
    for (u64 i = lo + lane; i < hi; i += 32) {
      const u64 e = SIGNED ? ((u64)(i64)v[i * STRIDE] ^ 0x8000000000000000ull) : (u64)v[i * STRIDE];
      mn = e < mn ? e : mn;
      mx = e > mx ? e : mx;
    }
    for (int o = 16; o; o >>= 1) {
      const u64 a = __shfl_xor_sync(0xffffffffu, mn, o), b = __shfl_xor_sync(0xffffffffu, mx, o);
      mn = a < mn ? a : mn;
      mx = b > mx ? b : mx;
    }
    if (lane == 0) {
      zones[2 * z] = SIGNED ? (mn ^ 0x8000000000000000ull) : mn;
      zones[2 * z + 1] = SIGNED ? (mx ^ 0x8000000000000000ull) : mx;
    }
  }
}
// Utf8 (offsets + data) -> packed short-string keys: bytes big-endian from the top byte, length in the low byte
// (`data` holds the chunk's slice of the data buffer: offsets are relative to `first`)
__global__ void pack_utf8_kernel(const int* __restrict__ off, const unsigned char* __restrict__ data, int first, u64 n, u64* __restrict__ out,
                                 DevStats* st) {
  unsigned int mx = 0, mn = 0xffffffffu, bad = 0;
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
    const int b = off[i] - first, e = off[i + 1] - first;
    const unsigned int len = (unsigned int)(e - b);
    u64 k = 0;
    if (len > 7) bad |= 1;
    else {
      for (unsigned int j = 0; j < len; ++j) k |= (u64)data[b + j] << (56 - 8 * j);
      k |= len;
    }
    out[i] = k;
    if (k & 0x8080808080808000ull) bad |= 2;  // (a byte >= 0x80: case-insensitive patterns need to know)
    mx = len > mx ? len : mx;
    mn = len < mn ? len : mn;
  }
  if (mx || mn != 0xffffffffu) {
    atomicMax(&st->max_strlen, mx);
    atomicMin(&st->min_strlen, mn);
  }
  if (bad) atomicOr(&st->bad_string, bad);
}
// dictionary-coded strings: codes -> ranks after the dictionary has been re-ordered at seal
__global__ void remap_codes_kernel(u64* __restrict__ v, u64 n, const unsigned int* __restrict__ remap) {
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) v[i] = remap[v[i]];
}
__global__ void narrow_str_kernel(const u64* __restrict__ in, unsigned char* __restrict__ out, u64 n) {
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) out[i] = (unsigned char)(in[i] >> 56);
}
__global__ void narrow_dec_kernel(const ulonglong2* __restrict__ in, u64* __restrict__ out, u64 n) {
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) out[i] = in[i].x;
}
// the same narrowing for chunks that crossed the link in the Arrow layout (the DMA share of a hybrid upload): the fit
// check the host workers make is made here, a value that does not fit raises *bad
__global__ void narrow_dec32_check_kernel(const ulonglong2* __restrict__ in, int* __restrict__ out, u64 n, unsigned int* bad) {
  bool b = false;
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
    const ulonglong2 w = in[i];
    out[i] = (int)w.x;
    b = b || (i64)w.y != ((i64)w.x >> 63) || (i64)w.x != (i64)(int)w.x;
  }
  if (b) atomicOr(bad, 1u);
}
__global__ void narrow_dec64_check_kernel(const ulonglong2* __restrict__ in, u64* __restrict__ out, u64 n, unsigned int* bad) {
  bool b = false;
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
    const ulonglong2 w = in[i];
    out[i] = w.x;
    b = b || (i64)w.y != ((i64)w.x >> 63);
  }
  if (b) atomicOr(bad, 1u);
}
__global__ void narrow_dec32_kernel(const ulonglong2* __restrict__ in, int* __restrict__ out, u64 n) {
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) out[i] = (int)in[i].x;
}
__global__ void widen_dec32_kernel(const int* __restrict__ in, ulonglong2* __restrict__ out, u64 n) {
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
    const i64 v = in[i];
    out[i] = make_ulonglong2((u64)v, (u64)(v >> 63));
  }
}
__global__ void widen_dec_kernel(const u64* __restrict__ in, ulonglong2* __restrict__ out, u64 n) {
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
    const u64 v = in[i];
    out[i] = make_ulonglong2(v, (u64)((i64)v >> 63));
  }
}
__global__ void widen_str_kernel(const unsigned char* __restrict__ in, u64* __restrict__ out, u64 n) {
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) out[i] = ((u64)in[i] << 56) | 1ull;
}
// validity bitmaps: OR `n` source bits into dst starting at bit `dst_off`
__global__ void or_bits_kernel(unsigned int* __restrict__ dst, u64 dst_off, const unsigned char* __restrict__ src, u64 n) {
  const u64 nw = (n + 31) / 32;
  for (u64 w = (u64)blockIdx.x * blockDim.x + threadIdx.x; w < nw; w += (u64)gridDim.x * blockDim.x) {
    unsigned int bits = 0;
    for (int b = 0; b < 4; ++b) {
      const u64 byte = w * 4 + b;
      if (byte * 8 < n) bits |= (unsigned int)src[byte] << (8 * b);
    }
    const u64 rem = n - w * 32;
    if (rem < 32) bits &= (1u << rem) - 1u;
    if (!bits) continue;
    const u64 pos = dst_off + w * 32;
    const unsigned int sh = (unsigned int)(pos & 31);
    atomicOr(&dst[pos >> 5], bits << sh);
    if (sh && (bits >> (32 - sh))) atomicOr(&dst[(pos >> 5) + 1], bits >> (32 - sh));
  }
}
__global__ void fill_bits_kernel(unsigned int* __restrict__ dst, u64 bit_begin, u64 bit_end) {
  if (bit_end <= bit_begin) return;
  const u64 w0 = bit_begin >> 5, w1 = (bit_end - 1) >> 5;
  for (u64 w = w0 + (u64)blockIdx.x * blockDim.x + threadIdx.x; w <= w1; w += (u64)gridDim.x * blockDim.x) {
    unsigned int m = 0xffffffffu;
    if (w == w0) m &= 0xffffffffu << (bit_begin & 31);
    if (w == w1 && (bit_end & 31)) m &= (1u << (bit_end & 31)) - 1u;
    atomicOr(&dst[w], m);
  }
}

// Row-id-sparse appends (ColumnStore::append with arbitrary row ids, llkv-column-map/src/store/core.rs:787-1126): row i of the
// chunk lands at position row_ids[i] - origin, and its validity bit is set.  Chunks are applied in append order on one
// stream, so a row id that arrives again overwrites the earlier value (last writer wins, core.rs:1128-1390).  Rows the
// chunk marks NULL are skipped: the reference drops NULLs at append (core.rs:918-942).
template <typename T>
__global__ void scatter_rows_kernel(T* __restrict__ dst, unsigned int* __restrict__ valid, const T* __restrict__ src, const u64* __restrict__ ids,
                                    const unsigned char* __restrict__ src_valid, u64 n, u64 origin) {
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
    if (src_valid && !((src_valid[i >> 3] >> (i & 7)) & 1)) continue;
    const u64 pos = ids[i] - origin;
    dst[pos] = src[i];
    atomicOr(&valid[pos >> 5], 1u << (pos & 31));
  }
}
// Block-wide max / min string length and bad-string bits (1: longer than 7 bytes, 2: a byte >= 0x80) folded into *st with
// one atomic per field.  Every thread of the block calls it; blockDim.x is a multiple of 32, at most 1024.
__device__ __forceinline__ void block_str_stats(unsigned int mx, unsigned int mn, unsigned int bad, DevStats* st) {
  __shared__ unsigned int s_mx[32], s_mn[32], s_bad[32];
  mx = __reduce_max_sync(0xffffffffu, mx);
  mn = __reduce_min_sync(0xffffffffu, mn);
  bad = __reduce_or_sync(0xffffffffu, bad);
  const unsigned int w = threadIdx.x >> 5, nw = blockDim.x >> 5;
  if ((threadIdx.x & 31) == 0) {
    s_mx[w] = mx;
    s_mn[w] = mn;
    s_bad[w] = bad;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (unsigned int i = 1; i < nw; ++i) {
      mx = s_mx[i] > mx ? s_mx[i] : mx;
      mn = s_mn[i] < mn ? s_mn[i] : mn;
      bad |= s_bad[i];
    }
    if (mx || mn != 0xffffffffu) {
      atomicMax(&st->max_strlen, mx);
      atomicMin(&st->min_strlen, mn);
    }
    if (bad) atomicOr(&st->bad_string, bad);
  }
}
// Row-id-sparse appends of a packed Utf8 column: the rules of scatter_rows_kernel, with each string packed into its 8-byte
// key on the way (as pack_utf8_kernel: `data` is the chunk's slice of the data buffer, offsets are relative to `first`).
// Lengths and bytes of the rows written feed the statistics.
__global__ void scatter_utf8_kernel(u64* __restrict__ dst, unsigned int* __restrict__ valid, const int* __restrict__ off,
                                    const unsigned char* __restrict__ data, int first, const u64* __restrict__ ids,
                                    const unsigned char* __restrict__ src_valid, u64 n, u64 origin, DevStats* st) {
  unsigned int mx = 0, mn = 0xffffffffu, bad = 0;
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
    if (src_valid && !((src_valid[i >> 3] >> (i & 7)) & 1)) continue;
    const int b = off[i] - first, e = off[i + 1] - first;
    const unsigned int len = (unsigned int)(e - b);
    u64 k = 0;
    if (len > 7) bad |= 1;
    else {
      for (unsigned int j = 0; j < len; ++j) k |= (u64)data[b + j] << (56 - 8 * j);
      k |= len;
    }
    const u64 pos = ids[i] - origin;
    dst[pos] = k;
    atomicOr(&valid[pos >> 5], 1u << (pos & 31));
    if (k & 0x8080808080808000ull) bad |= 2;
    mx = len > mx ? len : mx;
    mn = len < mn ? len : mn;
  }
  block_str_stats(mx, mn, bad, st);
}
// Statistics of a packed Utf8 column over the positions whose validity bit is set (a sparse column at seal: gaps, deleted
// rows and overwritten values must not count).  The length is the key's low byte, the bytes are the key's upper bytes.
__global__ void str_stats_kernel(const u64* __restrict__ keys, const unsigned int* __restrict__ valid, u64 n, DevStats* st) {
  unsigned int mx = 0, mn = 0xffffffffu, bad = 0;
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
    if (valid && !((valid[i >> 5] >> (i & 31)) & 1u)) continue;
    const u64 k = keys[i];
    const unsigned int len = (unsigned int)(k & 0xff);
    if (len > 7) bad |= 1;
    if (k & 0x8080808080808000ull) bad |= 2;
    mx = len > mx ? len : mx;
    mn = len < mn ? len : mn;
  }
  block_str_stats(mx, mn, bad, st);
}
// ColumnStore::delete_rows (store/core.rs:1392-1776): the rows leave the column; their positions stay as gaps
__global__ void clear_rows_kernel(unsigned int* __restrict__ valid, const u64* __restrict__ ids, u64 n, u64 origin, u64 n_rows) {
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
    const u64 pos = ids[i] - origin;
    if (ids[i] >= origin && pos < n_rows) atomicAnd(&valid[pos >> 5], ~(1u << (pos & 31)));
  }
}
// gather_row_window (llkv-column-map/src/store/projection.rs:929-1352) under GatherNullPolicy::IncludeNulls: the values of the
// given row ids in request order; a row id the column does not hold is NULL
template <typename T>
__global__ void gather_rows_kernel(const T* __restrict__ src, const unsigned int* __restrict__ valid, const u64* __restrict__ ids, u64 n, u64 origin,
                                   u64 n_rows, T* __restrict__ out, unsigned char* __restrict__ out_valid) {
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
    const u64 id = ids[i], pos = id - origin;
    const bool have = id >= origin && pos < n_rows && (!valid || ((valid[pos >> 5] >> (pos & 31)) & 1u));
    T v;
    memset(&v, 0, sizeof(T));
    if (have) v = src[pos];
    out[i] = v;
    out_valid[i] = have ? 1 : 0;
  }
}
__global__ void or_words_kernel(unsigned int* __restrict__ dst, const unsigned int* __restrict__ src, u64 n_words) {
  for (u64 w = (u64)blockIdx.x * blockDim.x + threadIdx.x; w < n_words; w += (u64)gridDim.x * blockDim.x) dst[w] |= src[w];
}
__global__ void popcount_bits_kernel(const unsigned int* __restrict__ bits, u64 n_bits, u64* __restrict__ out) {
  u64 c = 0;
  const u64 n_words = (n_bits + 31) / 32;
  for (u64 w = (u64)blockIdx.x * blockDim.x + threadIdx.x; w < n_words; w += (u64)gridDim.x * blockDim.x) {
    unsigned int v = bits[w];
    if (w == n_words - 1 && (n_bits & 31)) v &= (1u << (n_bits & 31)) - 1u;
    c += __popc(v);
  }
  for (int o = 16; o; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
  if ((threadIdx.x & 31) == 0 && c) atomicAdd(out, c);
}

// Wide GROUP BY keys (Plan::single_wide_key == 2): groups are keyed by a 64-bit hash of the keys' images.  After a run the
// verification pass recomputes every row's hash, finds its group and compares the row's key fields with those of the
// group's first row: two different keys in one group raise FLAG_KEY_COLLISION (the run is then an error, never a wrong
// answer).  The gather pass reads the key fields of each group's first row: that is where the key values come from.
struct WideKeyCols {
  const void* values[kMaxKeys];
  const unsigned int* validity[kMaxKeys];
  uint32_t load_kind[kMaxKeys];
  uint32_t n_keys;
};
__device__ __forceinline__ u64 wide_key_image(const WideKeyCols& c, int k, u64 pos, bool* isnull) {
  const unsigned int* v = c.validity[k];
  *isnull = v && !((v[pos >> 5] >> (pos & 31)) & 1u);
  const void* b = c.values[k];
  switch (c.load_kind[k]) {  // the image the scan kernels hash: (u64)(i64) of the value as they load it
    case LK_I8: return (u64)(i64) static_cast<const signed char*>(b)[pos];
    case LK_I16: return (u64)(i64) static_cast<const short*>(b)[pos];
    case LK_I32: case LK_D32: return (u64)(i64) static_cast<const int*>(b)[pos];
    case LK_U8: return (u64) static_cast<const unsigned char*>(b)[pos];
    case LK_U16: return (u64) static_cast<const unsigned short*>(b)[pos];
    case LK_U32: return (u64) static_cast<const unsigned int*>(b)[pos];
    case LK_STR8: return ((u64) static_cast<const unsigned char*>(b)[pos] << 56) | 1ull;
    default: return static_cast<const u64*>(b)[pos];
  }
}
__device__ __forceinline__ u64 wide_key_mix(u64 x) {  // = mix64 of device_util.cuh (the table's home-slot hash)
  x ^= x >> 33;
  x *= 0xff51afd7ed558ccdULL;
  x ^= x >> 33;
  x *= 0xc4ceb9fe1a85ec53ULL;
  x ^= x >> 33;
  return x;
}
__global__ void wide_key_verify_kernel(WideKeyCols c, u64 n_rows, u64 origin, const u64* __restrict__ gkeys, const u64* __restrict__ gwords, u64 gcap,
                                       uint32_t n_gwords, unsigned int* flag) {
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n_rows; i += (u64)gridDim.x * blockDim.x) {
    u64 img[kMaxKeys];
    bool nul[kMaxKeys];
    u64 K = key_hash_init();
    for (uint32_t k = 0; k < c.n_keys; ++k) {
      img[k] = wide_key_image(c, (int)k, i, &nul[k]);
      K = key_hash_step(K, img[k], nul[k]);
    }
    K = key_hash_done(K);
    const u64 mask = gcap - 1;
    u64 h = wide_key_mix(K) & mask;
    for (u64 probe = 0; probe <= mask; ++probe) {
      const u64 cur = gkeys[h];
      if (cur == kEmptyKey) break;  // no group has this hash: the row was not selected
      if (cur == K) {
        const u64 first = gwords[h * n_gwords + 1] - origin;  // (word 1: the group's first row id)
        if (first < n_rows && first != i) {
          bool same = true;
          for (uint32_t k = 0; k < c.n_keys; ++k) {
            bool fn;
            const u64 fi = wide_key_image(c, (int)k, first, &fn);
            same = same && fn == nul[k] && (fn || fi == img[k]);
          }
          if (!same) atomicOr(flag, 1u);
        }
        break;
      }
      h = (h + 1) & mask;
    }
  }
}
__global__ void wide_key_gather_kernel(WideKeyCols c, const u64* __restrict__ first_pos, u64 n_groups, u64 n_rows, u64* __restrict__ out_bits,
                                       unsigned char* __restrict__ out_null) {
  for (u64 g = (u64)blockIdx.x * blockDim.x + threadIdx.x; g < n_groups; g += (u64)gridDim.x * blockDim.x) {
    const u64 pos = first_pos[g];
    for (uint32_t k = 0; k < c.n_keys; ++k) {
      bool n = true;
      u64 v = 0;
      if (pos < n_rows) v = wide_key_image(c, (int)k, pos, &n);
      out_bits[g * c.n_keys + k] = n ? 0 : v;
      out_null[g * c.n_keys + k] = n ? 1 : 0;
    }
  }
}

// Sort index (SortIndexOps::stage_build_for_chunk, llkv-column-map/src/store/indexing/sort.rs:150-172): for every chunk the
// permutation that lists its rows in ascending value order (lexsort_to_indices).  One CTA sorts one chunk: a stable LSD radix
// sort over 4-bit digits of the order-preserving 64-bit image of the values, (key, index) pairs ping-ponging between two
// scratch buffers.  Every thread owns a contiguous segment of the chunk, counts its digits, a block-wide scan of the
// [digit][thread] counters gives each (digit, thread) its first output position, and the thread scatters its segment in
// order — which is what keeps equal keys in row order.  Index maintenance, not the scan path: a chunk is at most 1 MiB.
constexpr int kSortThreads = 512;
template <typename T, int KIND>  // KIND: 0 signed integer, 1 unsigned integer, 2 f32, 3 f64
__device__ __forceinline__ u64 sort_key_of(T v) {
  if (KIND == 0) return (u64)(i64)v ^ 0x8000000000000000ull;
  if (KIND == 1) return (u64)v;
  u64 b;
  if (KIND == 2) {
    const double d = (double)v;  // f32 through f64, as the reference's sortable encoding (codecs.rs:33-65)
    b = (u64)__double_as_longlong(d);
  } else {
    b = (u64)__double_as_longlong((double)v);
  }
  return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
template <typename T, int KIND>
__global__ void __launch_bounds__(kSortThreads) chunk_sort_kernel(const T* __restrict__ values, u64 n_rows, u64 chunk_rows, int passes, u64* key_a, u64* key_b,
                                                                  unsigned int* idx_a, unsigned int* idx_b, unsigned int* __restrict__ perm) {
  __shared__ unsigned int s_cnt[16][kSortThreads];
  __shared__ unsigned int s_part[kSortThreads];
  const u64 base = (u64)blockIdx.x * chunk_rows;
  if (base >= n_rows) return;
  const unsigned int m = (unsigned int)(n_rows - base < chunk_rows ? n_rows - base : chunk_rows);
  const unsigned int t = threadIdx.x;
  const unsigned int per = (m + kSortThreads - 1) / kSortThreads;
  const unsigned int lo = t * per < m ? t * per : m, hi = lo + per < m ? lo + per : m;
  u64* ka = key_a + base;
  u64* kb = key_b + base;
  unsigned int* ia = idx_a + base;
  unsigned int* ib = idx_b + base;
  for (unsigned int i = t; i < m; i += kSortThreads) {
    ka[i] = sort_key_of<T, KIND>(values[base + i]);
    ia[i] = i;
  }
  __syncthreads();
  for (int p = 0; p < passes; ++p) {
    const int shift = 4 * p;
    unsigned int c[16];
#pragma unroll
    for (int d = 0; d < 16; ++d) c[d] = 0;
    for (unsigned int i = lo; i < hi; ++i) {
      const unsigned int d = (unsigned int)(ka[i] >> shift) & 15u;
#pragma unroll
      for (int q = 0; q < 16; ++q) c[q] += (d == (unsigned)q);
    }
#pragma unroll
    for (int d = 0; d < 16; ++d) s_cnt[d][t] = c[d];
    __syncthreads();
    // exclusive scan of the 16 x kSortThreads counters in digit-major order: thread t owns counters [16 t, 16 t + 16)
    unsigned int* flat = &s_cnt[0][0];
    unsigned int sum = 0;
#pragma unroll
    for (int q = 0; q < 16; ++q) sum += flat[16 * t + q];
    unsigned int inc = sum;
    const unsigned int lane = t & 31, wid = t >> 5;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned int y = __shfl_up_sync(0xffffffffu, inc, o);
      if (lane >= (unsigned)o) inc += y;
    }
    if (lane == 31) s_part[wid] = inc;
    __syncthreads();
    unsigned int wbase = 0;
    for (unsigned int w = 0; w < wid; ++w) wbase += s_part[w];
    unsigned int run = wbase + inc - sum;
#pragma unroll
    for (int q = 0; q < 16; ++q) {
      const unsigned int v = flat[16 * t + q];
      flat[16 * t + q] = run;
      run += v;
    }
    __syncthreads();
#pragma unroll
    for (int d = 0; d < 16; ++d) c[d] = s_cnt[d][t];
    for (unsigned int i = lo; i < hi; ++i) {
      const u64 k = ka[i];
      const unsigned int d = (unsigned int)(k >> shift) & 15u;
      unsigned int dst = 0;
#pragma unroll
      for (int q = 0; q < 16; ++q)
        if (d == (unsigned)q) dst = c[q]++;
      kb[dst] = k;
      ib[dst] = ia[i];
    }
    __syncthreads();
    u64* tk = ka;
    ka = kb;
    kb = tk;
    unsigned int* ti = ia;
    ia = ib;
    ib = ti;
  }
  for (unsigned int i = t; i < m; i += kSortThreads) perm[base + i] = ia[i];
}

// Whole-column sort for sorted scans (ColumnStore::scan with ScanOptions::sorted, llkv-column-map/src/store/scan/sorted.rs:
// the reference merges its per-chunk value_order_perm runs on the CPU).  A stable LSD radix sort over 4-bit digits of the
// order-preserving key image across the whole grid: every thread of every CTA owns one contiguous segment, counts its
// digits (gsort_count), one CTA scans the [digit][segment] counters (gsort_scan), every thread scatters its segment in
// order (gsort_scatter) — equal keys keep row order.  Pass "-1" partitions by a flag instead of a digit: rows the column
// does not hold or that fall outside the requested value range go behind the others, which the digit passes then ignore.
constexpr unsigned kGsortThreads = 512;
__device__ __forceinline__ u64 gs_min(u64 a, u64 b) { return a < b ? a : b; }
template <typename T, int KIND>
__global__ void gsort_init_kernel(const T* __restrict__ v, const unsigned int* __restrict__ validity, u64 n, u64 lo, u64 hi, u64* __restrict__ key,
                                  unsigned int* __restrict__ idx, unsigned char* __restrict__ flag, u64* red) {
  u64 a = ~0ull, o = 0;
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
    const u64 k = sort_key_of<T, KIND>(v[i]);
    const bool keep = (!validity || ((validity[i >> 5] >> (i & 31)) & 1u)) && k >= lo && k <= hi;
    key[i] = k;
    idx[i] = (unsigned int)i;
    flag[i] = keep ? 0 : 1;
    if (keep) {
      a &= k;
      o |= k;
    }
  }
  for (int w = 16; w; w >>= 1) {
    a &= __shfl_xor_sync(0xffffffffu, a, w);
    o |= __shfl_xor_sync(0xffffffffu, o, w);
  }
  if ((threadIdx.x & 31) == 0) {
    atomicAnd((unsigned long long*)&red[0], (unsigned long long)a);
    atomicOr((unsigned long long*)&red[1], (unsigned long long)o);
  }
}
__device__ __forceinline__ unsigned gsort_digit(const u64* key, const unsigned char* flag, u64 i, int shift) {
  return shift < 0 ? (unsigned)flag[i] : (unsigned)(key[i] >> shift) & 15u;
}
__global__ void __launch_bounds__(kGsortThreads) gsort_count_kernel(const u64* __restrict__ key, const unsigned char* __restrict__ flag, u64 n, int shift,
                                                                    unsigned int* __restrict__ counts, u64 seg, unsigned S) {
  const unsigned g = blockIdx.x * kGsortThreads + threadIdx.x;
  const u64 lo = gs_min((u64)g * seg, n), hi = gs_min(lo + seg, n);
  unsigned c[16];
#pragma unroll
  for (int d = 0; d < 16; ++d) c[d] = 0;
  for (u64 i = lo; i < hi; ++i) {
    const unsigned d = gsort_digit(key, flag, i, shift);
#pragma unroll
    for (int q = 0; q < 16; ++q) c[q] += (d == (unsigned)q);
  }
#pragma unroll
  for (int d = 0; d < 16; ++d) counts[(size_t)d * S + g] = c[d];
}
__global__ void __launch_bounds__(1024) gsort_scan_kernel(unsigned int* counts, u64 total) {  // one CTA: exclusive scan in place
  __shared__ unsigned int part[1024];
  const u64 per = (total + 1023) / 1024;
  const u64 lo = gs_min((u64)threadIdx.x * per, total), hi = gs_min(lo + per, total);
  unsigned int sum = 0;
  for (u64 i = lo; i < hi; ++i) sum += counts[i];
  part[threadIdx.x] = sum;
  __syncthreads();
  for (unsigned o = 1; o < 1024; o <<= 1) {
    const unsigned int y = threadIdx.x >= o ? part[threadIdx.x - o] : 0;
    __syncthreads();
    part[threadIdx.x] += y;
    __syncthreads();
  }
  unsigned int run = part[threadIdx.x] - sum;
  for (u64 i = lo; i < hi; ++i) {
    const unsigned int v = counts[i];
    counts[i] = run;
    run += v;
  }
}
__global__ void __launch_bounds__(kGsortThreads) gsort_scatter_kernel(const u64* __restrict__ kin, const unsigned int* __restrict__ iin,
                                                                      const unsigned char* __restrict__ flag, u64 n, int shift,
                                                                      const unsigned int* __restrict__ counts, u64 seg, unsigned S, u64* __restrict__ kout,
                                                                      unsigned int* __restrict__ iout) {
  const unsigned g = blockIdx.x * kGsortThreads + threadIdx.x;
  const u64 lo = gs_min((u64)g * seg, n), hi = gs_min(lo + seg, n);
  unsigned c[16];
#pragma unroll
  for (int d = 0; d < 16; ++d) c[d] = counts[(size_t)d * S + g];
  for (u64 i = lo; i < hi; ++i) {
    const unsigned d = gsort_digit(kin, flag, i, shift);
    unsigned dst = 0;
#pragma unroll
    for (int q = 0; q < 16; ++q)
      if (d == (unsigned)q) dst = c[q]++;
    kout[dst] = kin[i];
    iout[dst] = iin[i];
  }
}

// ------------------------------------------------------------------------------------------------ handles
struct MvccState {
  llkv_gpu_column* created_by = nullptr;
  llkv_gpu_column* deleted_by = nullptr;
  uint64_t txn_id = 0, snapshot_id = 0;
  std::vector<uint64_t> noncommitted;
};

struct NcclIdByValue {  // ncclUniqueId
  char internal[128];
};
typedef int (*nccl_get_unique_id_fn)(void*);
typedef int (*nccl_comm_init_rank_fn)(void**, int, NcclIdByValue, int);
typedef int (*nccl_all_gather_fn)(const void*, void*, size_t, int, void*, cudaStream_t);
typedef int (*nccl_all_reduce_fn)(const void*, void*, size_t, int, int, void*, cudaStream_t);
typedef int (*nccl_comm_destroy_fn)(void*);
typedef const char* (*nccl_get_error_string_fn)(int);

struct NcclApi {
  void* lib = nullptr;
  nccl_get_unique_id_fn get_unique_id = nullptr;
  nccl_comm_init_rank_fn comm_init_rank = nullptr;
  nccl_all_gather_fn all_gather = nullptr;
  nccl_all_reduce_fn all_reduce = nullptr;
  nccl_comm_destroy_fn comm_destroy = nullptr;
  nccl_get_error_string_fn get_error_string = nullptr;
};
static NcclApi g_nccl;

static int32_t load_nccl() {
  if (g_nccl.lib) return LLKV_OK;
  // prefer a libnccl already mapped into the process (torch's bundled copy), then the system one
  void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD | RTLD_GLOBAL);
  if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
  if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
  if (!h) return set_error(LLKV_ERR_IO, "NCCL is not available: %s", dlerror());
  g_nccl.get_unique_id = (nccl_get_unique_id_fn)dlsym(h, "ncclGetUniqueId");
  g_nccl.comm_init_rank = (nccl_comm_init_rank_fn)dlsym(h, "ncclCommInitRank");
  g_nccl.all_gather = (nccl_all_gather_fn)dlsym(h, "ncclAllGather");
  g_nccl.all_reduce = (nccl_all_reduce_fn)dlsym(h, "ncclAllReduce");
  g_nccl.comm_destroy = (nccl_comm_destroy_fn)dlsym(h, "ncclCommDestroy");
  g_nccl.get_error_string = (nccl_get_error_string_fn)dlsym(h, "ncclGetErrorString");
  if (!g_nccl.get_unique_id || !g_nccl.comm_init_rank || !g_nccl.all_gather || !g_nccl.all_reduce || !g_nccl.comm_destroy)
    return set_error(LLKV_ERR_IO, "libnccl lacks the expected symbols");
  g_nccl.lib = h;
  return LLKV_OK;
}
#define NCCL_TRY(expr)                                                                                                   \
  do {                                                                                                                   \
    int _r = (expr);                                                                                                     \
    if (_r != 0) return set_error(LLKV_ERR_IO, "NCCL error %d (%s) at %s:%d", _r,                                         \
                                  g_nccl.get_error_string ? g_nccl.get_error_string(_r) : "?", __FILE__, __LINE__);        \
  } while (0)

struct llkv_gpu_ctx {
  int device = 0;
  int sm_count = 148;
  int max_smem = 227 * 1024;
  cudaStream_t stream = nullptr;
  std::vector<cudaStream_t> copy_streams;
  std::vector<cudaEvent_t> slot_events;
  unsigned char* pinned = nullptr;
  uint64_t slot_bytes = 0;
  int next_slot = 0;
  std::map<uint64_t, llkv_gpu_column*> columns;  // LogicalFieldId -> column
  std::map<uint64_t, MvccState> mvcc;            // table id -> snapshot
  struct ExistsCache {  // row-id-sparse tables without MVCC columns: OR of the columns' validity bitmaps
    unsigned int* bits = nullptr;
    uint64_t words = 0, key = 0;
  };
  std::map<uint64_t, ExistsCache> exists;        // table id -> bitmap
  bool timing = false;
  int tune_ctas = 0, tune_block = 0, tune_stages = 0, tune_rpt = 0, tune_force_wide = 0;
  int jit_mode = 1;  // 0 never, 1 specialise a plan shape from its second run on, 2 always
  int partition_mode = 1;  // partitioned high-cardinality GROUP BY: 0 never, 1 when the table exceeds L2, 2 whenever possible,
                           // 3 as 2 but never in packed tuples
  int prune_mode = 1;      // zone-map tile skipping: 0 never, 1 columns scanned again unchanged + >= 1/8 of the tiles, 2 always
  std::map<std::string, uint32_t> shape_runs;
  bool keep_wide_decimals = false;  // LLKV_GPU_KEEP_WIDE_DECIMALS=1: never narrow Decimal128 columns at seal
  bool no_d32 = false;              // LLKV_GPU_NO_D32=1: narrow to i64 only (experiments)
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  cudaEvent_t ev2 = nullptr, ev3 = nullptr;  // around the peer-mailbox merge kernel (timing)
  void* nccl_comm = nullptr;
  int n_ranks = 1, rank = 0;
  // peer-memory mailboxes for the ungrouped merge (scan_kernel.cu: merge_ungrouped_p2p_kernel): every rank maps every
  // other rank's mailbox through CUDA IPC at llkv_gpu_comm_init; all ranks use this path or none does
  u64* mbox = nullptr;            // this rank's mailbox: [n_ranks][2][128] words, then [n_ranks][2][kGroupSlotWords]
  u64* peer_gbox[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};  // the group-table region of every rank's mailbox
  u64* peer_mbox[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  bool p2p_merge = false;
  u64* d_epoch = nullptr;  // merges so far, in device memory (the merge kernels advance it: their launches carry no per-merge value)
  // Calls that share this context's state (column registry, staging ring, stream, snapshots, plan cache) are serialised
  // here, so handles of one context may be used from several threads (the Rust wrapper's `Sync`).
  std::recursive_mutex mu;
  uint64_t state_epoch = 1;  // bumped by every call that can change what a compiled plan depends on (columns, snapshots, knobs)
  int graph_mode = 1;        // llkv_gpu_agg_execute: 1 = replay a captured CUDA graph once a step repeats unchanged, 0 = never
  // host workers that narrow Decimal128 chunks from page-locked sources before the DMA (upload.h); created on first use
  int upload_threads = -1;  // -1 = default (min(32, hardware threads - 1)), 0 = never narrow on the host
  int dma_share = -1;       // percent of the Decimal128 bytes of a hybrid upload that take the copy engine; -1 = from the thread count
  std::unique_ptr<UploadPool> pool;
};
#define CTX_LOCK(c) std::lock_guard<std::recursive_mutex> _ctx_lock((c)->mu)

// live contexts: llkv_gpu_host_free / _host_unregister must not pull memory from under a copy that is still pending
static std::mutex g_registry_mu;
static std::vector<llkv_gpu_ctx*> g_contexts;

struct NarrowChunk {  // a chunk appended through the host-narrowing path since the last seal (re-uploaded wide on failure)
  const void* src;
  uint64_t first_row, n_rows;
};

// Dictionary of a Utf8 column that holds strings longer than the 7 bytes of a packed key (llkv_gpu.h, "Utf8 columns").
// Ids are handed out in order of first appearance by the host side of append; seal orders the entries byte-wise and turns
// the resident codes into ranks.  Between seals codes below `sealed` are ranks, codes from `sealed` up are raw ids.
struct StrDict {
  std::deque<std::string> strings;  // by id; a deque keeps the addresses the map's keys point to
  std::unordered_map<std::string_view, uint32_t> id_of;
  std::vector<uint32_t> rank_of_id, id_of_rank;  // over ids < sealed
  std::vector<std::string> sorted;               // by rank: what plans search and finalize decodes
  uint32_t sealed = 0;
  uint64_t epoch = 0;
  bool non_ascii = false;
  uint32_t intern(const char* p, size_t n) {
    auto it = id_of.find(std::string_view(p, n));
    if (it != id_of.end()) return it->second;
    strings.emplace_back(p, n);
    const uint32_t id = (uint32_t)strings.size() - 1;
    id_of.emplace(std::string_view(strings.back()), id);
    for (size_t i = 0; i < n && !non_ascii; ++i) non_ascii = (unsigned char)p[i] >= 0x80;
    return id;
  }
  uint64_t code_of(uint32_t id) const { return id < sealed ? rank_of_id[id] : id; }
};
constexpr size_t kMaxDictEntries = 1u << 24;

struct llkv_gpu_column {
  llkv_gpu_ctx* ctx = nullptr;
  std::unique_ptr<StrDict> dict;
  // Hybrid upload of Decimal128 chunks from page-locked memory: the host workers narrow their share before the DMA, the
  // pool's DMA thread takes the rest as it lies (16 B/value) and a kernel narrows it on the device; both feed the same
  // narrow column.
  unsigned int* d_fit = nullptr;  // device flag: a value of the DMA share did not fit
  bool dma_used = false;
  uint64_t lfid = 0;
  int32_t type = 0;
  uint8_t precision = 0;
  int8_t scale = 0;
  void* values = nullptr;
  unsigned int* validity = nullptr;
  uint64_t cap_rows = 0;
  uint64_t n_rows = 0;
  uint32_t elem_bytes = 0;
  uint8_t load_kind = 0;
  DevStats* dstats = nullptr;
  DevStats hstats;
  bool sealed = false;
  bool has_origin = false;
  uint64_t row_id_origin = 0;
  int stream_index = 0;
  uint64_t stats_rows = 0;  // rows already covered by the statistics pass (run at seal, not per chunk)
  // Decimal128 narrowing: `values` is what scans read.  While narrow (LK_D64) the Arrow-layout landing buffer can stay
  // allocated (`landing`, after a clear(): the caller re-uploads the column every batch) so no allocation happens per batch.
  void* landing = nullptr;     // parked Arrow-layout buffer (16 B per row), capacity landing_cap rows
  uint64_t landing_cap = 0;
  void* narrow = nullptr;      // parked narrow buffer (narrow_width bytes per row), capacity narrow_cap rows
  uint64_t narrow_cap = 0;
  uint32_t narrow_width = 8;
  bool reupload_hint = false;  // set by clear(): keep both buffers across batches
  // host-side narrowing of page-locked Decimal128 chunks (upload.h): the width tried next (-1 = look at the first chunk,
  // -2 = a chunk did not fit i64: never again for this column), the jobs in flight, the chunks since the last seal
  int host_kind = -1;
  UploadTicket ticket;
  std::vector<NarrowChunk> narrow_chunks;
  uint64_t h2d_bytes = 0;      // bytes this column's appends put on the link since it was registered
  unsigned int* d_perm = nullptr;  // sort index: per chunk of perm_chunk_rows rows, the rows in ascending value order
  uint64_t perm_chunk_rows = 0, perm_version = 0;
  bool sparse = false;         // some chunk arrived with row ids that do not continue the column: positions = row id - origin,
                               // absent rows are invalid bits, statistics are recomputed over the whole column at seal
  // pending coalesced upload from page-locked host memory (upload() / flush_upload())
  void* pend_dst = nullptr;
  const void* pend_src = nullptr;
  uint64_t pend_bytes = 0;
  std::vector<void*> deferred_free;  // temp device buffers released at seal
  // zone maps (minimum / maximum per kZoneRows rows, as the 64-bit values the lean kernel's leaves compare), computed on
  // the device when a scan first wants them and mirrored on the host, where tile lists are built
  uint64_t version = 1;          // bumped whenever the content changes (append, clear)
  uint64_t zones_version = 0;    // content version h_zones describes
  u64* d_zones = nullptr;
  size_t d_zones_cap = 0;        // zones
  std::vector<u64> h_zones;      // [zone][min, max]
  uint32_t scans_unchanged = 0;  // fused scans with a range leaf on this column since the content last changed
};

// String literals passed by reference are copied into storage the receiving handle owns (shared: handles are copied)
typedef std::shared_ptr<std::deque<std::string>> StringStore;
static void own_string_literal(llkv_literal& l, StringStore& store) {
  if (l.kind != LLKV_LIT_STRING || l.precision != LLKV_LIT_STRING_BY_REF) return;
  if (!store) store = std::make_shared<std::deque<std::string>>();
  store->emplace_back(reinterpret_cast<const char*>(static_cast<uintptr_t>(l.lo)), static_cast<size_t>(l.hi));
  l.lo = static_cast<uint64_t>(reinterpret_cast<uintptr_t>(store->back().data()));
}

struct llkv_gpu_program {
  uint64_t serial = 0;  // identity of the compiled program (handles can be freed and their addresses reused)
  StringStore strings;
  std::vector<llkv_eval_op> ops;
  std::vector<llkv_literal> literals;
  std::vector<llkv_scalar_node> nodes;
  std::vector<int32_t> list_roots;
  ProgramView view;
  void bind() {
    view.ops = ops.data();
    view.n_ops = (int32_t)ops.size();
    view.literals = literals.data();
    view.n_literals = (int32_t)literals.size();
    view.nodes = nodes.data();
    view.n_nodes = (int32_t)nodes.size();
    view.list_roots = list_roots.data();
    view.n_list_roots = (int32_t)list_roots.size();
  }
};

struct PendingRun {
  bool active = false;
  bool has_prog = false;
  llkv_gpu_program prog;
  int apply_mvcc = 0;
  uint64_t row_begin = 0, row_end = 0;
  bool wide = false;
  bool has_backup = false;
  bool timed = false;
  bool is_merge = false;  // a grouped peer-mailbox merge is queued behind the run (agg_resolve settles both)
  bool timed_merge = false;
  bool from_reset = false;  // the run started from the initial state: a rerun re-initialises instead of restoring a backup
};

// The forms a lean plan runs in: the interpreting build, the build specialised on the plan shape, and the two partitioned
// forms of a high-cardinality GROUP BY (specialised builds only) — multi-field tuples, and packed tuples
enum LeanForm { LEAN_INTERPRETED, LEAN_SPECIALISED, LEAN_PARTITIONED, LEAN_PACKED, kLeanForms };
struct LeanFormGeometry {
  LeanPlan plan;
  uint32_t grid = 0, ctas = 1;
  bool have = false;
};

// Partition layout of the packed form.  Dense integer keys (the packed key range is within 4x the expected groups) make a
// partition a key range whose shared-memory slots are indexed directly; otherwise partitions are ranges of the key's hash
// with a small open-addressing table in shared memory (load factor <= 1/2 when the keys spread evenly).
struct PackedLayout {
  uint32_t parts = 0, shift = 0, slots = 0, dense = 0, key_bits = 0, row_bits = 0, n_ops = 0;
  uint32_t op_bits[8] = {0, 0, 0, 0, 0, 0, 0, 0};
};

struct llkv_gpu_agg {
  llkv_gpu_ctx* ctx = nullptr;
  StringStore strings;
  uint64_t dict_agreed_epoch = ~0ull;  // context state the ranks last agreed their key dictionaries at
  uint64_t runs_done = 0, wide_verified = ~0ull;  // hashed wide keys: the run the verification pass last covered
  uint64_t table_id = 0;
  std::vector<llkv_agg_spec> specs;
  std::vector<llkv_scalar_node> nodes;
  std::vector<uint64_t> keys;
  int32_t expr_mode = LLKV_EXPR_ARROW;
  uint64_t hint = 0;
  uint64_t observed_groups = 0;  // groups a finalize has seen: the next run sizes its CTA-local slot table for at least that many
  // accumulator state
  bool frozen = false;
  uint32_t n_gwords = 0;
  std::vector<uint8_t> gclass;
  uint8_t* d_gclass = nullptr;
  u64 gcap = 0;
  u64* gkeys = nullptr;
  u64* gwords = nullptr;
  u64* bk_keys = nullptr;
  u64* bk_words = nullptr;
  u64 bk_cap = 0;
  // gather buffers of the multi-GPU merge, kept across calls
  u64* mg_keys = nullptr;
  u64* mg_words = nullptr;
  size_t mg_key_elems = 0, mg_word_elems = 0;
  u64* mg_cap = nullptr;
  u64* mg_stats = nullptr;  // scratch of agree_key_stats
  size_t mg_stats_elems = 0;
  std::vector<u64> agreed_stats;  // what the ranks agreed on in the current run (reused by this rank's reruns)
  uint64_t agreed_epoch = 0;      // ctx->state_epoch at that time
  bool in_rerun = false;
  // the lean plan of the previous run, reusable while request_signature() does not change
  LeanPlan lean;
  LeanFormGeometry forms[kLeanForms];  // the geometry of each form, computed when a run first asks for it
  PackedLayout packed;                 // packed form: partition layout of the current plan
  void forget_forms() {
    for (LeanFormGeometry& f : forms) f.have = false;
  }
  // partitioned high-cardinality GROUP BY: tuple partitions and their fill counters, kept across runs
  u64* part_out = nullptr;
  size_t part_out_elems = 0;
  uint32_t* part_cursor = nullptr;
  // zone-map pruning: the surviving tiles of the last pruned scan (reused while its key — plan, geometry, row range and
  // the content versions of the predicate columns — does not change)
  uint32_t* d_tile_list = nullptr;
  size_t tile_list_cap = 0;
  std::vector<uint32_t> h_tile_list;
  uint64_t tile_list_key = 0;
  uint64_t tile_list_total = 0;
  bool tile_list_use = false;
  uint64_t lean_sig = 0;
  uint32_t lean_jit_runs = 0;
  uint32_t* d_flags = nullptr;
  uint32_t* h_flags = nullptr;  // pinned
  unsigned char* h_stage = nullptr;  // pinned landing buffer of finalize (small tables)
  size_t h_stage_bytes = 0;
  bool prefetched = false;  // h_stage holds the table as the last run left it (copy queued right behind the scan)
  // One-kernel steps (step_publishes): `armed` = in stream order the status word, ticket and table hold their initial values,
  // so a reset queues nothing.  `published` = the last run's scan copied its status word and table to h_pub (page-locked,
  // mapped: [status][words][keys]) and re-armed the device state; h_pub is the result until something continues from it.
  bool armed = false;
  bool published = false;
  u64* h_pub = nullptr;
  u64* d_pub = nullptr;
  cudaEvent_t stage_ev = nullptr;  // recorded behind that copy
  Plan* d_plan = nullptr;
  Plan* h_plan = nullptr;  // pinned
  CompileResult cr;
  PendingRun pending;
  bool reset_pending = false;   // llkv_gpu_agg_reset is applied by whatever touches the state next (in stream order)
  uint64_t plan_epoch = 1;      // bumped when this aggregate's own launch state changes (table grown, geometry re-chosen)
  // llkv_gpu_agg_execute: one step = reset -> scan -> [merge] -> result copy.  Once a step repeats with nothing changed
  // it is captured as a CUDA graph and replayed: one launch call per step.
  uint64_t exec_key = 0;
  uint32_t exec_same = 0;       // consecutive clean steps with this key
  cudaGraphExec_t graph_exec = nullptr;
  uint64_t graph_key = 0;
  PendingRun graph_pending;     // the pending-run bookkeeping of the captured step (without the program copy)
  bool graph_prefetched = false;
  bool graph_from_armed = false;  // the captured step has no reset launches: it replays only onto an armed state
  bool graph_published = false, graph_armed_after = false;
  uint32_t graph_launches = 0;
  bool in_capture = false;
  uint32_t capture_failures = 0;
  bool stage_ev_valid = false;
  // output shaping at finalize (llkv_gpu_agg_set_output): HAVING terms, ORDER BY keys, OFFSET / LIMIT
  std::vector<llkv_having_term> having;
  std::vector<llkv_order_key> order;
  uint64_t out_offset = 0, out_limit = 0;
  // DISTINCT aggregates: the distinct values are the groups of an inner aggregation over the argument column
  llkv_gpu_agg* inner = nullptr;
  bool skip_scan_copy = false;      // llkv_gpu_agg_execute with a peer-mailbox merge behind the scan: the merge queues the result copy
  bool p2p_group_disabled = false;  // a rank's group table outgrew a mailbox slot once: this aggregate merges over NCCL from then on
  int32_t err_code = 0;
  std::string err_msg;
  llkv_run_info info;
};

// ------------------------------------------------------------------------------------------------ library / context
extern "C" int32_t llkv_gpu_abi_version(void) { return LLKV_GPU_ABI_VERSION; }

extern "C" size_t llkv_gpu_last_error(char* buf, size_t cap) {
  if (buf && cap) {
    const size_t n = g_last_error.size() < cap - 1 ? g_last_error.size() : cap - 1;
    memcpy(buf, g_last_error.data(), n);
    buf[n] = 0;
  }
  return g_last_error.size();
}

extern "C" int32_t llkv_gpu_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

extern "C" int32_t llkv_gpu_ctx_create(int32_t device_ordinal, int32_t n_streams, uint64_t pinned_bytes, llkv_gpu_ctx** out) {
  if (!out) return set_error(LLKV_ERR_INVALID_ARGUMENT, "out is NULL");
  *out = nullptr;
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n <= 0) {
    cudaGetLastError();
    return set_error(LLKV_ERR_IO, "no CUDA device available (%s): this library has no CPU fallback",
                     e != cudaSuccess ? cudaGetErrorString(e) : "device count 0");
  }
  if (device_ordinal < 0 || device_ordinal >= n) return set_error(LLKV_ERR_INVALID_ARGUMENT, "device ordinal %d out of range (%d devices)", device_ordinal, n);
  CUDA_TRY(cudaSetDevice(device_ordinal));
  cudaDeviceProp prop;
  CUDA_TRY(cudaGetDeviceProperties(&prop, device_ordinal));
  if (prop.major < 10) return set_error(LLKV_ERR_IO, "device %d is sm_%d%d; this library is built for sm_100a only", device_ordinal, prop.major, prop.minor);
  llkv_gpu_ctx* c = new llkv_gpu_ctx();
  c->device = device_ordinal;
  c->sm_count = prop.multiProcessorCount;
  c->max_smem = (int)prop.sharedMemPerBlockOptin;
  {
    const char* e = getenv("LLKV_GPU_KEEP_WIDE_DECIMALS");
    c->keep_wide_decimals = e && e[0] == '1';
    const char* e32 = getenv("LLKV_GPU_NO_D32");
    c->no_d32 = e32 && e32[0] == '1';
    const char* ed = getenv("LLKV_GPU_DMA_SHARE");  // percent (experiments)
    if (ed && ed[0]) c->dma_share = std::max(-1, std::min(100, atoi(ed)));
    const char* eg = getenv("LLKV_GPU_NO_GRAPHS");  // (profilers that want plain launches)
    if (eg && eg[0] == '1') c->graph_mode = 0;
  }
  if (n_streams < 1) n_streams = 2;
  if (n_streams > 16) n_streams = 16;
  if (pinned_bytes < ((uint64_t)n_streams << 20)) pinned_bytes = (uint64_t)n_streams << 22;
  CUDA_TRY(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
  c->copy_streams.resize((size_t)n_streams);
  c->slot_events.resize((size_t)n_streams);
  for (int i = 0; i < n_streams; ++i) {
    CUDA_TRY(cudaStreamCreateWithFlags(&c->copy_streams[(size_t)i], cudaStreamNonBlocking));
    CUDA_TRY(cudaEventCreateWithFlags(&c->slot_events[(size_t)i], cudaEventDisableTiming));
  }
  c->slot_bytes = (pinned_bytes / (uint64_t)n_streams) & ~(uint64_t)255;
  CUDA_TRY(cudaHostAlloc((void**)&c->pinned, c->slot_bytes * (uint64_t)n_streams, cudaHostAllocDefault));
  CUDA_TRY(cudaEventCreate(&c->ev0));
  CUDA_TRY(cudaEventCreate(&c->ev1));
  CUDA_TRY(cudaEventCreate(&c->ev2));
  CUDA_TRY(cudaEventCreate(&c->ev3));
  {
    std::lock_guard<std::mutex> lk(g_registry_mu);
    g_contexts.push_back(c);
  }
  *out = c;
  return LLKV_OK;
}

static void comm_teardown_p2p(llkv_gpu_ctx* ctx);
extern "C" void llkv_gpu_ctx_destroy(llkv_gpu_ctx* c) {
  if (!c) return;
  {
    std::lock_guard<std::mutex> lk(g_registry_mu);
    g_contexts.erase(std::remove(g_contexts.begin(), g_contexts.end(), c), g_contexts.end());
  }
  cudaSetDevice(c->device);
  cudaDeviceSynchronize();
  std::vector<llkv_gpu_column*> cols;
  for (auto& kv : c->columns) cols.push_back(kv.second);
  for (llkv_gpu_column* col : cols) llkv_gpu_column_destroy(col);
  c->pool.reset();
  if (c->nccl_comm && g_nccl.comm_destroy) {
    comm_teardown_p2p(c);
    g_nccl.comm_destroy(c->nccl_comm);
  }
  for (cudaStream_t s : c->copy_streams) cudaStreamDestroy(s);
  for (cudaEvent_t e : c->slot_events) cudaEventDestroy(e);
  if (c->stream) cudaStreamDestroy(c->stream);
  if (c->pinned) cudaFreeHost(c->pinned);
  if (c->ev0) cudaEventDestroy(c->ev0);
  if (c->ev1) cudaEventDestroy(c->ev1);
  if (c->ev2) cudaEventDestroy(c->ev2);
  if (c->ev3) cudaEventDestroy(c->ev3);
  delete c;
}

extern "C" int32_t llkv_gpu_ctx_synchronize(llkv_gpu_ctx* c) {
  if (!c) return set_error(LLKV_ERR_INVALID_ARGUMENT, "ctx is NULL");
  CTX_LOCK(c);
  CUDA_TRY(cudaSetDevice(c->device));
  for (cudaStream_t s : c->copy_streams) CUDA_TRY(cudaStreamSynchronize(s));
  CUDA_TRY(cudaStreamSynchronize(c->stream));
  return LLKV_OK;
}

extern "C" int32_t llkv_gpu_ctx_stream(llkv_gpu_ctx* c, void** out_stream) {
  if (!c || !out_stream) return set_error(LLKV_ERR_INVALID_ARGUMENT, "NULL argument");
  *out_stream = (void*)c->stream;
  return LLKV_OK;
}

extern "C" int32_t llkv_gpu_ctx_set_timing(llkv_gpu_ctx* c, int32_t enabled) {
  if (!c) return set_error(LLKV_ERR_INVALID_ARGUMENT, "ctx is NULL");
  c->timing = enabled != 0;
  ++c->state_epoch;
  return LLKV_OK;
}

extern "C" int32_t llkv_gpu_ctx_set_jit(llkv_gpu_ctx* c, int32_t mode) {
  if (!c) return set_error(LLKV_ERR_INVALID_ARGUMENT, "ctx is NULL");
  if (mode < 0 || mode > 2) return set_error(LLKV_ERR_INVALID_ARGUMENT, "jit mode must be 0, 1 or 2");
  c->jit_mode = mode;
  ++c->state_epoch;
  return LLKV_OK;
}

extern "C" int32_t llkv_gpu_ctx_set_partitioning(llkv_gpu_ctx* c, int32_t mode) {
  if (!c) return set_error(LLKV_ERR_INVALID_ARGUMENT, "ctx is NULL");
  if (mode < 0 || mode > 3) return set_error(LLKV_ERR_INVALID_ARGUMENT, "partitioning mode must be 0, 1, 2 or 3");
  c->partition_mode = mode;
  ++c->state_epoch;
  return LLKV_OK;
}

extern "C" int32_t llkv_gpu_ctx_set_pruning(llkv_gpu_ctx* c, int32_t mode) {
  if (!c) return set_error(LLKV_ERR_INVALID_ARGUMENT, "ctx is NULL");
  if (mode < 0 || mode > 2) return set_error(LLKV_ERR_INVALID_ARGUMENT, "pruning mode must be 0, 1 or 2");
  c->prune_mode = mode;
  ++c->state_epoch;
  return LLKV_OK;
}

extern "C" int32_t llkv_gpu_ctx_set_tuning(llkv_gpu_ctx* c, int32_t ctas_per_sm, int32_t block_threads, int32_t stages,
                                            int32_t rows_per_thread, int32_t force_wide) {
  if (!c) return set_error(LLKV_ERR_INVALID_ARGUMENT, "ctx is NULL");
  if (block_threads && (block_threads < 32 || block_threads > 512 || (block_threads & 31)))
    return set_error(LLKV_ERR_INVALID_ARGUMENT, "block_threads must be a multiple of 32 in [32, 512]");
  if (rows_per_thread && rows_per_thread != 1 && rows_per_thread != 2 && rows_per_thread != 4 && rows_per_thread != 8)
    return set_error(LLKV_ERR_INVALID_ARGUMENT, "rows_per_thread must be 1, 2, 4 or 8");
  if (stages < 0 || stages > 8 || ctas_per_sm < 0 || ctas_per_sm > 8) return set_error(LLKV_ERR_INVALID_ARGUMENT, "tuning value out of range");
  c->tune_ctas = ctas_per_sm;
  c->tune_block = block_threads;
  c->tune_stages = stages;
  c->tune_rpt = rows_per_thread;
  c->tune_force_wide = force_wide;
  ++c->state_epoch;
  return LLKV_OK;
}

extern "C" int32_t llkv_gpu_host_alloc(uint64_t bytes, void** out) {
  if (!out) return set_error(LLKV_ERR_INVALID_ARGUMENT, "out is NULL");
  CUDA_TRY(cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocDefault));
  return LLKV_OK;
}
extern "C" int32_t llkv_gpu_host_register(const void* p, uint64_t bytes) {
  if (!p || !bytes) return set_error(LLKV_ERR_INVALID_ARGUMENT, "nothing to register");
  cudaError_t e = cudaHostRegister(const_cast<void*>(p), bytes, cudaHostRegisterPortable | cudaHostRegisterReadOnly);
  if (e != cudaSuccess) {  // (read-only registration needs driver support; plain registration needs a writable mapping)
    cudaGetLastError();
    e = cudaHostRegister(const_cast<void*>(p), bytes, cudaHostRegisterPortable);
  }
  if (e != cudaSuccess) {
    cudaGetLastError();
    return set_error(LLKV_ERR_IO, "cudaHostRegister: %s", cudaGetErrorString(e));
  }
  return LLKV_OK;
}
// Page-locked memory is about to go away: every copy an append left pending (coalesced DMA, host-narrowing jobs) may
// still read it, so all of them are issued and waited for first.
static int32_t column_flush(llkv_gpu_column* col);
static int32_t flush_all_pending() {
  std::vector<llkv_gpu_ctx*> ctxs;
  {
    std::lock_guard<std::mutex> lk(g_registry_mu);
    ctxs = g_contexts;
  }
  int cur = 0;
  cudaGetDevice(&cur);
  int32_t first = LLKV_OK;
  for (llkv_gpu_ctx* c : ctxs) {
    CTX_LOCK(c);
    if (cudaSetDevice(c->device) != cudaSuccess) continue;
    for (auto& kv : c->columns) {
      llkv_gpu_column* col = kv.second;
      if (!col->pend_bytes && col->narrow_chunks.empty() && col->ticket.outstanding.load() == 0) continue;
      const int32_t rc = column_flush(col);
      if (rc && !first) first = rc;
    }
  }
  cudaSetDevice(cur);
  return first;
}
extern "C" int32_t llkv_gpu_host_unregister(const void* p) {
  if (!p) return LLKV_OK;
  int32_t rc = flush_all_pending();
  if (rc) return rc;
  CUDA_TRY(cudaHostUnregister(const_cast<void*>(p)));
  return LLKV_OK;
}

extern "C" int32_t llkv_gpu_host_free(void* p) {
  if (!p) return LLKV_OK;
  int32_t rc = flush_all_pending();
  if (rc) return rc;
  CUDA_TRY(cudaFreeHost(p));
  return LLKV_OK;
}

extern "C" int32_t llkv_gpu_ctx_set_upload_threads(llkv_gpu_ctx* c, int32_t n_threads) {
  if (!c) return set_error(LLKV_ERR_INVALID_ARGUMENT, "ctx is NULL");
  if (n_threads < -1 || n_threads > 64) return set_error(LLKV_ERR_INVALID_ARGUMENT, "upload threads must be -1 (default), 0 (off) or 1..64");
  CTX_LOCK(c);
  if (c->pool && c->pool->threads() != n_threads) {
    for (auto& kv : c->columns) {
      const int32_t rc = column_flush(kv.second);
      if (rc) return rc;
    }
    c->pool.reset();
  }
  c->upload_threads = n_threads;
  return LLKV_OK;
}

extern "C" int32_t llkv_gpu_ctx_set_dma_share(llkv_gpu_ctx* c, int32_t percent) {
  if (!c) return set_error(LLKV_ERR_INVALID_ARGUMENT, "ctx is NULL");
  if (percent < -1 || percent > 100) return set_error(LLKV_ERR_INVALID_ARGUMENT, "the DMA share is -1 (from the worker count) or 0..100 percent");
  CTX_LOCK(c);
  for (auto& kv : c->columns) {
    const int32_t rc = column_flush(kv.second);
    if (rc) return rc;
  }
  c->dma_share = percent;
  return LLKV_OK;
}

// ------------------------------------------------------------------------------------------------ columns
static uint32_t device_elem_bytes(int32_t type) {
  if (type == LLKV_PT_UTF8) return 8;
  return (uint32_t)prim_type_width(type);
}
static uint8_t device_load_kind(int32_t type) {
  switch (type) {
    case LLKV_PT_INT8: return LK_I8;
    case LLKV_PT_INT16: return LK_I16;
    case LLKV_PT_INT32: case LLKV_PT_DATE32: return LK_I32;
    case LLKV_PT_INT64: case LLKV_PT_DATE64: return LK_I64;
    case LLKV_PT_UINT8: case LLKV_PT_BOOLEAN: return LK_U8;
    case LLKV_PT_UINT16: return LK_U16;
    case LLKV_PT_UINT32: return LK_U32;
    case LLKV_PT_UINT64: case LLKV_PT_UTF8: return LK_U64;
    case LLKV_PT_FLOAT32: return LK_F32;
    case LLKV_PT_FLOAT64: return LK_F64;
    default: return LK_D128;
  }
}
static bool is_narrow_decimal(const llkv_gpu_column* col) { return col->load_kind == LK_D64 || col->load_kind == LK_D32; }

extern "C" int32_t llkv_gpu_column_register(llkv_gpu_ctx* c, uint64_t lfid, int32_t prim_type, uint8_t precision, int8_t scale,
                                             llkv_gpu_column** out) {
  if (!c || !out) return set_error(LLKV_ERR_INVALID_ARGUMENT, "NULL argument");
  CTX_LOCK(c);
  *out = nullptr;
  if (device_elem_bytes(prim_type) == 0) return set_error(LLKV_ERR_INVALID_ARGUMENT, "column type %d does not cross this boundary", prim_type);
  if (prim_type == LLKV_PT_DECIMAL128 && (precision < 1 || precision > 38)) return set_error(LLKV_ERR_INVALID_ARGUMENT, "Decimal128 precision %d out of range", precision);
  if (c->columns.count(lfid)) return set_error(LLKV_ERR_INVALID_ARGUMENT, "column %llu is already registered", (unsigned long long)lfid);
  CUDA_TRY(cudaSetDevice(c->device));
  llkv_gpu_column* col = new llkv_gpu_column();
  col->ctx = c;
  col->lfid = lfid;
  col->type = prim_type;
  col->precision = precision;
  col->scale = scale;
  col->elem_bytes = device_elem_bytes(prim_type);
  col->load_kind = device_load_kind(prim_type);
  col->stream_index = (int)(c->columns.size() % c->copy_streams.size());
  DevStats init;
  memset(&init, 0, sizeof(init));
  init.min_enc = ~0ull;
  init.min_strlen = 0xffffffffu;
  col->hstats = init;
  cudaError_t e = cudaMalloc((void**)&col->dstats, sizeof(DevStats));
  if (e == cudaSuccess) e = cudaMemcpy(col->dstats, &init, sizeof(init), cudaMemcpyHostToDevice);
  if (e != cudaSuccess) {
    delete col;
    return set_error(LLKV_ERR_IO, "CUDA error %s allocating column state", cudaGetErrorString(e));
  }
  c->columns[lfid] = col;
  ++c->state_epoch;
  *out = col;
  return LLKV_OK;
}

// Issues the column's pending coalesced host->device copy (see upload()).  Must run before anything on the column's
// stream reads or moves the destination: follow-up kernels, seal, grow, clear, destroy.
// Which way a Decimal128 chunk of a hybrid upload goes: by 8 MiB blocks of the column's Arrow image, so that the chunks of
// one block form one copy, `share` percent of the blocks to the copy engine.
static bool route_to_dma(const llkv_gpu_column* col, uint64_t first_row) {
  const llkv_gpu_ctx* c = col->ctx;
  int share = c->dma_share;
  if (share < 0) {
    // Both ways read the column's Arrow bytes from host memory, and that is the shared limit: measured on the 16-core hosts of
    // this pool a worker streams about 6.4 GB/s and the host's memory system gives out near 78 GB/s in total (15 workers:
    // 37 ms per 2.9 GB with or without help from the copy engine; 8 workers: 56 ms alone, 48 ms with half the bytes on the
    // copy engine).  The copy engine gets what the workers leave of that budget.
    // (6.4 GB/s is the SSE2 form of the narrowing loop; the AVX2 / AVX-512 forms with their software prefetch stream about
    // 11 GB/s per worker, so from eight workers on nothing is left for the copy engine)
    const double workers = c->pool ? (double)c->pool->threads() : 0.0;
    const double left = 78.0 - (llkv::narrow_isa() >= 2 ? 11.0 : 6.4) * workers;
    share = left <= 0 ? 0 : (int)(100.0 * left / 78.0);
  }
  if (share <= 0) return false;
  if (share >= 100) return true;
  const uint64_t block = (first_row * 16) >> 23;
  return (block + 1) * (uint64_t)share / 100 > block * (uint64_t)share / 100;
}

static int32_t flush_upload(llkv_gpu_column* col) {
  if (!col->pend_bytes) return LLKV_OK;
  cudaStream_t cs = col->ctx->copy_streams[(size_t)col->stream_index];
  const uint64_t n = col->pend_bytes;
  col->pend_bytes = 0;
  CUDA_TRY(cudaMemcpyAsync(col->pend_dst, col->pend_src, n, cudaMemcpyHostToDevice, cs));
  return LLKV_OK;
}
// ... and waits for the host workers' jobs of this column (their destination is the values buffer too)
static int32_t drain_jobs(llkv_gpu_column* col) {
  llkv_gpu_ctx* c = col->ctx;
  if (!c->pool || (col->ticket.outstanding.load() == 0 && col->narrow_chunks.empty())) return LLKV_OK;
  const cudaError_t e = c->pool->wait(&col->ticket);
  col->ticket.cuda_error.store(0);
  if (e != cudaSuccess) return set_error(LLKV_ERR_IO, "CUDA error %s in a chunk upload worker", cudaGetErrorString(e));
  return LLKV_OK;
}

static int32_t column_grow(llkv_gpu_column* col, uint64_t need_rows) {
  if (need_rows + kPadRows <= col->cap_rows) return LLKV_OK;
  {  // pending copies target the buffer that is about to move
    int32_t frc = flush_upload(col);
    if (!frc) frc = drain_jobs(col);
    if (frc) return frc;
  }
  llkv_gpu_ctx* c = col->ctx;
  cudaStream_t s = c->copy_streams[(size_t)col->stream_index];
  uint64_t cap = col->cap_rows * 2;
  if (cap < need_rows + kPadRows) cap = need_rows + kPadRows;
  cap = (cap + kPadRows - 1) / kPadRows * kPadRows;
  void* nv = nullptr;
  CUDA_TRY(cudaMalloc(&nv, cap * col->elem_bytes));
  if (col->n_rows) CUDA_TRY(cudaMemcpyAsync(nv, col->values, col->n_rows * col->elem_bytes, cudaMemcpyDeviceToDevice, s));
  // the padding is read by bulk copies of the last tile: keep it defined
  CUDA_TRY(cudaMemsetAsync((char*)nv + col->n_rows * col->elem_bytes, 0, (cap - col->n_rows) * col->elem_bytes, s));
  unsigned int* nb = nullptr;
  if (col->validity) {
    const uint64_t words = cap / 32 + 4;
    CUDA_TRY(cudaMalloc((void**)&nb, words * 4));
    CUDA_TRY(cudaMemsetAsync(nb, 0, words * 4, s));
    CUDA_TRY(cudaMemcpyAsync(nb, col->validity, (col->n_rows + 31) / 32 * 4, cudaMemcpyDeviceToDevice, s));
  }
  CUDA_TRY(cudaStreamSynchronize(s));
  if (col->values) CUDA_TRY(cudaFree(col->values));
  if (col->validity) CUDA_TRY(cudaFree(col->validity));
  col->values = nv;
  col->validity = nb;
  col->cap_rows = cap;
  ++col->ctx->state_epoch;
  return LLKV_OK;
}

extern "C" int32_t llkv_gpu_column_reserve(llkv_gpu_column* col, uint64_t n_rows) {
  if (!col) return set_error(LLKV_ERR_INVALID_ARGUMENT, "column is NULL");
  CTX_LOCK(col->ctx);
  CUDA_TRY(cudaSetDevice(col->ctx->device));
  return column_grow(col, n_rows);
}

enum SrcKind { SRC_PAGEABLE = 0, SRC_PINNED = 1, SRC_DEVICE = 2 };
static SrcKind source_kind(const void* p) {
  cudaPointerAttributes attr;
  if (cudaPointerGetAttributes(&attr, p) == cudaSuccess) {
    if (attr.type == cudaMemoryTypeHost) return SRC_PINNED;
    if (attr.type == cudaMemoryTypeDevice || attr.type == cudaMemoryTypeManaged) return SRC_DEVICE;
    return SRC_PAGEABLE;
  }
  cudaGetLastError();
  return SRC_PAGEABLE;
}

// host -> device through the pinned staging ring (or directly when the source is already page-locked)
static int32_t upload(llkv_gpu_column* col, void* dst, const void* src, uint64_t bytes, SrcKind kind) {
  llkv_gpu_ctx* c = col->ctx;
  cudaStream_t cs = c->copy_streams[(size_t)col->stream_index];
  if (bytes == 0) return LLKV_OK;
  if (kind == SRC_DEVICE) {  // the chunk already sits in device memory (a decoder or generator running on the GPU): one D2D copy
    int32_t rc = flush_upload(col);
    if (rc) return rc;
    CUDA_TRY(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, cs));
    return LLKV_OK;
  }
  col->h2d_bytes += bytes;
  if (kind == SRC_PINNED) {
    // Page-locked source: DMA straight from the caller's buffer.  Chunks that continue the previous one on both sides
    // (a column appended chunk by chunk from one contiguous buffer) are coalesced into copies of up to 32 MiB: a 1 MiB
    // copy reaches 46 GB/s on this box's PCIe link, a large one 55 GB/s (tools/pcie.py).  The copy is issued by the next
    // append that does not continue it, by llkv_gpu_column_flush or by seal: the source must stay valid and unmodified
    // until one of the latter two returns (include/llkv_gpu.h).
    constexpr uint64_t kMaxCoalesced = 32ull << 20;
    if (col->pend_bytes && (const char*)col->pend_src + col->pend_bytes == (const char*)src &&
        (char*)col->pend_dst + col->pend_bytes == (char*)dst && col->pend_bytes + bytes <= kMaxCoalesced) {
      col->pend_bytes += bytes;
      return LLKV_OK;
    }
    int32_t rc = flush_upload(col);
    if (rc) return rc;
    col->pend_dst = dst;
    col->pend_src = src;
    col->pend_bytes = bytes;
    return LLKV_OK;
  }
  int32_t rc = flush_upload(col);
  if (rc) return rc;
  uint64_t done = 0;
  while (done < bytes) {
    const int slot = c->next_slot;
    c->next_slot = (c->next_slot + 1) % (int)c->copy_streams.size();
    const uint64_t n = bytes - done < c->slot_bytes ? bytes - done : c->slot_bytes;
    CUDA_TRY(cudaEventSynchronize(c->slot_events[(size_t)slot]));  // the slot's previous copy has drained
    unsigned char* stage = c->pinned + (uint64_t)slot * c->slot_bytes;
    memcpy(stage, (const char*)src + done, n);
    cudaStream_t s = c->copy_streams[(size_t)slot];
    CUDA_TRY(cudaMemcpyAsync((char*)dst + done, stage, n, cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaEventRecord(c->slot_events[(size_t)slot], s));
    if (s != cs) CUDA_TRY(cudaStreamWaitEvent(cs, c->slot_events[(size_t)slot], 0));  // the column's stream runs the follow-up kernels
    done += n;
  }
  return LLKV_OK;
}

static int32_t ensure_validity(llkv_gpu_column* col) {
  if (col->validity) return LLKV_OK;
  cudaStream_t s = col->ctx->copy_streams[(size_t)col->stream_index];
  const uint64_t words = col->cap_rows / 32 + 4;
  CUDA_TRY(cudaMalloc((void**)&col->validity, words * 4));
  CUDA_TRY(cudaMemsetAsync(col->validity, 0, words * 4, s));
  if (col->n_rows) {
    fill_bits_kernel<<<256, 256, 0, s>>>(col->validity, 0, col->n_rows);
    CUDA_TRY(cudaGetLastError());
  }
  return LLKV_OK;
}

static int32_t launch_stats(llkv_gpu_column* col, uint64_t first_row, uint64_t n) {
  if (n == 0) return LLKV_OK;
  cudaStream_t s = col->ctx->copy_streams[(size_t)col->stream_index];
  unsigned int blocks = (unsigned int)std::min<uint64_t>((n + 1023) / 1024, 1184);
  const char* base = (const char*)col->values + first_row * col->elem_bytes;
  if (col->load_kind == LK_D64) {  // narrow images of a Decimal128 column: the values are the sign-extended low halves
    stats_kernel<i64, true><<<blocks, 256, 0, s>>>((const i64*)base, n, col->dstats);
    CUDA_TRY(cudaGetLastError());
    return LLKV_OK;
  }
  if (col->load_kind == LK_D32) {
    stats_kernel<int, true><<<blocks, 256, 0, s>>>((const int*)base, n, col->dstats);
    CUDA_TRY(cudaGetLastError());
    return LLKV_OK;
  }
  switch (col->type) {
    case LLKV_PT_INT8: stats_kernel<signed char, true><<<blocks, 256, 0, s>>>((const signed char*)base, n, col->dstats); break;
    case LLKV_PT_INT16: stats_kernel<short, true><<<blocks, 256, 0, s>>>((const short*)base, n, col->dstats); break;
    case LLKV_PT_INT32: case LLKV_PT_DATE32: stats_kernel<int, true><<<blocks, 256, 0, s>>>((const int*)base, n, col->dstats); break;
    case LLKV_PT_INT64: case LLKV_PT_DATE64: stats_kernel<i64, true><<<blocks, 256, 0, s>>>((const i64*)base, n, col->dstats); break;
    case LLKV_PT_UINT8: case LLKV_PT_BOOLEAN: stats_kernel<unsigned char, false><<<blocks, 256, 0, s>>>((const unsigned char*)base, n, col->dstats); break;
    case LLKV_PT_UINT16: stats_kernel<unsigned short, false><<<blocks, 256, 0, s>>>((const unsigned short*)base, n, col->dstats); break;
    case LLKV_PT_UINT32: stats_kernel<unsigned int, false><<<blocks, 256, 0, s>>>((const unsigned int*)base, n, col->dstats); break;
    case LLKV_PT_UINT64: stats_kernel<u64, false><<<blocks, 256, 0, s>>>((const u64*)base, n, col->dstats); break;
    case LLKV_PT_DECIMAL128: stats_dec_kernel<<<blocks, 256, 0, s>>>((const ulonglong2*)base, n, col->dstats); break;
    default: return LLKV_OK;  // floats: no statistics needed; Utf8: gathered by the pack kernel (str_stats_kernel at seal when sparse)
  }
  CUDA_TRY(cudaGetLastError());
  return LLKV_OK;
}

// Zone map of the resident image, on the host (false: this column's layout has none: floats, strings, wide decimals).
static int32_t ensure_zones(llkv_gpu_column* col, bool* ok) {
  *ok = false;
  llkv_gpu_ctx* c = col->ctx;
  const u64 n = col->n_rows;
  if (n == 0) return LLKV_OK;
  const u64 n_zones = (n + kZoneRows - 1) / kZoneRows;
  if (col->zones_version == col->version && col->h_zones.size() == 2 * n_zones) {
    *ok = true;
    return LLKV_OK;
  }
  switch (col->type) {
    case LLKV_PT_INT8: case LLKV_PT_INT16: case LLKV_PT_INT32: case LLKV_PT_INT64: case LLKV_PT_DATE32: case LLKV_PT_DATE64:
    case LLKV_PT_UINT8: case LLKV_PT_UINT16: case LLKV_PT_UINT32: case LLKV_PT_UINT64: case LLKV_PT_BOOLEAN: break;
    case LLKV_PT_DECIMAL128: if (is_narrow_decimal(col)) break; return LLKV_OK;
    default: return LLKV_OK;
  }
  if (col->d_zones_cap < n_zones) {
    if (col->d_zones) CUDA_TRY(cudaFree(col->d_zones));
    col->d_zones = nullptr;
    col->d_zones_cap = 0;
    CUDA_TRY(cudaMalloc((void**)&col->d_zones, n_zones * 16));
    col->d_zones_cap = n_zones;
  }
  cudaStream_t s = c->stream;
  const unsigned blocks = (unsigned)std::min<u64>((n_zones + 7) / 8, 1184);
  const void* v = col->values;
  switch (col->load_kind) {
    case LK_I8: zone_minmax_kernel<signed char, true, 1><<<blocks, 256, 0, s>>>((const signed char*)v, n, col->d_zones); break;
    case LK_I16: zone_minmax_kernel<short, true, 1><<<blocks, 256, 0, s>>>((const short*)v, n, col->d_zones); break;
    case LK_I32: case LK_D32: zone_minmax_kernel<int, true, 1><<<blocks, 256, 0, s>>>((const int*)v, n, col->d_zones); break;
    case LK_I64: case LK_D64: zone_minmax_kernel<i64, true, 1><<<blocks, 256, 0, s>>>((const i64*)v, n, col->d_zones); break;
    case LK_U8: zone_minmax_kernel<unsigned char, false, 1><<<blocks, 256, 0, s>>>((const unsigned char*)v, n, col->d_zones); break;
    case LK_U16: zone_minmax_kernel<unsigned short, false, 1><<<blocks, 256, 0, s>>>((const unsigned short*)v, n, col->d_zones); break;
    case LK_U32: zone_minmax_kernel<unsigned int, false, 1><<<blocks, 256, 0, s>>>((const unsigned int*)v, n, col->d_zones); break;
    case LK_U64: zone_minmax_kernel<u64, false, 1><<<blocks, 256, 0, s>>>((const u64*)v, n, col->d_zones); break;
    default: return LLKV_OK;
  }
  CUDA_TRY(cudaGetLastError());
  col->h_zones.resize(2 * n_zones);
  CUDA_TRY(cudaMemcpyAsync(col->h_zones.data(), col->d_zones, n_zones * 16, cudaMemcpyDeviceToHost, s));
  CUDA_TRY(cudaStreamSynchronize(s));
  col->zones_version = col->version;
  *ok = true;
  return LLKV_OK;
}

// A Decimal128 column resident as i64 / i32 goes back to the Arrow layout (more chunks arrive that are not narrowed on the
// host, or a narrowed chunk did not fit).  Rows [0, rows) are widened on the device; the narrow buffer is parked.
static int32_t widen_decimal(llkv_gpu_column* col, uint64_t rows) {
  CUDA_TRY(cudaDeviceSynchronize());
  ulonglong2* wide = (ulonglong2*)col->landing;
  if (!wide || col->landing_cap < col->cap_rows) {
    if (wide) CUDA_TRY(cudaFree(wide));
    col->landing = nullptr;
    CUDA_TRY(cudaMalloc((void**)&wide, col->cap_rows * 16));
    CUDA_TRY(cudaMemset(wide, 0, col->cap_rows * 16));
    col->landing_cap = col->cap_rows;
  }
  if (rows) {
    if (col->load_kind == LK_D32) widen_dec32_kernel<<<1184, 256>>>((const int*)col->values, wide, rows);
    else widen_dec_kernel<<<1184, 256>>>((const u64*)col->values, wide, rows);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaDeviceSynchronize());
  }
  if (col->narrow && col->narrow != col->values) CUDA_TRY(cudaFree(col->narrow));
  col->narrow = col->values;  // parked for the next seal
  col->narrow_cap = col->cap_rows;
  col->narrow_width = col->elem_bytes;
  col->landing = nullptr;
  col->landing_cap = 0;
  col->values = wide;
  col->elem_bytes = 16;
  col->load_kind = LK_D128;
  ++col->ctx->state_epoch;
  return LLKV_OK;
}

// An empty Decimal128 column starts receiving host-narrowed chunks: `values` becomes a buffer of `width` bytes per row
// (the parked one when it fits), the Arrow-layout buffer is parked.
static int32_t begin_narrow_landing(llkv_gpu_column* col, uint32_t width, uint64_t need_rows) {
  uint64_t cap = std::max<uint64_t>(col->cap_rows, (need_rows + 2 * kPadRows - 1) / kPadRows * kPadRows);
  void* nv = col->narrow;
  if (!nv || col->narrow_width != width || col->narrow_cap < cap) {
    if (nv) CUDA_TRY(cudaFree(nv));
    col->narrow = nullptr;
    CUDA_TRY(cudaMalloc(&nv, cap * width));
    CUDA_TRY(cudaMemset(nv, 0, cap * width));
  } else {
    cap = col->narrow_cap;
  }
  if (col->landing && col->landing != col->values) CUDA_TRY(cudaFree(col->landing));
  col->landing = col->values;
  col->landing_cap = col->values ? col->cap_rows : 0;
  col->narrow = nullptr;
  col->narrow_cap = 0;
  col->values = nv;
  col->cap_rows = cap;
  col->elem_bytes = width;
  col->load_kind = width == 4 ? LK_D32 : LK_D64;
  ++col->ctx->state_epoch;
  if (col->validity) {  // sized by the old capacity
    CUDA_TRY(cudaFree(col->validity));
    col->validity = nullptr;
  }
  return LLKV_OK;
}

static cudaError_t launch_narrow_check(int kind, const void* wide, void* dst, uint64_t n_rows, unsigned int* d_flag, cudaStream_t s) {
  const unsigned blocks = (unsigned)std::min<uint64_t>((n_rows + 255) / 256, 592);
  if (kind == UP_NARROW_D128_I32) narrow_dec32_check_kernel<<<blocks, 256, 0, s>>>((const ulonglong2*)wide, (int*)dst, n_rows, d_flag);
  else narrow_dec64_check_kernel<<<blocks, 256, 0, s>>>((const ulonglong2*)wide, (u64*)dst, n_rows, d_flag);
  return cudaGetLastError();
}

static UploadPool* upload_pool(llkv_gpu_ctx* c) {
  if (c->upload_threads == 0) return nullptr;
  if (!c->pool) {
    int n = c->upload_threads;
    if (n < 0) {  // one thread streams ~5 GB/s of Arrow bytes; the caller's thread keeps a core for issuing the appends
      const unsigned hw = std::thread::hardware_concurrency();
      n = (int)std::min<unsigned>(32u, hw > 2 ? hw - 1 : 1u);
    }
    c->pool.reset(new UploadPool(c->device, n));
    c->pool->set_narrow_launcher(launch_narrow_check);
  }
  return c->pool.get();
}

// A Utf8 chunk (offsets n_rows + 1 in `off`, data bytes in `aux`) is checked on the host before anything is uploaded.
static int32_t utf8_chunk_shape(const int32_t* off, uint64_t n_rows, const void* aux, SrcKind src_kind, int64_t* first, int64_t* data_bytes,
                                bool* has_long) {
  if (src_kind == SRC_DEVICE) return set_error(LLKV_ERR_INVALID_ARGUMENT, "Utf8 chunks must come from host memory (the offsets are validated on the host)");
  *first = off[0];
  *data_bytes = (int64_t)off[n_rows] - *first;
  if (*first < 0 || *data_bytes < 0) return set_error(LLKV_ERR_INVALID_ARGUMENT, "Utf8 offsets are negative or not monotonic");
  *has_long = false;
  for (uint64_t i = 0; i < n_rows; ++i) {
    if (off[i + 1] < off[i]) return set_error(LLKV_ERR_INVALID_ARGUMENT, "Utf8 offsets are not monotonic at row %llu", (unsigned long long)i);
    *has_long = *has_long || off[i + 1] - off[i] > 7;
  }
  if (*data_bytes && !aux) return set_error(LLKV_ERR_INVALID_ARGUMENT, "Utf8 data buffer is NULL");
  return LLKV_OK;
}

// Host side of an append to a dictionary-coded column: the chunk's valid strings are interned, codes[i] is row i's code
// (0 under a NULL: the row's validity bit stays clear).
static int32_t intern_chunk(StrDict& d, const int32_t* off, const char* data, const uint8_t* validity, uint64_t n_rows, std::vector<u64>& codes) {
  codes.resize((size_t)n_rows);
  for (uint64_t i = 0; i < n_rows; ++i) {
    const bool valid = !validity || ((validity[i >> 3] >> (i & 7)) & 1);
    codes[(size_t)i] = valid ? d.code_of(d.intern(data + off[i], (size_t)(off[i + 1] - off[i]))) : 0;
  }
  if (d.strings.size() > kMaxDictEntries) return set_error(LLKV_ERR_INVALID_ARGUMENT, "more than %zu distinct strings in a dictionary-coded column", kMaxDictEntries);
  return LLKV_OK;
}

static int32_t widen_str8(llkv_gpu_column* col);
static int32_t enter_dict_mode(llkv_gpu_column* col);

// A chunk whose row ids do not continue the column densely (rows appended after deletes, updates of existing rows, columns
// that skip rows because the value is NULL): positions are row id - origin, rows nobody wrote are invalid bits.  Utf8 chunks
// are packed into 8-byte keys by scatter_utf8_kernel, or interned on the host and scattered as codes once the column is
// dictionary-coded.
static int32_t append_sparse(llkv_gpu_column* col, const void* values, uint64_t n_rows, const uint8_t* validity, const uint64_t* row_ids,
                             const void* aux) {
  llkv_gpu_ctx* c = col->ctx;
  uint64_t lo = ~0ull, hi = 0;
  for (uint64_t i = 0; i < n_rows; ++i) {
    lo = std::min(lo, row_ids[i]);
    hi = std::max(hi, row_ids[i]);
  }
  if (lo < col->row_id_origin)
    return set_error(LLKV_ERR_INVALID_ARGUMENT, "row id %llu lies below the column's first row id %llu (name the table's first row id in row_id_base with the first chunk)",
                     (unsigned long long)lo, (unsigned long long)col->row_id_origin);
  const uint64_t span = hi - col->row_id_origin + 1;
  if (span > (1ull << 40)) return set_error(LLKV_ERR_INVALID_ARGUMENT, "row ids span %llu positions: too sparse for a resident image", (unsigned long long)span);
  const bool utf8 = col->type == LLKV_PT_UTF8;
  const int32_t* off = (const int32_t*)values;
  int64_t first = 0, data_bytes = 0;
  bool has_long = false;
  int32_t rc;
  if (utf8 && (rc = utf8_chunk_shape(off, n_rows, aux, source_kind(values), &first, &data_bytes, &has_long))) return rc;
  if ((rc = flush_upload(col)) || (rc = drain_jobs(col))) return rc;
  if (is_narrow_decimal(col) && (rc = widen_decimal(col, col->n_rows))) return rc;
  if (col->load_kind == LK_STR8 && (rc = widen_str8(col))) return rc;  // sealed as one byte per string: back to packed keys
  if (has_long && !col->dict && (rc = enter_dict_mode(col))) return rc;
  std::vector<u64> codes;
  if (utf8 && col->dict && (rc = intern_chunk(*col->dict, off, (const char*)aux, validity, n_rows, codes))) return rc;
  const bool packed_utf8 = utf8 && !col->dict;
  col->sealed = false;
  const uint64_t new_rows = std::max<uint64_t>(col->n_rows, span);
  if ((rc = column_grow(col, new_rows))) return rc;
  if ((rc = ensure_validity(col))) return rc;  // rows so far are valid, everything behind them is not (yet)
  cudaStream_t s = c->copy_streams[(size_t)col->stream_index];
  void* d_vals = nullptr;  // values, codes, or a packed column's offsets
  unsigned char* d_data = nullptr;
  u64* d_ids = nullptr;
  unsigned char* d_bits = nullptr;
  const uint64_t val_bytes = packed_utf8 ? (n_rows + 1) * 4 : n_rows * col->elem_bytes;
  CUDA_TRY(cudaMalloc(&d_vals, val_bytes));
  CUDA_TRY(cudaMalloc((void**)&d_ids, n_rows * 8));
  if (utf8 && col->dict) rc = upload(col, d_vals, codes.data(), val_bytes, SRC_PAGEABLE);
  else rc = upload(col, d_vals, values, val_bytes, source_kind(values));
  if (rc) return rc;
  if (packed_utf8 && data_bytes > 0) {  // the chunk's slice of the data buffer
    CUDA_TRY(cudaMalloc((void**)&d_data, (size_t)data_bytes));
    if ((rc = upload(col, d_data, (const char*)aux + first, (uint64_t)data_bytes, source_kind(aux)))) return rc;
  }
  if ((rc = upload(col, d_ids, row_ids, n_rows * 8, source_kind(row_ids)))) return rc;
  if (validity) {
    CUDA_TRY(cudaMalloc((void**)&d_bits, (n_rows + 7) / 8));
    if ((rc = upload(col, d_bits, validity, (n_rows + 7) / 8, source_kind(validity)))) return rc;
  }
  if ((rc = flush_upload(col))) return rc;
  const unsigned blocks = (unsigned)std::min<uint64_t>((n_rows + 255) / 256, 1184);
  const u64 origin = col->row_id_origin;
  if (packed_utf8) {
    scatter_utf8_kernel<<<blocks, 256, 0, s>>>((u64*)col->values, col->validity, (const int*)d_vals, d_data, (int)first, d_ids, d_bits, n_rows, origin,
                                               col->dstats);
  } else {
    switch (col->elem_bytes) {
      case 1: scatter_rows_kernel<unsigned char><<<blocks, 256, 0, s>>>((unsigned char*)col->values, col->validity, (const unsigned char*)d_vals, d_ids, d_bits, n_rows, origin); break;
      case 2: scatter_rows_kernel<unsigned short><<<blocks, 256, 0, s>>>((unsigned short*)col->values, col->validity, (const unsigned short*)d_vals, d_ids, d_bits, n_rows, origin); break;
      case 4: scatter_rows_kernel<unsigned int><<<blocks, 256, 0, s>>>((unsigned int*)col->values, col->validity, (const unsigned int*)d_vals, d_ids, d_bits, n_rows, origin); break;
      case 8: scatter_rows_kernel<u64><<<blocks, 256, 0, s>>>((u64*)col->values, col->validity, (const u64*)d_vals, d_ids, d_bits, n_rows, origin); break;
      default: scatter_rows_kernel<ulonglong2><<<blocks, 256, 0, s>>>((ulonglong2*)col->values, col->validity, (const ulonglong2*)d_vals, d_ids, d_bits, n_rows, origin); break;
    }
  }
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaFreeAsync(d_vals, s));
  CUDA_TRY(cudaFreeAsync(d_ids, s));
  if (d_data) CUDA_TRY(cudaFreeAsync(d_data, s));
  if (d_bits) CUDA_TRY(cudaFreeAsync(d_bits, s));
  CUDA_TRY(cudaStreamSynchronize(s));  // (the sources were pageable staging copies or page-locked: either way they are free now)
  if (utf8) col->hstats.data_bytes += (u64)data_bytes;
  col->n_rows = new_rows;
  col->sparse = true;
  ++col->version;
  ++c->state_epoch;
  col->scans_unchanged = 0;
  return LLKV_OK;
}

static int32_t widen_str8(llkv_gpu_column* col) {
  u64* wide = nullptr;
  CUDA_TRY(cudaDeviceSynchronize());
  CUDA_TRY(cudaMalloc((void**)&wide, col->cap_rows * 8));
  CUDA_TRY(cudaMemset(wide, 0, col->cap_rows * 8));
  widen_str_kernel<<<1184, 256>>>((const unsigned char*)col->values, wide, col->n_rows);
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaDeviceSynchronize());
  CUDA_TRY(cudaFree(col->values));
  col->values = wide;
  col->elem_bytes = 8;
  col->load_kind = LK_U64;
  return LLKV_OK;
}

// A Utf8 column meets its first string longer than 7 bytes: the rows it already holds (packed keys, which carry their bytes)
// are read back once, interned, and rewritten as dictionary codes.  Only positions whose validity bit is set are interned:
// a gap, a deleted row or a NULL holds no string (its code is 0 under a clear bit).
static int32_t enter_dict_mode(llkv_gpu_column* col) {
  llkv_gpu_ctx* c = col->ctx;
  int32_t rc = flush_upload(col);
  if (rc) return rc;
  cudaStream_t s = c->copy_streams[(size_t)col->stream_index];
  CUDA_TRY(cudaStreamSynchronize(s));
  CUDA_TRY(cudaStreamSynchronize(c->stream));
  col->dict.reset(new StrDict());
  StrDict& d = *col->dict;
  if (col->n_rows) {
    std::vector<u64> keys((size_t)col->n_rows);
    CUDA_TRY(cudaMemcpy(keys.data(), col->values, col->n_rows * 8, cudaMemcpyDeviceToHost));
    std::vector<unsigned int> bits;
    if (col->validity) {
      bits.resize((size_t)((col->n_rows + 31) / 32));
      CUDA_TRY(cudaMemcpy(bits.data(), col->validity, bits.size() * 4, cudaMemcpyDeviceToHost));
    }
    std::unordered_map<u64, uint32_t> seen;
    for (size_t i = 0; i < keys.size(); ++i) {
      u64& k = keys[i];
      if (!bits.empty() && !((bits[i >> 5] >> (i & 31)) & 1u)) {
        k = 0;
        continue;
      }
      auto it = seen.find(k);
      if (it == seen.end()) {
        char b[8];
        const size_t len = (size_t)(k & 0xff) > 7 ? 0 : (size_t)(k & 0xff);
        for (size_t j = 0; j < len; ++j) b[j] = (char)(k >> (56 - 8 * j));
        it = seen.emplace(k, d.intern(b, len)).first;
      }
      k = it->second;
    }
    CUDA_TRY(cudaMemcpy(col->values, keys.data(), col->n_rows * 8, cudaMemcpyHostToDevice));
    col->h2d_bytes += col->n_rows * 8;
  }
  return LLKV_OK;
}

// seal of a dictionary-coded column: entries in byte order (str: Ord), resident codes -> ranks
static int32_t dict_seal(llkv_gpu_column* col) {
  llkv_gpu_ctx* c = col->ctx;
  StrDict& d = *col->dict;
  const uint32_t D = (uint32_t)d.strings.size();
  if (D == d.sealed) return LLKV_OK;
  std::vector<uint32_t> order(D);
  for (uint32_t i = 0; i < D; ++i) order[i] = i;
  std::sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return d.strings[a] < d.strings[b]; });  // (char_traits<char>::compare is memcmp)
  std::vector<uint32_t> new_rank(D), remap(D);
  for (uint32_t r = 0; r < D; ++r) new_rank[order[r]] = r;
  for (uint32_t code = 0; code < D; ++code) remap[code] = code < d.sealed ? new_rank[d.id_of_rank[code]] : new_rank[code];
  unsigned int* d_remap = nullptr;
  cudaStream_t s = c->copy_streams[(size_t)col->stream_index];
  CUDA_TRY(cudaMalloc((void**)&d_remap, (size_t)D * 4));
  CUDA_TRY(cudaMemcpyAsync(d_remap, remap.data(), (size_t)D * 4, cudaMemcpyHostToDevice, s));
  if (col->n_rows) {
    remap_codes_kernel<<<1184, 256, 0, s>>>((u64*)col->values, col->n_rows, d_remap);
    CUDA_TRY(cudaGetLastError());
  }
  CUDA_TRY(cudaStreamSynchronize(s));
  CUDA_TRY(cudaFree(d_remap));
  d.rank_of_id = new_rank;
  d.id_of_rank = order;
  d.sorted.resize(D);
  for (uint32_t r = 0; r < D; ++r) d.sorted[r] = d.strings[order[r]];
  d.sealed = D;
  ++d.epoch;
  return LLKV_OK;
}

static int32_t append_chunk_impl(llkv_gpu_column* col, const void* values, uint64_t n_rows, const uint8_t* validity, const uint64_t* row_ids,
                                 uint64_t row_id_base, const void* aux) {
  llkv_gpu_ctx* c = col->ctx;
  // Dense run (the usual case: rows appended in row-id order to a table nobody deleted from) or arbitrary row ids?
  uint64_t first_id = row_ids && n_rows ? row_ids[0] : row_id_base;
  bool dense_run = true;
  if (row_ids)
    for (uint64_t i = 1; i < n_rows && dense_run; ++i) dense_run = row_ids[i] == first_id + i;
  if (!col->has_origin) {
    // position 0 = the chunk's first row id, except for a first chunk of scattered ids: then row_id_base names it
    col->row_id_origin = dense_run ? first_id : std::min<uint64_t>(row_id_base, first_id);
    col->has_origin = true;
  }
  if (!dense_run || first_id != col->row_id_origin + col->n_rows) {
    if (!row_ids)
      return set_error(LLKV_ERR_INVALID_ARGUMENT, "chunk row ids start at %llu but the column continues at %llu: pass the row ids of a chunk that does not continue the column",
                       (unsigned long long)first_id, (unsigned long long)(col->row_id_origin + col->n_rows));
    if (n_rows == 0) return LLKV_OK;
    return append_sparse(col, values, n_rows, validity, row_ids, aux);
  }
  if (n_rows == 0) return LLKV_OK;
  col->sealed = false;
  const SrcKind src_kind = source_kind(values);
  const bool pinned_src = src_kind == SRC_PINNED;
  int32_t rc0;
  if (col->load_kind == LK_STR8 && (rc0 = widen_str8(col))) return rc0;  // sealed as one byte per string: back to packed keys before more chunks arrive
  // Decimal128: chunks from page-locked memory are narrowed by the host workers while the column's values keep fitting
  // (upload.h); everything else lands in the Arrow layout and is narrowed on the device at seal.
  int host_kind = -2;
  int32_t rc;
  if (col->type == LLKV_PT_DECIMAL128) {
    UploadPool* pool = (pinned_src && !c->keep_wide_decimals && col->host_kind != -2) ? upload_pool(c) : nullptr;
    if (pool && is_narrow_decimal(col)) {
      host_kind = col->load_kind == LK_D32 ? UP_NARROW_D128_I32 : UP_NARROW_D128_I64;
      if (col->host_kind == UP_NARROW_D128_I64 && host_kind == UP_NARROW_D128_I32) host_kind = -2;  // i32 failed before
    } else if (pool && col->n_rows == 0) {
      host_kind = col->host_kind;
      if (host_kind == -1) {  // look at the first chunk
        const int64_t* v = static_cast<const int64_t*>(values);
        bool fits32 = true, fits64 = true;
        for (uint64_t i = 0; i < n_rows && fits64; ++i) {
          const int64_t lo = v[2 * i], hi = v[2 * i + 1];
          fits64 = hi == (lo >> 63);
          fits32 = fits32 && lo == (int64_t)(int32_t)lo;
        }
        host_kind = !fits64 ? -2 : (fits32 && !c->no_d32 ? UP_NARROW_D128_I32 : UP_NARROW_D128_I64);
        col->host_kind = host_kind;
      }
      if (host_kind >= 0 && (rc = begin_narrow_landing(col, host_kind == UP_NARROW_D128_I32 ? 4u : 8u, n_rows))) return rc;
    }
    if (host_kind < 0 && is_narrow_decimal(col)) {
      if ((rc = flush_upload(col)) || (rc = drain_jobs(col))) return rc;
      if ((rc = widen_decimal(col, col->n_rows))) return rc;
    }
  }
  if ((rc = column_grow(col, col->n_rows + n_rows))) return rc;
  cudaStream_t s = c->copy_streams[(size_t)col->stream_index];
  if (col->type == LLKV_PT_UTF8) {
    // the chunk's slice of the data buffer is uploaded and the offsets are rebased on the device (a column appended in many
    // chunks from one data buffer uploads every byte once)
    const int32_t* off = (const int32_t*)values;
    int64_t first, data_bytes;
    bool has_long;
    if ((rc = utf8_chunk_shape(off, n_rows, aux, src_kind, &first, &data_bytes, &has_long))) return rc;
    if (has_long && !col->dict && (rc = enter_dict_mode(col))) return rc;
    if (col->dict) {
      // the host interns every string; 8 bytes of code per row cross the link, the bytes of the strings never do
      std::vector<u64> codes;
      if ((rc = intern_chunk(*col->dict, off, (const char*)aux, validity, n_rows, codes))) return rc;
      if ((rc = upload(col, (u64*)col->values + col->n_rows, codes.data(), n_rows * 8, SRC_PAGEABLE))) return rc;
      if ((rc = flush_upload(col))) return rc;
      CUDA_TRY(cudaStreamSynchronize(s));  // `codes` goes away with this scope
      col->hstats.data_bytes += (u64)data_bytes;
    } else {
    int* d_off = nullptr;
    unsigned char* d_data = nullptr;
    CUDA_TRY(cudaMalloc((void**)&d_off, (n_rows + 1) * 4));
    CUDA_TRY(cudaMalloc((void**)&d_data, (size_t)(data_bytes > 0 ? data_bytes : 1)));
    if ((rc = upload(col, d_off, off, (n_rows + 1) * 4, src_kind))) return rc;
    if (data_bytes > 0 && (rc = upload(col, d_data, (const char*)aux + first, (uint64_t)data_bytes, source_kind(aux)))) return rc;
    const unsigned int blocks = (unsigned int)std::min<uint64_t>((n_rows + 255) / 256, 1184);
    if ((rc = flush_upload(col))) return rc;
    pack_utf8_kernel<<<blocks, 256, 0, s>>>(d_off, d_data, (int)first, n_rows, (u64*)col->values + col->n_rows, col->dstats);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaFreeAsync(d_off, s));  // stream-ordered: released once the pack kernel has read them
    CUDA_TRY(cudaFreeAsync(d_data, s));
    col->hstats.data_bytes += (u64)data_bytes;
    }
  } else if (host_kind >= 0) {
    col->narrow_chunks.push_back(NarrowChunk{values, col->n_rows, n_rows});
    if (route_to_dma(col, col->n_rows)) {
      if (!col->d_fit) {
        CUDA_TRY(cudaMalloc((void**)&col->d_fit, 4));
        CUDA_TRY(cudaMemset(col->d_fit, 0, 4));
      }
      col->dma_used = true;
      col->h2d_bytes += n_rows * 16;
      c->pool->submit_dma(&col->ticket, values, (char*)col->values + col->n_rows * col->elem_bytes, n_rows, host_kind, col->d_fit);
    } else {
      col->h2d_bytes += n_rows * col->elem_bytes;
      c->pool->submit(&col->ticket, values, (char*)col->values + col->n_rows * col->elem_bytes, n_rows, host_kind);
    }
  } else {
    if ((rc = upload(col, (char*)col->values + col->n_rows * col->elem_bytes, values, n_rows * col->elem_bytes, src_kind))) return rc;
  }
  if (validity) {
    if ((rc = ensure_validity(col))) return rc;
    unsigned char* d_bits = nullptr;
    const uint64_t nb = (n_rows + 7) / 8;
    CUDA_TRY(cudaMalloc((void**)&d_bits, nb));
    if ((rc = upload(col, d_bits, validity, nb, source_kind(validity)))) return rc;
    const unsigned int blocks = (unsigned int)std::min<uint64_t>((n_rows / 32 + 256) / 256, 1184);
    if ((rc = flush_upload(col))) return rc;
    or_bits_kernel<<<blocks, 256, 0, s>>>(col->validity, col->n_rows, d_bits, n_rows);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaFreeAsync(d_bits, s));
  } else if (col->validity) {
    fill_bits_kernel<<<256, 256, 0, s>>>(col->validity, col->n_rows, col->n_rows + n_rows);
    CUDA_TRY(cudaGetLastError());
  }
  col->n_rows += n_rows;
  ++col->version;
  ++c->state_epoch;
  col->scans_unchanged = 0;
  return LLKV_OK;
}

extern "C" int32_t llkv_gpu_column_append_chunk(llkv_gpu_column* col, uint64_t chunk_pk, const void* values, uint64_t n_rows,
                                                 const uint8_t* validity, const uint64_t* row_ids, uint64_t row_id_base,
                                                 const void* aux) {
  (void)chunk_pk;
  if (!col) return set_error(LLKV_ERR_INVALID_ARGUMENT, "column is NULL");
  if (n_rows && !values) return set_error(LLKV_ERR_INVALID_ARGUMENT, "values is NULL");
  llkv_gpu_ctx* c = col->ctx;
  CTX_LOCK(c);
  CUDA_TRY(cudaSetDevice(c->device));
  const int32_t rc = append_chunk_impl(col, values, n_rows, validity, row_ids, row_id_base, aux);
  if (rc) {  // what earlier chunks left pending still belongs to the column; nothing of the failed chunk stays referenced
    const std::string msg = g_last_error;
    flush_upload(col);
    g_last_error = msg;
  }
  return rc;
}

extern "C" int32_t llkv_gpu_column_append_blob(llkv_gpu_column* col, uint64_t chunk_pk, const void* blob, uint64_t blob_len,
                                                const uint64_t* row_ids, uint64_t row_id_base) {
  if (!col || !blob) return set_error(LLKV_ERR_INVALID_ARGUMENT, "NULL argument");
  // "ARR0" | layout u8 | PrimType u8 | precision u8 | scale u8 | len u64 | extra_a u32 | extra_b u32 | payload
  // (llkv-column-map/src/serialization.rs:41-53,264-307)
  const unsigned char* b = (const unsigned char*)blob;
  if (blob_len < 24) return set_error(LLKV_ERR_IO, "chunk blob too short for its header");
  if (memcmp(b, "ARR0", 4) != 0) return set_error(LLKV_ERR_IO, "chunk blob has a bad magic");
  if (b[4] != 0) return set_error(LLKV_ERR_INVALID_ARGUMENT, "only the Primitive chunk layout crosses this boundary (layout %d)", b[4]);
  if ((int32_t)b[5] != col->type) return set_error(LLKV_ERR_INVALID_ARGUMENT, "chunk PrimType %d does not match the column type %d", b[5], col->type);
  if (col->type == LLKV_PT_DECIMAL128 && (b[6] != col->precision || (int8_t)b[7] != col->scale))
    return set_error(LLKV_ERR_INVALID_ARGUMENT, "chunk Decimal128(%d,%d) does not match the column", b[6], (int8_t)b[7]);
  uint64_t len;
  uint32_t values_len;
  memcpy(&len, b + 8, 8);
  memcpy(&values_len, b + 16, 4);
  const uint64_t w = (uint64_t)prim_type_width(col->type);
  if (values_len != len * w || 24 + (uint64_t)values_len > blob_len) return set_error(LLKV_ERR_IO, "chunk blob payload length mismatch");
  return llkv_gpu_column_append_chunk(col, chunk_pk, b + 24, len, nullptr, row_ids, row_id_base, nullptr);
}

// A host-narrowed chunk did not fit: the column goes back to the Arrow layout and the chunks appended since the last seal
// are copied again, wide, straight from their (page-locked, still valid: llkv_gpu.h) sources.
static int32_t recover_wide(llkv_gpu_column* col) {
  llkv_gpu_ctx* c = col->ctx;
  const uint64_t keep = col->narrow_chunks.empty() ? col->n_rows : col->narrow_chunks.front().first_row;
  col->host_kind = col->load_kind == LK_D32 ? (int)UP_NARROW_D128_I64 : -2;  // next time: the wider form, or none
  int32_t rc = widen_decimal(col, keep);
  if (rc) return rc;
  cudaStream_t s = c->copy_streams[(size_t)col->stream_index];
  for (const NarrowChunk& ch : col->narrow_chunks) {
    CUDA_TRY(cudaMemcpyAsync((char*)col->values + ch.first_row * 16, ch.src, ch.n_rows * 16, cudaMemcpyHostToDevice, s));
    col->h2d_bytes += ch.n_rows * 16;
  }
  CUDA_TRY(cudaStreamSynchronize(s));
  col->ticket.failed.store(0);
  return LLKV_OK;
}

// Issues and waits for everything the column's appends left in flight.  After it returns the sources may be reused.
static int32_t column_flush(llkv_gpu_column* col) {
  llkv_gpu_ctx* c = col->ctx;
  int32_t rc = flush_upload(col);
  if (rc) return rc;
  if ((rc = drain_jobs(col))) return rc;
  if (col->dma_used) {  // the DMA share's fit check ran on the device
    unsigned int bad = 0;
    cudaStream_t cs = c->copy_streams[(size_t)col->stream_index];
    CUDA_TRY(cudaMemcpyAsync(&bad, col->d_fit, 4, cudaMemcpyDeviceToHost, cs));
    CUDA_TRY(cudaMemsetAsync(col->d_fit, 0, 4, cs));
    CUDA_TRY(cudaStreamSynchronize(cs));
    col->dma_used = false;
    if (bad) col->ticket.failed.store(1);
  }
  if (col->ticket.failed.load() && (rc = recover_wide(col))) return rc;
  col->narrow_chunks.clear();
  for (cudaStream_t s : c->copy_streams) CUDA_TRY(cudaStreamSynchronize(s));
  return LLKV_OK;
}

extern "C" int32_t llkv_gpu_column_flush(llkv_gpu_column* col) {
  if (!col) return set_error(LLKV_ERR_INVALID_ARGUMENT, "column is NULL");
  CTX_LOCK(col->ctx);
  CUDA_TRY(cudaSetDevice(col->ctx->device));
  return column_flush(col);
}

extern "C" int32_t llkv_gpu_column_seal(llkv_gpu_column* col) {
  if (!col) return set_error(LLKV_ERR_INVALID_ARGUMENT, "column is NULL");
  llkv_gpu_ctx* c = col->ctx;
  CTX_LOCK(c);
  CUDA_TRY(cudaSetDevice(c->device));
  {
    int32_t frc = column_flush(col);
    if (frc) return frc;
  }
  for (void* p : col->deferred_free) cudaFree(p);
  col->deferred_free.clear();
  if (col->sparse && col->load_kind != LK_STR8) {  // scattered writes: the statistics start over (values under invalid bits are zeros)
    DevStats init;
    memset(&init, 0, sizeof(init));
    init.min_enc = ~0ull;
    init.min_strlen = 0xffffffffu;
    cudaStream_t ss = c->copy_streams[(size_t)col->stream_index];
    CUDA_TRY(cudaMemcpyAsync(col->dstats, &init, sizeof(init), cudaMemcpyHostToDevice, ss));
    col->stats_rows = 0;
    if (col->type == LLKV_PT_UTF8 && !col->dict && col->n_rows) {  // packed keys: lengths and bytes of the rows that exist
      const unsigned blocks = (unsigned)std::min<uint64_t>((col->n_rows + 1023) / 1024, 1184);
      str_stats_kernel<<<blocks, 256, 0, ss>>>((const u64*)col->values, col->validity, col->n_rows, col->dstats);
      CUDA_TRY(cudaGetLastError());
    }
    CUDA_TRY(cudaStreamSynchronize(ss));
  }
  if (col->stats_rows < col->n_rows && col->load_kind != LK_STR8) {  // min / max / fits-i64 over the rows appended since the last seal
    int32_t rc = launch_stats(col, col->stats_rows, col->n_rows - col->stats_rows);
    if (rc) return rc;
    CUDA_TRY(cudaStreamSynchronize(c->copy_streams[(size_t)col->stream_index]));
    col->stats_rows = col->n_rows;
  }
  const u64 data_bytes = col->hstats.data_bytes;
  CUDA_TRY(cudaMemcpy(&col->hstats, col->dstats, sizeof(DevStats), cudaMemcpyDeviceToHost));
  col->hstats.data_bytes = data_bytes;
  if (col->type == LLKV_PT_UTF8 && col->dict) {
    int32_t rc = dict_seal(col);
    if (rc) return rc;
  } else if (col->type == LLKV_PT_UTF8) {
    if (col->hstats.bad_string & 1u) return set_error(LLKV_ERR_INTERNAL, "string longer than 7 bytes in a packed short-string column");
    // every string exactly one byte long: keep one byte per row
    if (col->load_kind == LK_U64 && col->n_rows && col->hstats.max_strlen == 1 && col->hstats.min_strlen == 1) {
      unsigned char* nv = nullptr;
      CUDA_TRY(cudaMalloc((void**)&nv, col->cap_rows));
      CUDA_TRY(cudaMemset(nv, 0, col->cap_rows));
      narrow_str_kernel<<<1184, 256>>>((const u64*)col->values, nv, col->n_rows);
      CUDA_TRY(cudaGetLastError());
      CUDA_TRY(cudaDeviceSynchronize());
      CUDA_TRY(cudaFree(col->values));
      col->values = nv;
      col->elem_bytes = 1;
      col->load_kind = LK_STR8;
    }
  }
  // Decimal128 whose every value is a sign-extended i64 (i32): keep 8 (4) bytes per row resident — half (a quarter of) the
  // HBM traffic and shared-memory tile of every scan; the Arrow layout is restored if chunks arrive that do not fit
  if (col->type == LLKV_PT_DECIMAL128 && col->load_kind == LK_D128 && col->n_rows && col->hstats.not_i64 == 0 && !c->keep_wide_decimals) {
    const i64 mn = (i64)(col->hstats.min_enc ^ 0x8000000000000000ull), mx = (i64)(col->hstats.max_enc ^ 0x8000000000000000ull);
    const bool fits32 = mn >= (i64)INT32_MIN && mx <= (i64)INT32_MAX && !c->no_d32;
    const uint32_t width = fits32 ? 4u : 8u;
    void* nv = col->narrow;
    if (!nv || col->narrow_cap < col->cap_rows || col->narrow_width != width) {
      if (nv) CUDA_TRY(cudaFree(nv));
      col->narrow = nullptr;
      CUDA_TRY(cudaMalloc(&nv, col->cap_rows * width));
      CUDA_TRY(cudaMemset(nv, 0, col->cap_rows * width));
    }
    cudaStream_t ns = c->copy_streams[(size_t)col->stream_index];
    if (fits32) narrow_dec32_kernel<<<1184, 256, 0, ns>>>((const ulonglong2*)col->values, (int*)nv, col->n_rows);
    else narrow_dec_kernel<<<1184, 256, 0, ns>>>((const ulonglong2*)col->values, (u64*)nv, col->n_rows);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaStreamSynchronize(ns));
    if (col->reupload_hint) {  // the Arrow-layout buffer stays for the next batch
      col->landing = col->values;
      col->landing_cap = col->cap_rows;
    } else {
      CUDA_TRY(cudaFree(col->values));
      col->landing = nullptr;
      col->landing_cap = 0;
    }
    col->narrow = nullptr;
    col->narrow_cap = 0;
    col->values = nv;
    col->elem_bytes = width;
    col->load_kind = fits32 ? LK_D32 : LK_D64;
  }
  col->sealed = true;
  ++c->state_epoch;
  return LLKV_OK;
}

extern "C" int32_t llkv_gpu_column_rows(const llkv_gpu_column* col, uint64_t* out_rows) {
  if (!col || !out_rows) return set_error(LLKV_ERR_INVALID_ARGUMENT, "NULL argument");
  *out_rows = col->n_rows;
  return LLKV_OK;
}

extern "C" int32_t llkv_gpu_column_delete_rows(llkv_gpu_column* col, const uint64_t* row_ids, uint64_t n) {
  if (!col || (n && !row_ids)) return set_error(LLKV_ERR_INVALID_ARGUMENT, "NULL argument");
  llkv_gpu_ctx* c = col->ctx;
  CTX_LOCK(c);
  CUDA_TRY(cudaSetDevice(c->device));
  if (n == 0 || col->n_rows == 0) return LLKV_OK;
  int32_t rc;
  if ((rc = column_flush(col))) return rc;
  if ((rc = ensure_validity(col))) return rc;
  cudaStream_t s = c->copy_streams[(size_t)col->stream_index];
  u64* d_ids = nullptr;
  CUDA_TRY(cudaMalloc((void**)&d_ids, n * 8));
  if ((rc = upload(col, d_ids, row_ids, n * 8, source_kind(row_ids))) || (rc = flush_upload(col))) return rc;
  clear_rows_kernel<<<(unsigned)std::min<uint64_t>((n + 255) / 256, 1184), 256, 0, s>>>(col->validity, d_ids, n, col->row_id_origin, col->n_rows);
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaFreeAsync(d_ids, s));
  CUDA_TRY(cudaStreamSynchronize(s));
  col->sparse = true;
  col->sealed = false;
  ++col->version;
  ++c->state_epoch;
  col->scans_unchanged = 0;
  return LLKV_OK;
}

extern "C" int32_t llkv_gpu_column_gather(llkv_gpu_column* col, const uint64_t* row_ids, uint64_t n, void* out_values, uint64_t out_bytes,
                                           uint8_t* out_valid) {
  if (!col || (n && (!row_ids || !out_values || !out_valid))) return set_error(LLKV_ERR_INVALID_ARGUMENT, "NULL argument");
  if (col->type == LLKV_PT_UTF8) return set_error(LLKV_ERR_INVALID_ARGUMENT, "llkv_gpu_column_gather does not support Utf8 columns");
  llkv_gpu_ctx* c = col->ctx;
  CTX_LOCK(c);
  CUDA_TRY(cudaSetDevice(c->device));
  if (!col->sealed) {
    int32_t rc = llkv_gpu_column_seal(col);
    if (rc) return rc;
  }
  const uint64_t width = (uint64_t)prim_type_width(col->type);
  if (out_bytes < n * width) return set_error(LLKV_ERR_INVALID_ARGUMENT, "output buffer too small");
  if (n == 0) return LLKV_OK;
  cudaStream_t s = c->stream;
  u64* d_ids = nullptr;
  void* d_out = nullptr;
  ulonglong2* d_wide = nullptr;
  unsigned char* d_valid = nullptr;
  cudaError_t e = cudaMalloc((void**)&d_ids, n * 8);
  if (e == cudaSuccess) e = cudaMalloc(&d_out, n * col->elem_bytes);
  if (e == cudaSuccess) e = cudaMalloc((void**)&d_valid, n);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_ids, row_ids, n * 8, cudaMemcpyHostToDevice, s);
  const unsigned blocks = (unsigned)std::min<uint64_t>((n + 255) / 256, 1184);
  if (e == cudaSuccess) {
    const u64 origin = col->row_id_origin, rows = col->n_rows;
    switch (col->elem_bytes) {
      case 1: gather_rows_kernel<unsigned char><<<blocks, 256, 0, s>>>((const unsigned char*)col->values, col->validity, d_ids, n, origin, rows, (unsigned char*)d_out, d_valid); break;
      case 2: gather_rows_kernel<unsigned short><<<blocks, 256, 0, s>>>((const unsigned short*)col->values, col->validity, d_ids, n, origin, rows, (unsigned short*)d_out, d_valid); break;
      case 4: gather_rows_kernel<unsigned int><<<blocks, 256, 0, s>>>((const unsigned int*)col->values, col->validity, d_ids, n, origin, rows, (unsigned int*)d_out, d_valid); break;
      case 8: gather_rows_kernel<u64><<<blocks, 256, 0, s>>>((const u64*)col->values, col->validity, d_ids, n, origin, rows, (u64*)d_out, d_valid); break;
      default: gather_rows_kernel<ulonglong2><<<blocks, 256, 0, s>>>((const ulonglong2*)col->values, col->validity, d_ids, n, origin, rows, (ulonglong2*)d_out, d_valid); break;
    }
    e = cudaGetLastError();
  }
  const void* result = d_out;
  if (e == cudaSuccess && is_narrow_decimal(col)) {  // back to the Arrow layout
    e = cudaMalloc((void**)&d_wide, n * 16);
    if (e == cudaSuccess) {
      if (col->load_kind == LK_D32) widen_dec32_kernel<<<blocks, 256, 0, s>>>((const int*)d_out, d_wide, n);
      else widen_dec_kernel<<<blocks, 256, 0, s>>>((const u64*)d_out, d_wide, n);
      e = cudaGetLastError();
      result = d_wide;
    }
  }
  if (e == cudaSuccess) e = cudaMemcpyAsync(out_values, result, n * width, cudaMemcpyDeviceToHost, s);
  if (e == cudaSuccess) e = cudaMemcpyAsync(out_valid, d_valid, n, cudaMemcpyDeviceToHost, s);
  if (e == cudaSuccess) e = cudaStreamSynchronize(s);
  cudaFree(d_ids);
  cudaFree(d_out);
  cudaFree(d_valid);
  if (d_wide) cudaFree(d_wide);
  if (e != cudaSuccess) return set_error(LLKV_ERR_IO, "CUDA error %s gathering rows", cudaGetErrorString(e));
  return LLKV_OK;
}

// ColumnStore::scan with an unsorted visitor (llkv-column-map/src/store/scan/mod.rs:191-260, scan/unsorted.rs:202-345): the
// column's rows chunk by chunk, values in the Arrow layout, optionally with their row ids.  Rows the column does not hold
// (NULL by absence, deleted rows) are skipped, as with ScanOptions::include_nulls = false.
extern "C" int32_t llkv_gpu_column_visit(llkv_gpu_column* col, uint64_t chunk_rows, int32_t with_row_ids, llkv_chunk_visitor visit, void* user) {
  if (!col || !visit) return set_error(LLKV_ERR_INVALID_ARGUMENT, "NULL argument");
  if (col->type == LLKV_PT_UTF8) return set_error(LLKV_ERR_INVALID_ARGUMENT, "llkv_gpu_column_visit does not support Utf8 columns");
  llkv_gpu_ctx* c = col->ctx;
  CTX_LOCK(c);
  CUDA_TRY(cudaSetDevice(c->device));
  if (!col->sealed) {
    int32_t rc = llkv_gpu_column_seal(col);
    if (rc) return rc;
  }
  const uint64_t width = (uint64_t)prim_type_width(col->type);
  if (chunk_rows == 0) chunk_rows = width <= 8 ? (1ull << 20) / width : 4096;  // the append path's chunking (store/slicing.rs:33-43,155-166)
  chunk_rows = (chunk_rows + 31) / 32 * 32;
  std::vector<unsigned char> vals(chunk_rows * width), packed;
  std::vector<unsigned int> bits(chunk_rows / 32 + 1);
  std::vector<uint64_t> ids;
  for (uint64_t lo = 0; lo < col->n_rows; lo += chunk_rows) {
    const uint64_t n = std::min<uint64_t>(chunk_rows, col->n_rows - lo);
    int32_t rc = llkv_gpu_column_read(col, lo, n, vals.data(), vals.size());
    if (rc) return rc;
    const unsigned char* out_vals = vals.data();
    uint64_t out_n = n;
    if (col->validity) {  // keep the rows the column holds
      CUDA_TRY(cudaMemcpy(bits.data(), col->validity + lo / 32, ((n + 31) / 32) * 4, cudaMemcpyDeviceToHost));
      packed.resize(n * width);
      ids.clear();
      out_n = 0;
      for (uint64_t i = 0; i < n; ++i) {
        if (!((bits[i >> 5] >> (i & 31)) & 1u)) continue;
        memcpy(packed.data() + out_n * width, vals.data() + i * width, width);
        if (with_row_ids) ids.push_back(col->row_id_origin + lo + i);
        ++out_n;
      }
      out_vals = packed.data();
    } else if (with_row_ids) {
      ids.resize(n);
      for (uint64_t i = 0; i < n; ++i) ids[i] = col->row_id_origin + lo + i;
    }
    if (out_n == 0) continue;
    const int32_t vrc = visit(user, col->type, out_vals, with_row_ids ? ids.data() : nullptr, out_n);
    if (vrc) return set_error(vrc, "the chunk visitor stopped the scan with status %d", vrc);
  }
  return LLKV_OK;
}

// ColumnStore::scan(field, ScanOptions, visitor) (llkv-column-map/src/store/scan/mod.rs:191-1080): unsorted or sorted,
// forward or reverse, paginated, optionally with the rows the column does not hold as null runs.
struct ScanEmit {
  llkv_gpu_column* col;
  llkv_chunk_visitor visit;
  void* user;
  uint64_t skip, left;  // pagination state across chunks (PaginateVisitor)
  bool bounded, with_ids;
  int32_t emit(const void* values, const uint64_t* ids, uint64_t n, uint64_t width) {
    if (skip >= n) { skip -= n; return LLKV_OK; }
    const uint64_t first = skip;
    skip = 0;
    uint64_t m = n - first;
    if (bounded) {
      if (left == 0) return LLKV_OK;
      m = std::min(m, left);
      left -= m;
    }
    const int32_t vrc = visit(user, col->type, values ? (const char*)values + first * width : nullptr, ids && (with_ids || !values) ? ids + first : nullptr, m);
    return vrc ? set_error(vrc, "the visitor stopped the scan with status %d", vrc) : LLKV_OK;
  }
  bool done() const { return bounded && left == 0; }
};

extern "C" int32_t llkv_gpu_column_scan(llkv_gpu_column* col, llkv_gpu_column* anchor, const llkv_scan_options* o, uint64_t chunk_rows,
                                         llkv_chunk_visitor visit, void* user) {
  if (!col || !o || !visit) return set_error(LLKV_ERR_INVALID_ARGUMENT, "NULL argument");
  if (col->type == LLKV_PT_UTF8) return set_error(LLKV_ERR_INVALID_ARGUMENT, "llkv_gpu_column_scan does not support Utf8 columns");
  if (o->include_nulls && (!o->with_row_ids || !anchor)) return set_error(LLKV_ERR_INVALID_ARGUMENT, "include_nulls needs with_row_ids and an anchor column");
  if (o->include_nulls && !o->sorted) return set_error(LLKV_ERR_INVALID_ARGUMENT, "null runs are emitted by sorted scans on this path");
  llkv_gpu_ctx* c = col->ctx;
  CTX_LOCK(c);
  CUDA_TRY(cudaSetDevice(c->device));
  int32_t rc;
  if (!col->sealed && (rc = llkv_gpu_column_seal(col))) return rc;
  if (anchor && !anchor->sealed && (rc = llkv_gpu_column_seal(anchor))) return rc;
  if (o->sorted && col->load_kind == LK_D128) return set_error(LLKV_ERR_INVALID_ARGUMENT, "sorted scans take Decimal128 columns whose values fit i64");
  const uint64_t width = (uint64_t)prim_type_width(col->type);
  if (chunk_rows == 0) chunk_rows = width <= 8 ? (1ull << 20) / width : 4096;
  ScanEmit em{col, visit, user, o->offset, o->limit, o->limit != 0, o->with_row_ids != 0};
  const uint64_t n = col->n_rows, origin = col->row_id_origin;
  if (n >= (1ull << 32)) return set_error(LLKV_ERR_INVALID_ARGUMENT, "llkv_gpu_column_scan handles columns of up to 2^32 positions");
  if (!o->sorted) {  // append order; rows the column does not hold are skipped
    std::vector<unsigned char> vals(chunk_rows * width), packed(chunk_rows * width);
    std::vector<unsigned int> bits(chunk_rows / 32 + 2);
    std::vector<uint64_t> ids(chunk_rows);
    for (uint64_t lo = 0; lo < n && !em.done(); lo += chunk_rows) {
      const uint64_t m = std::min<uint64_t>(chunk_rows, n - lo);
      if ((rc = llkv_gpu_column_read(col, lo, m, vals.data(), vals.size()))) return rc;
      uint64_t out_n = 0;
      if (col->validity) CUDA_TRY(cudaMemcpy(bits.data(), col->validity + lo / 32, ((lo % 32 + m + 31) / 32) * 4, cudaMemcpyDeviceToHost));
      for (uint64_t i = 0; i < m; ++i) {
        const uint64_t b = lo % 32 + i;
        if (col->validity && !((bits[b >> 5] >> (b & 31)) & 1u)) continue;
        memcpy(packed.data() + out_n * width, vals.data() + i * width, width);
        ids[out_n++] = origin + lo + i;
      }
      if (out_n && (rc = em.emit(packed.data(), ids.data(), out_n, width))) return rc;
    }
    return LLKV_OK;
  }
  // ---- sorted: the order-preserving key image of every row, a stable partition (held and in range first), LSD passes
  u64 klo = 0, khi = ~0ull;
  auto image = [&](uint64_t bits) -> u64 {  // bound given as the value's bits in the column's type
    switch (col->load_kind) {
      case LK_F32: case LK_F64: {
        double d;
        if (col->load_kind == LK_F32) { float f; uint32_t b = (uint32_t)bits; memcpy(&f, &b, 4); d = f; } else memcpy(&d, &bits, 8);
        u64 b; memcpy(&b, &d, 8);
        return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
      }
      case LK_U8: case LK_U16: case LK_U32: case LK_U64: return bits;
      default: return bits ^ 0x8000000000000000ull;  // signed (sign-extended by the caller)
    }
  };
  if (o->has_lower) { klo = image(o->lower_bits); if (!o->lower_inclusive) { if (klo == ~0ull) return LLKV_OK; ++klo; } }
  if (o->has_upper) { khi = image(o->upper_bits); if (!o->upper_inclusive) { if (khi == 0) return LLKV_OK; --khi; } }
  uint64_t m = 0;
  unsigned int* d_perm = nullptr;  // (points into the scratch below)
  u64 *ka = nullptr, *kb = nullptr, *d_red = nullptr;
  unsigned int *ia = nullptr, *ib = nullptr, *d_counts = nullptr;
  unsigned char* d_flag = nullptr;
  cudaStream_t s = c->stream;
  const unsigned G = 148, S = G * kGsortThreads;
  auto release = [&]() {
    cudaFree(ka); cudaFree(kb); cudaFree(ia); cudaFree(ib); cudaFree(d_flag); cudaFree(d_counts); cudaFree(d_red);
  };
  if (n) {
    cudaError_t e = cudaMalloc((void**)&ka, n * 8);
    if (e == cudaSuccess) e = cudaMalloc((void**)&kb, n * 8);
    if (e == cudaSuccess) e = cudaMalloc((void**)&ia, n * 4);
    if (e == cudaSuccess) e = cudaMalloc((void**)&ib, n * 4);
    if (e == cudaSuccess) e = cudaMalloc((void**)&d_flag, n);
    if (e == cudaSuccess) e = cudaMalloc((void**)&d_counts, (size_t)16 * S * 4);
    if (e == cudaSuccess) e = cudaMalloc((void**)&d_red, 16);
    u64 red[2] = {~0ull, 0};
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_red, red, 16, cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) {
      const void* v = col->values;
#define LLKV_GSORT_INIT(T, KIND) gsort_init_kernel<T, KIND><<<1184, 256, 0, s>>>((const T*)v, col->validity, n, klo, khi, ka, ia, d_flag, d_red)
      switch (col->load_kind) {
        case LK_I8: LLKV_GSORT_INIT(signed char, 0); break;
        case LK_I16: LLKV_GSORT_INIT(short, 0); break;
        case LK_I32: case LK_D32: LLKV_GSORT_INIT(int, 0); break;
        case LK_I64: case LK_D64: LLKV_GSORT_INIT(i64, 0); break;
        case LK_U8: LLKV_GSORT_INIT(unsigned char, 1); break;
        case LK_U16: LLKV_GSORT_INIT(unsigned short, 1); break;
        case LK_U32: LLKV_GSORT_INIT(unsigned int, 1); break;
        case LK_U64: LLKV_GSORT_INIT(u64, 1); break;
        case LK_F32: LLKV_GSORT_INIT(float, 2); break;
        case LK_F64: LLKV_GSORT_INIT(double, 3); break;
        default: e = cudaErrorInvalidValue; break;
      }
#undef LLKV_GSORT_INIT
      if (e == cudaSuccess) e = cudaGetLastError();
    }
    auto pass = [&](int shift, u64 count) -> cudaError_t {
      const u64 seg = (count + S - 1) / S;
      gsort_count_kernel<<<G, kGsortThreads, 0, s>>>(ka, d_flag, count, shift, d_counts, seg, S);
      gsort_scan_kernel<<<1, 1024, 0, s>>>(d_counts, (u64)16 * S);
      gsort_scatter_kernel<<<G, kGsortThreads, 0, s>>>(ka, ia, d_flag, count, shift, d_counts, seg, S, kb, ib);
      std::swap(ka, kb);
      std::swap(ia, ib);
      return cudaGetLastError();
    };
    m = n;
    const bool filtered = col->validity || o->has_lower || o->has_upper;
    if (e == cudaSuccess && filtered) {
      e = pass(-1, n);
      unsigned int kept = 0;  // exclusive offset of the first flagged row = rows kept
      if (e == cudaSuccess) e = cudaMemcpyAsync(&kept, d_counts + S, 4, cudaMemcpyDeviceToHost, s);
      if (e == cudaSuccess) e = cudaStreamSynchronize(s);
      m = kept;
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(red, d_red, 16, cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    const u64 varying = m ? (red[0] ^ red[1]) : 0;  // bits in which the kept keys differ: the other digits need no pass
    for (int shift = 0; shift < 64 && e == cudaSuccess && m > 1; shift += 4)
      if ((varying >> shift) & 15u) e = pass(shift, m);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    if (e != cudaSuccess) {
      release();
      return set_error(LLKV_ERR_IO, "CUDA error %s sorting the column", cudaGetErrorString(e));
    }
    d_perm = ia;
  }
  // rows of the anchor that the column does not hold, ascending (descending for reverse scans)
  std::vector<uint64_t> nulls;
  if (o->include_nulls) {
    const uint64_t an = anchor->n_rows;
    std::vector<unsigned int> av((an + 31) / 32 + 1, 0xffffffffu), cv((n + 31) / 32 + 1, 0xffffffffu);
    cudaError_t e = cudaSuccess;
    if (anchor->validity && an) e = cudaMemcpy(av.data(), anchor->validity, ((an + 31) / 32) * 4, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess && col->validity && n) e = cudaMemcpy(cv.data(), col->validity, ((n + 31) / 32) * 4, cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) { release(); return set_error(LLKV_ERR_IO, "CUDA error %s", cudaGetErrorString(e)); }
    for (uint64_t i = 0; i < an; ++i) {
      if (!((av[i >> 5] >> (i & 31)) & 1u)) continue;
      const uint64_t rid = anchor->row_id_origin + i, pos = rid - origin;
      const bool held = rid >= origin && pos < n && ((cv[pos >> 5] >> (pos & 31)) & 1u);
      if (!held) nulls.push_back(rid);
    }
    if (o->reverse) std::reverse(nulls.begin(), nulls.end());
  }
  auto emit_nulls = [&]() -> int32_t {
    for (uint64_t lo = 0; lo < nulls.size() && !em.done(); lo += chunk_rows) {
      const int32_t r = em.emit(nullptr, nulls.data() + lo, std::min<uint64_t>(chunk_rows, nulls.size() - lo), 0);
      if (r) return r;
    }
    return LLKV_OK;
  };
  auto emit_values = [&]() -> int32_t {
    std::vector<unsigned int> perm(chunk_rows);
    std::vector<uint64_t> ids(chunk_rows);
    std::vector<unsigned char> vals(chunk_rows * width), valid(chunk_rows);
    uint64_t at = 0;
    if (em.skip >= m) { em.skip -= m; return LLKV_OK; }  // the page starts behind the values
    at = em.skip;
    em.skip = 0;
    while (at < m && !em.done()) {
      uint64_t k = std::min<uint64_t>(chunk_rows, m - at);
      if (em.bounded) k = std::min(k, em.left);
      const uint64_t src = o->reverse ? m - at - k : at;
      CUDA_TRY(cudaMemcpy(perm.data(), d_perm + src, k * 4, cudaMemcpyDeviceToHost));
      for (uint64_t i = 0; i < k; ++i) ids[i] = origin + perm[o->reverse ? k - 1 - i : i];
      int32_t r = llkv_gpu_column_gather(col, ids.data(), k, vals.data(), vals.size(), valid.data());
      if (r) return r;
      if ((r = em.emit(vals.data(), ids.data(), k, width))) return r;
      at += k;
    }
    return LLKV_OK;
  };
  rc = LLKV_OK;
  if (o->include_nulls && o->nulls_first) rc = emit_nulls();
  if (!rc && m) rc = emit_values();
  else if (!rc && !m) { /* nothing held */ }
  if (!rc && o->include_nulls && !o->nulls_first) rc = emit_nulls();
  release();
  return rc;
}

extern "C" int32_t llkv_gpu_column_dict_size(llkv_gpu_column* col, uint64_t* out_entries) {
  if (!col || !out_entries) return set_error(LLKV_ERR_INVALID_ARGUMENT, "NULL argument");
  CTX_LOCK(col->ctx);
  if (col->dict && !col->sealed) {
    int32_t rc = llkv_gpu_column_seal(col);
    if (rc) return rc;
  }
  *out_entries = col->dict ? col->dict->sorted.size() : 0;
  return LLKV_OK;
}

extern "C" int32_t llkv_gpu_column_dict_entry(llkv_gpu_column* col, uint64_t code, const uint8_t** out_bytes, uint64_t* out_len) {
  if (!col || !out_bytes || !out_len) return set_error(LLKV_ERR_INVALID_ARGUMENT, "NULL argument");
  CTX_LOCK(col->ctx);
  if (!col->dict) return set_error(LLKV_ERR_INVALID_ARGUMENT, "the column is not dictionary-coded");
  if (code >= col->dict->sorted.size()) return set_error(LLKV_ERR_NOT_FOUND, "no dictionary entry %llu", (unsigned long long)code);
  const std::string& e = col->dict->sorted[(size_t)code];
  *out_bytes = (const uint8_t*)e.data();
  *out_len = e.size();
  return LLKV_OK;
}

extern "C" int32_t llkv_gpu_column_build_sort_index(llkv_gpu_column* col, uint64_t chunk_rows) {
  if (!col) return set_error(LLKV_ERR_INVALID_ARGUMENT, "column is NULL");
  llkv_gpu_ctx* c = col->ctx;
  CTX_LOCK(c);
  CUDA_TRY(cudaSetDevice(c->device));
  if (!col->sealed) {
    int32_t rc = llkv_gpu_column_seal(col);
    if (rc) return rc;
  }
  if (col->validity) return set_error(LLKV_ERR_INVALID_ARGUMENT, "the sort index covers columns without gaps or NULLs");
  if (col->type == LLKV_PT_UTF8 || col->load_kind == LK_D128) return set_error(LLKV_ERR_INVALID_ARGUMENT, "no sort index for this column type");
  const uint64_t width = (uint64_t)prim_type_width(col->type);
  if (chunk_rows == 0) chunk_rows = width <= 8 ? (1ull << 20) / width : 4096;  // the append path's chunking (store/slicing.rs:33-43,155-166)
  if (chunk_rows > (1ull << 20)) return set_error(LLKV_ERR_INVALID_ARGUMENT, "sort-index chunks hold at most 2^20 rows");
  const uint64_t n = col->n_rows;
  if (n == 0) return LLKV_OK;
  if (col->d_perm) CUDA_TRY(cudaFree(col->d_perm));
  col->d_perm = nullptr;
  CUDA_TRY(cudaMalloc((void**)&col->d_perm, n * 4));
  u64 *ka = nullptr, *kb = nullptr;
  unsigned int *ia = nullptr, *ib = nullptr;
  cudaError_t e = cudaMalloc((void**)&ka, n * 8);
  if (e == cudaSuccess) e = cudaMalloc((void**)&kb, n * 8);
  if (e == cudaSuccess) e = cudaMalloc((void**)&ia, n * 4);
  if (e == cudaSuccess) e = cudaMalloc((void**)&ib, n * 4);
  const unsigned grid = (unsigned)((n + chunk_rows - 1) / chunk_rows);
  cudaStream_t s = c->stream;
  if (e == cudaSuccess) {
    const void* v = col->values;
#define LLKV_SORT(T, KIND, BYTES) chunk_sort_kernel<T, KIND><<<grid, kSortThreads, 0, s>>>((const T*)v, n, chunk_rows, 2 * (BYTES), ka, kb, ia, ib, col->d_perm)
    switch (col->load_kind) {
      case LK_I8: LLKV_SORT(signed char, 0, 8); break;  // (the sign-extended image: all 64 bits take part)
      case LK_I16: LLKV_SORT(short, 0, 8); break;
      case LK_I32: case LK_D32: LLKV_SORT(int, 0, 8); break;
      case LK_I64: case LK_D64: LLKV_SORT(i64, 0, 8); break;
      case LK_U8: LLKV_SORT(unsigned char, 1, 1); break;
      case LK_U16: LLKV_SORT(unsigned short, 1, 2); break;
      case LK_U32: LLKV_SORT(unsigned int, 1, 4); break;
      case LK_U64: LLKV_SORT(u64, 1, 8); break;
      case LK_F32: LLKV_SORT(float, 2, 8); break;
      case LK_F64: LLKV_SORT(double, 3, 8); break;
      default: e = cudaErrorInvalidValue; break;
    }
#undef LLKV_SORT
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
  }
  cudaFree(ka);
  cudaFree(kb);
  cudaFree(ia);
  cudaFree(ib);
  if (e != cudaSuccess) return set_error(LLKV_ERR_IO, "CUDA error %s building the sort index", cudaGetErrorString(e));
  col->perm_chunk_rows = chunk_rows;
  col->perm_version = col->version;
  return LLKV_OK;
}

extern "C" int32_t llkv_gpu_column_sort_index_blob(llkv_gpu_column* col, uint64_t chunk_index, void* out_blob, uint64_t cap, uint64_t* out_len) {
  if (!col || !out_len) return set_error(LLKV_ERR_INVALID_ARGUMENT, "NULL argument");
  llkv_gpu_ctx* c = col->ctx;
  CTX_LOCK(c);
  CUDA_TRY(cudaSetDevice(c->device));
  if (!col->d_perm || col->perm_version != col->version) return set_error(LLKV_ERR_NOT_FOUND, "the column has no current sort index (llkv_gpu_column_build_sort_index)");
  const uint64_t base = chunk_index * col->perm_chunk_rows;
  if (base >= col->n_rows) return set_error(LLKV_ERR_NOT_FOUND, "chunk %llu is past the column's end", (unsigned long long)chunk_index);
  const uint64_t m = std::min<uint64_t>(col->perm_chunk_rows, col->n_rows - base);
  *out_len = 24 + 4 * m;
  if (!out_blob) return LLKV_OK;  // (size query)
  if (cap < *out_len) return set_error(LLKV_ERR_INVALID_ARGUMENT, "blob buffer too small (%llu bytes needed)", (unsigned long long)*out_len);
  // "ARR0" | layout 0 (Primitive) | PrimType UInt32 | 0 | 0 | len u64 | values bytes u32 | 0  (serialization.rs:41-53,264-307)
  unsigned char* b = (unsigned char*)out_blob;
  memcpy(b, "ARR0", 4);
  b[4] = 0;
  b[5] = (unsigned char)LLKV_PT_UINT32;
  b[6] = b[7] = 0;
  const uint64_t len = m;
  const uint32_t bytes = (uint32_t)(4 * m), zero = 0;
  memcpy(b + 8, &len, 8);
  memcpy(b + 16, &bytes, 4);
  memcpy(b + 20, &zero, 4);
  CUDA_TRY(cudaMemcpy(b + 24, col->d_perm + base, 4 * m, cudaMemcpyDeviceToHost));
  return LLKV_OK;
}

extern "C" int32_t llkv_gpu_column_present_rows(llkv_gpu_column* col, uint64_t* out_rows) {
  if (!col || !out_rows) return set_error(LLKV_ERR_INVALID_ARGUMENT, "NULL argument");
  llkv_gpu_ctx* c = col->ctx;
  CTX_LOCK(c);
  CUDA_TRY(cudaSetDevice(c->device));
  int32_t rc = column_flush(col);
  if (rc) return rc;
  *out_rows = col->n_rows;
  if (!col->validity || col->n_rows == 0) return LLKV_OK;
  u64* d = nullptr;
  CUDA_TRY(cudaMalloc((void**)&d, 8));
  cudaStream_t s = c->copy_streams[(size_t)col->stream_index];
  cudaError_t e = cudaMemsetAsync(d, 0, 8, s);
  if (e == cudaSuccess) {
    popcount_bits_kernel<<<(unsigned)std::min<uint64_t>((col->n_rows / 32 + 256) / 256, 1184), 256, 0, s>>>(col->validity, col->n_rows, d);
    e = cudaGetLastError();
  }
  u64 h = 0;
  if (e == cudaSuccess) e = cudaMemcpyAsync(&h, d, 8, cudaMemcpyDeviceToHost, s);
  if (e == cudaSuccess) e = cudaStreamSynchronize(s);
  cudaFree(d);
  if (e != cudaSuccess) return set_error(LLKV_ERR_IO, "CUDA error %s counting rows", cudaGetErrorString(e));
  *out_rows = h;
  return LLKV_OK;
}

extern "C" int32_t llkv_gpu_column_h2d_bytes(const llkv_gpu_column* col, uint64_t* out_bytes) {
  if (!col || !out_bytes) return set_error(LLKV_ERR_INVALID_ARGUMENT, "NULL argument");
  *out_bytes = col->h2d_bytes;
  return LLKV_OK;
}

extern "C" int32_t llkv_gpu_column_read(llkv_gpu_column* col, uint64_t row_begin, uint64_t n_rows, void* out, uint64_t out_bytes) {
  if (!col || (n_rows && !out)) return set_error(LLKV_ERR_INVALID_ARGUMENT, "NULL argument");
  if (col->type == LLKV_PT_UTF8) return set_error(LLKV_ERR_INVALID_ARGUMENT, "llkv_gpu_column_read does not support Utf8 columns");
  llkv_gpu_ctx* c = col->ctx;
  CTX_LOCK(c);
  CUDA_TRY(cudaSetDevice(c->device));
  if (!col->sealed) {
    int32_t rc = llkv_gpu_column_seal(col);
    if (rc) return rc;
  }
  if (row_begin > col->n_rows || n_rows > col->n_rows - row_begin)
    return set_error(LLKV_ERR_INVALID_ARGUMENT, "rows [%llu, +%llu) beyond the column's %llu rows", (unsigned long long)row_begin, (unsigned long long)n_rows,
                     (unsigned long long)col->n_rows);
  const uint64_t width = (uint64_t)prim_type_width(col->type);
  if (out_bytes < n_rows * width) return set_error(LLKV_ERR_INVALID_ARGUMENT, "output buffer too small");
  if (n_rows == 0) return LLKV_OK;
  if (is_narrow_decimal(col)) {  // resident i64 / i32 image of a Decimal128 column: widen the range on the device first
    ulonglong2* wide = nullptr;
    CUDA_TRY(cudaMalloc((void**)&wide, n_rows * 16));
    const unsigned blocks = (unsigned)std::min<uint64_t>((n_rows + 255) / 256, 1184);
    if (col->load_kind == LK_D32) widen_dec32_kernel<<<blocks, 256, 0, c->stream>>>((const int*)col->values + row_begin, wide, n_rows);
    else widen_dec_kernel<<<blocks, 256, 0, c->stream>>>((const u64*)col->values + row_begin, wide, n_rows);
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaMemcpyAsync(out, wide, n_rows * 16, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    cudaFree(wide);
    if (e != cudaSuccess) return set_error(LLKV_ERR_IO, "CUDA error %s reading the column", cudaGetErrorString(e));
    return LLKV_OK;
  }
  CUDA_TRY(cudaMemcpyAsync(out, (const char*)col->values + row_begin * col->elem_bytes, n_rows * col->elem_bytes, cudaMemcpyDeviceToHost, c->stream));
  CUDA_TRY(cudaStreamSynchronize(c->stream));
  return LLKV_OK;
}

extern "C" int32_t llkv_gpu_column_clear(llkv_gpu_column* col) {
  if (!col) return set_error(LLKV_ERR_INVALID_ARGUMENT, "column is NULL");
  llkv_gpu_ctx* c = col->ctx;
  CTX_LOCK(c);
  CUDA_TRY(cudaSetDevice(c->device));
  cudaStream_t s = c->copy_streams[(size_t)col->stream_index];
  col->pend_bytes = 0;  // rows that were never copied are dropped with the rest
  {
    int32_t rc = drain_jobs(col);
    if (rc) return rc;
    col->narrow_chunks.clear();
    col->ticket.failed.store(0);
  }
  CUDA_TRY(cudaStreamSynchronize(c->stream));
  if (col->type == LLKV_PT_UTF8 && col->load_kind == LK_STR8) {  // back to the packed representation for new appends
    if (col->values) CUDA_TRY(cudaFree(col->values));
    col->values = nullptr;
    col->cap_rows = 0;
    col->elem_bytes = 8;
    col->load_kind = LK_U64;
  }
  col->dict.reset();
  col->reupload_hint = true;
  if (is_narrow_decimal(col)) {  // back to the Arrow layout for new appends; the narrow buffer is parked for the next batch
    if (col->narrow && col->narrow != col->values) CUDA_TRY(cudaFree(col->narrow));
    col->narrow = col->values;
    col->narrow_cap = col->cap_rows;
    col->narrow_width = col->elem_bytes;
    col->values = col->landing;
    col->cap_rows = col->landing ? col->landing_cap : 0;
    col->landing = nullptr;
    col->landing_cap = 0;
    col->elem_bytes = 16;
    col->load_kind = LK_D128;
    if (col->validity) {  // sized by the capacity that was just parked
      CUDA_TRY(cudaFree(col->validity));
      col->validity = nullptr;
    }
  }
  if (col->validity) CUDA_TRY(cudaMemsetAsync(col->validity, 0, (col->cap_rows / 32 + 4) * 4, s));
  DevStats init;
  memset(&init, 0, sizeof(init));
  init.min_enc = ~0ull;
  init.min_strlen = 0xffffffffu;
  col->hstats = init;
  CUDA_TRY(cudaMemcpyAsync(col->dstats, &col->hstats, sizeof(DevStats), cudaMemcpyHostToDevice, s));
  CUDA_TRY(cudaStreamSynchronize(s));
  col->n_rows = 0;
  col->stats_rows = 0;
  col->has_origin = false;
  col->sealed = false;
  col->sparse = false;
  ++col->version;
  ++c->state_epoch;
  col->scans_unchanged = 0;
  return LLKV_OK;
}

extern "C" int32_t llkv_gpu_column_destroy(llkv_gpu_column* col) {
  if (!col) return LLKV_OK;
  llkv_gpu_ctx* c = col->ctx;
  CTX_LOCK(c);
  cudaSetDevice(c->device);
  col->pend_bytes = 0;
  drain_jobs(col);
  cudaDeviceSynchronize();
  c->columns.erase(col->lfid);
  ++c->state_epoch;
  for (auto& kv : c->mvcc)
    if (kv.second.created_by == col || kv.second.deleted_by == col) kv.second.created_by = kv.second.deleted_by = nullptr;
  for (void* p : col->deferred_free) cudaFree(p);
  if (col->landing) cudaFree(col->landing);
  if (col->narrow) cudaFree(col->narrow);
  if (col->values) cudaFree(col->values);
  if (col->validity) cudaFree(col->validity);
  if (col->dstats) cudaFree(col->dstats);
  if (col->d_zones) cudaFree(col->d_zones);
  if (col->d_perm) cudaFree(col->d_perm);
  if (col->d_fit) cudaFree(col->d_fit);
  delete col;
  return LLKV_OK;
}

// ------------------------------------------------------------------------------------------------ programs / MVCC
extern "C" int32_t llkv_gpu_program_compile(llkv_gpu_ctx* ctx, const llkv_eval_op* ops, int32_t n_ops, const llkv_literal* literals,
                                             int32_t n_literals, const llkv_scalar_node* nodes, int32_t n_nodes,
                                             const int32_t* list_roots, int32_t n_list_roots, llkv_gpu_program** out) {
  (void)ctx;  // programs are host objects: a NULL context is accepted (llkv_gpu_debug_plan)
  if (!out) return set_error(LLKV_ERR_INVALID_ARGUMENT, "NULL argument");
  *out = nullptr;
  if (n_ops < 0 || n_literals < 0 || n_nodes < 0 || n_list_roots < 0) return set_error(LLKV_ERR_INVALID_ARGUMENT, "negative count");
  if ((n_ops && !ops) || (n_literals && !literals) || (n_nodes && !nodes) || (n_list_roots && !list_roots))
    return set_error(LLKV_ERR_INVALID_ARGUMENT, "NULL array with a non-zero count");
  for (int i = 0; i < n_ops; ++i) {
    const int t = ops[i].tag;
    if (!((t >= LLKV_EV_PUSH_PREDICATE && t <= LLKV_EV_NOT) || t == LLKV_EV_FILTER_ITEM))
      return set_error(LLKV_ERR_INTERNAL, "unknown eval op tag %d", t);
  }
  llkv_gpu_program* p = new llkv_gpu_program();
  static std::atomic<uint64_t> next_serial{1};
  p->serial = next_serial.fetch_add(1);
  p->ops.assign(ops, ops + n_ops);
  p->literals.assign(literals, literals + n_literals);
  p->nodes.assign(nodes, nodes + n_nodes);
  p->list_roots.assign(list_roots, list_roots + n_list_roots);
  for (llkv_literal& l : p->literals) own_string_literal(l, p->strings);
  for (llkv_scalar_node& nd : p->nodes)
    if (nd.tag == LLKV_SE_LITERAL) own_string_literal(nd.literal, p->strings);
  p->bind();
  *out = p;
  return LLKV_OK;
}

extern "C" void llkv_gpu_program_destroy(llkv_gpu_program* prog) { delete prog; }

extern "C" int32_t llkv_gpu_mvcc_set(llkv_gpu_ctx* ctx, uint64_t table_id, llkv_gpu_column* created_by, llkv_gpu_column* deleted_by,
                                      uint64_t txn_id, uint64_t snapshot_id, const uint64_t* noncommitted, int32_t n_noncommitted) {
  if (!ctx) return set_error(LLKV_ERR_INVALID_ARGUMENT, "ctx is NULL");
  if (n_noncommitted < 0 || (n_noncommitted && !noncommitted)) return set_error(LLKV_ERR_INVALID_ARGUMENT, "bad non-committed list");
  if (n_noncommitted > kMaxNoncommitted) return set_error(LLKV_ERR_INVALID_ARGUMENT, "more than %d non-committed transactions in one snapshot", kMaxNoncommitted);
  if ((created_by && created_by->type != LLKV_PT_UINT64) || (deleted_by && deleted_by->type != LLKV_PT_UINT64))
    return set_error(LLKV_ERR_INVALID_ARGUMENT, "MVCC columns must be UInt64");
  CTX_LOCK(ctx);
  MvccState& m = ctx->mvcc[table_id];
  m.created_by = created_by;
  m.deleted_by = deleted_by;
  m.txn_id = txn_id;
  m.snapshot_id = snapshot_id;
  m.noncommitted.assign(noncommitted, noncommitted + n_noncommitted);
  ++ctx->state_epoch;
  return LLKV_OK;
}

extern "C" int32_t llkv_gpu_mvcc_clear(llkv_gpu_ctx* ctx, uint64_t table_id) {
  if (!ctx) return set_error(LLKV_ERR_INVALID_ARGUMENT, "ctx is NULL");
  CTX_LOCK(ctx);
  ctx->mvcc.erase(table_id);
  ++ctx->state_epoch;
  return LLKV_OK;
}

// ------------------------------------------------------------------------------------------------ plan building
static uint64_t lfid_table(uint64_t lfid) { return (lfid >> 32) & 0xffffull; }  // llkv-types/src/ids.rs:133-152
static uint64_t lfid_field(uint64_t lfid) { return lfid & 0xffffffffull; }

// Row-id-sparse tables: every column covers positions [0, n) of the table's row-id range.  A column whose last rows are
// absent (NULL by absence) is shorter than the others: it grows to the table's span, the new positions invalid (Utf8 columns
// too, in whichever form they are resident: packed keys, one byte per row or dictionary codes).
static int32_t equalise_sparse_columns(llkv_gpu_ctx* ctx, uint64_t table_id) {
  uint64_t longest = 0;
  bool differ = false, any = false;
  for (auto& kv : ctx->columns) {
    llkv_gpu_column* col = kv.second;
    if (lfid_table(col->lfid) != (table_id & 0xffffull)) continue;
    if (any && col->n_rows != longest) differ = true;
    longest = std::max(longest, col->n_rows);
    any = true;
  }
  if (!differ) return LLKV_OK;
  bool sparse_table = false;
  for (auto& kv : ctx->columns)
    if (lfid_table(kv.second->lfid) == (table_id & 0xffffull) && kv.second->sparse) sparse_table = true;
  if (!sparse_table) return LLKV_OK;  // dense tables keep the old rule: scans cover the rows every column has
  for (auto& kv : ctx->columns) {
    llkv_gpu_column* col = kv.second;
    if (lfid_table(col->lfid) != (table_id & 0xffffull) || col->n_rows == longest) continue;
    int32_t rc;
    if ((rc = column_flush(col))) return rc;
    if (is_narrow_decimal(col) && (rc = widen_decimal(col, col->n_rows))) return rc;
    if ((rc = column_grow(col, longest)) || (rc = ensure_validity(col))) return rc;
    CUDA_TRY(cudaStreamSynchronize(ctx->copy_streams[(size_t)col->stream_index]));
    col->n_rows = longest;
    col->sparse = true;
    col->sealed = false;
    ++col->version;
    ++ctx->state_epoch;
  }
  return LLKV_OK;
}

// The table's rows when positions are row ids: the MVCC created_by column's rows when the table has one, else the union of
// the user columns' rows (Table::compute_table_row_ids, llkv-table/src/table.rs:1361-1421).  nullptr = every position.
static int32_t table_exists_bits(llkv_gpu_ctx* ctx, uint64_t table_id, const std::vector<llkv_gpu_column*>& handles, uint64_t rows,
                                 const unsigned char** out) {
  *out = nullptr;
  bool sparse_table = false;
  for (llkv_gpu_column* h : handles) sparse_table = sparse_table || h->sparse;
  if (!sparse_table) return LLKV_OK;  // chunks arrived as dense runs (NULLs, if any, as validity bits): every position is a row
  auto it = ctx->mvcc.find(table_id);
  llkv_gpu_column* created = nullptr;
  for (llkv_gpu_column* h : handles)
    if ((h->lfid >> 48) == 2 /* LogicalStorageNamespace::TxnCreatedBy */) created = h;
  if (it != ctx->mvcc.end() && it->second.created_by) created = it->second.created_by;
  if (created) {
    *out = (const unsigned char*)created->validity;
    return LLKV_OK;
  }
  uint64_t key = 0xcbf29ce484222325ull;
  std::vector<llkv_gpu_column*> users;
  for (llkv_gpu_column* h : handles) {
    if ((h->lfid >> 48) != 0) continue;  // user columns only
    if (!h->validity) return LLKV_OK;    // a column that holds every position: every position is a row
    users.push_back(h);
    key = fnv_pod(fnv_pod(key, (uint64_t)(uintptr_t)h), h->version);
  }
  if (users.empty() || rows == 0) return LLKV_OK;
  if (users.size() == 1) {
    *out = (const unsigned char*)users[0]->validity;
    return LLKV_OK;
  }
  llkv_gpu_ctx::ExistsCache& ec = ctx->exists[table_id];
  const uint64_t words = rows / 32 + 4 + kPadRows / 32;
  if (ec.key != key || ec.words < words) {
    if (ec.words < words) {
      if (ec.bits) CUDA_TRY(cudaFree(ec.bits));
      ec.bits = nullptr;
      ec.words = 0;
      CUDA_TRY(cudaMalloc((void**)&ec.bits, words * 4));
      ec.words = words;
    }
    CUDA_TRY(cudaMemsetAsync(ec.bits, 0, ec.words * 4, ctx->stream));
    const uint64_t nw = (rows + 31) / 32;
    for (llkv_gpu_column* h : users) {
      or_words_kernel<<<(unsigned)std::min<uint64_t>((nw + 255) / 256, 1184), 256, 0, ctx->stream>>>(ec.bits, h->validity, nw);
      CUDA_TRY(cudaGetLastError());
    }
    ec.key = key;
  }
  *out = (const unsigned char*)ec.bits;
  return LLKV_OK;
}

static int32_t collect_columns(llkv_gpu_ctx* ctx, uint64_t table_id, std::vector<ColumnMeta>& cols,
                               std::vector<llkv_gpu_column*>& handles, uint64_t* table_rows) {
  cols.clear();
  handles.clear();
  {
    int32_t erc = equalise_sparse_columns(ctx, table_id);
    if (erc) return erc;
  }
  bool have = false;
  uint64_t rows = 0;
  for (auto& kv : ctx->columns) {
    llkv_gpu_column* col = kv.second;
    if (lfid_table(col->lfid) != (table_id & 0xffffull)) continue;
    if (!col->sealed) {
      int32_t rc = llkv_gpu_column_seal(col);
      if (rc) return rc;
    }
    ColumnMeta m;
    m.field_id = lfid_field(col->lfid) | ((col->lfid >> 48) << 48);  // namespaced (MVCC) columns keep their namespace bits
    m.type = col->type;
    m.precision = col->precision;
    m.scale = col->scale;
    m.nullable = col->validity != nullptr;
    m.load_kind = col->load_kind;
    m.elem_bytes = col->elem_bytes;
    if (col->type == LLKV_PT_UTF8) m.arrow_bytes = 4 + (uint32_t)(col->n_rows ? (col->hstats.data_bytes + col->n_rows - 1) / col->n_rows : 0);
    else m.arrow_bytes = (uint32_t)prim_type_width(col->type);
    m.dev_values = col->values;
    m.dev_validity = (const unsigned char*)col->validity;
    m.n_rows = col->n_rows;
    m.dec_fits_i64 = col->hstats.not_i64 == 0;
    const bool is_signed = col->type == LLKV_PT_INT8 || col->type == LLKV_PT_INT16 || col->type == LLKV_PT_INT32 ||
                           col->type == LLKV_PT_INT64 || col->type == LLKV_PT_DATE32 || col->type == LLKV_PT_DATE64;
    const bool is_unsigned = col->type == LLKV_PT_UINT8 || col->type == LLKV_PT_UINT16 || col->type == LLKV_PT_UINT32 ||
                             col->type == LLKV_PT_UINT64 || col->type == LLKV_PT_BOOLEAN;
    const bool dec_narrow = col->type == LLKV_PT_DECIMAL128 && col->hstats.not_i64 == 0;
    if ((is_signed || is_unsigned || dec_narrow) && col->n_rows && col->hstats.min_enc <= col->hstats.max_enc) {
      m.has_minmax = true;
      m.min_bits = (is_signed || dec_narrow) ? (col->hstats.min_enc ^ 0x8000000000000000ull) : col->hstats.min_enc;
      m.max_bits = (is_signed || dec_narrow) ? (col->hstats.max_enc ^ 0x8000000000000000ull) : col->hstats.max_enc;
    }
    m.max_strlen = (uint8_t)col->hstats.max_strlen;
    m.str_non_ascii = (col->hstats.bad_string & 2u) != 0;
    if (col->dict) {  // codes are ranks 0 .. entries-1: an unsigned integer column as far as leaves and keys are concerned
      m.dict_sorted = &col->dict->sorted;
      m.dict_epoch = col->dict->epoch;
      m.str_non_ascii = col->dict->non_ascii;
      m.has_minmax = !col->dict->sorted.empty();
      m.min_bits = 0;
      m.max_bits = col->dict->sorted.empty() ? 0 : col->dict->sorted.size() - 1;
    }
    cols.push_back(m);
    handles.push_back(col);
    if (!have) {
      rows = col->n_rows;
      have = true;
    } else if (col->n_rows < rows) {
      rows = col->n_rows;
    }
  }
  *table_rows = have ? rows : 0;
  return LLKV_OK;
}

struct Geometry {
  uint32_t grid = 0, block = 0, R = 1, smem = 0;
};

static uint32_t align_up(uint32_t v, uint32_t a) { return (v + a - 1) / a * a; }
static u64 next_pow2(u64 v) {
  u64 p = 1;
  while (p < v) p <<= 1;
  return p;
}

// Rows of a grouped aggregate's global table at its first run: small when the caller knows the cardinality (Q1: 6 groups
// -> 32 rows), since finalize and the multi-GPU merge move the whole table; it grows x4 on FLAG_TABLE_FULL if the hint was wrong
static u64 group_table_cap(u64 hint) { return hint ? next_pow2(std::max<u64>(32, hint * 2)) : 1024; }

// General interpreter: chooses block size, rows per thread, pipeline depth and CTA-local group slots so that the plan fits
// in shared memory, and fills the launch-geometry / shared-memory fields of the plan.
static int32_t plan_geometry(llkv_gpu_ctx* ctx, Plan& p, bool wide, uint64_t row_begin, uint64_t row_end, uint64_t hint, Geometry& g) {
  const uint32_t vbytes = wide ? 16u : 8u;
  uint32_t NT = ctx->tune_block ? (uint32_t)ctx->tune_block : 512u;
  uint32_t R = ctx->tune_rpt ? (uint32_t)ctx->tune_rpt : (wide ? 1u : 2u);
  if (wide && R > 2) R = 2;
  if (R > 4) R = 4;
  uint32_t stages = ctx->tune_stages ? (uint32_t)ctx->tune_stages : 3u;
  uint32_t ctas = ctx->tune_ctas ? (uint32_t)ctx->tune_ctas : 2u;
  uint32_t FG = 0;
  if (p.n_fast_words) {
    if (p.n_keys == 0) FG = 1;
    else if (hint == 0) FG = 16;
    else if (hint <= 128) FG = (uint32_t)next_pow2(hint + hint / 2 + 1);
  }
  const uint32_t budget_total = (uint32_t)ctx->max_smem;
  for (int attempt = 0; attempt < 64; ++attempt) {
    const uint32_t T = NT * R;
    const bool staged = stages >= 2;
    uint32_t off = align_up((uint32_t)sizeof(Plan), 128);
    p.smem_bar_off = off;
    off += 128;
    p.smem_stage_off = off;
    uint32_t stage_bytes = 0, tx = 0;
    if (staged) {
      for (uint32_t c = 0; c < p.n_cols; ++c) {
        p.cols[c].smem_off = stage_bytes;
        stage_bytes += align_up(T * p.cols[c].elem_bytes, 128);
        tx += T * p.cols[c].elem_bytes;
        if (p.cols[c].validity) {
          p.cols[c].vsmem_off = stage_bytes;
          stage_bytes += align_up(T / 8, 128);
          tx += T / 8;
        }
      }
      off += stage_bytes * stages;
    }
    p.smem_acc_off = off;
    off += align_up(FG * p.n_fast_words * NT * 8, 128);
    p.smem_spill_off = off;
    const uint32_t spill_slots = p.max_depth > 2 ? p.max_depth - 2 : 0;
    off += align_up(spill_slots * R * NT * vbytes, 128);
    p.smem_tbl_off = off;
    off += align_up((FG ? FG : 1) * 8, 128);
    const uint32_t per_cta_budget = budget_total / ctas - 1024;
    if (off <= per_cta_budget) {
      p.tile_rows = T;
      p.stages = staged ? stages : 1;
      p.staged = staged ? 1 : 0;
      p.stage_bytes = stage_bytes;
      p.tx_bytes = tx;
      p.fast_groups = FG;
      p.smem_total = off;
      p.row_begin = row_begin;
      p.row_end = row_end;
      p.first_tile = row_begin / T;
      p.n_tiles = row_end > row_begin ? (row_end + T - 1) / T - p.first_tile : 0;
      g.block = NT;
      g.R = R;
      g.smem = off;
      u64 grid = (u64)ctx->sm_count * ctas;
      if (grid > p.n_tiles) grid = p.n_tiles;
      if (grid == 0) grid = 1;
      g.grid = (uint32_t)grid;
      return LLKV_OK;
    }
    // shrink: fewer CTAs per SM, shallower pipeline, fewer rows per thread, smaller block, fewer CTA-local groups
    if (ctas > 1) ctas -= 1;
    else if (stages > 2) stages -= 1;
    else if (R > 1) R /= 2;
    else if (FG > 4 && p.n_keys) FG /= 2;
    else if (NT > 128) NT /= 2;
    else if (FG > 0 && p.n_keys) FG = 0;
    else if (stages >= 2) stages = 1;
    else break;
  }
  return set_error(LLKV_ERR_INVALID_ARGUMENT, "query state does not fit in shared memory on this path");
}

// Lean kernel (lean_kernel.cuh): picks consumer threads, rows per thread, pipeline depth, CTAs per SM and CTA-local group
// slots so that stages + thread-private accumulators fit in shared memory, and builds the kernel's by-value plan.
struct LeanTune {
  int block = 0, rpt = 0, stages = 0, ctas = 0;
  int max_smem = 227 * 1024, sm_count = 148;
  bool interpreted = false;  // geometry for the ahead-of-time (interpreting) build: dispatch cost per instruction and tile
                             // is amortised over the rows per thread, so rows per thread weigh more than resident warps
  bool partition = false;    // partitioned high-cardinality GROUP BY: the scan emits tuples (LeanTile::scatter)
  // packed form of it (LeanTile::scatter_packed): one 64-bit tuple per row, partitions aggregated in shared memory
  const PackedLayout* packed = nullptr;
};

// The packed form needs: integer-packed keys narrower than 64 bits, after GROUP only COUNT / first row / SUMs whose
// operands are proven in [0, 2^32), and room for all of it plus >= 20 bits of launch-relative row in one 64-bit word.
// Returns the bits left for the row (0 = not eligible) and fills the operand widths.
static uint32_t packed_row_bits(const Plan& p, uint32_t* key_bits_out, uint32_t op_bits[8], uint32_t* n_ops_out) {
  if (p.n_keys == 0 || p.single_wide_key) return 0;
  uint32_t kb = 0;
  for (uint32_t k = 0; k < p.n_keys; ++k) kb += p.key_bits[k] + (p.key_nullable[k] ? 1u : 0u);
  if (kb == 0 || kb > 40) return 0;
  uint32_t used = kb, n_ops = 0;
  bool after_group = false;
  for (uint32_t i = 0; i < p.n_finstr; ++i) {
    const FInstr& in = p.fcode[i];
    if (in.op == FO_GROUP) { after_group = true; continue; }
    if (!after_group || in.op < FO_COUNT_STAR || in.op > FO_FIRSTNAN) continue;
    if (in.op == FO_COUNT_STAR || in.op == FO_COUNT || in.op == FO_FIRSTROW) continue;
    if (in.op != FO_SUM || in.g == 0 || in.g > 32 || n_ops >= 4) return 0;
    op_bits[n_ops++] = in.g;
    used += in.g;
  }
  if (used + 20 > 64) return 0;
  *key_bits_out = kb;
  *n_ops_out = n_ops;
  return std::min<uint32_t>(30u, 64u - used);
}

// A grouped lean plan can run partitioned when everything after GROUP is arithmetic plus aggregates whose row mask is the
// selection itself and whose update partition_apply_kernel knows (no NaN-dependent masks).
static bool partition_eligible(const Plan& p) {
  if (p.n_keys == 0) return false;
  bool after_group = false;
  uint32_t fields = 2;
  for (uint32_t i = 0; i < p.n_finstr; ++i) {
    const uint32_t op = p.fcode[i].op;
    if (op == FO_GROUP) {
      after_group = true;
      continue;
    }
    if (!after_group) continue;
    if (op == FO_LEAF || op == FO_MVCC || op == FO_SELECT_DONE || op == FO_MIN_F || op == FO_MAX_F || op == FO_FIRSTNAN || op == FO_VALID) return false;
    if (op >= FO_COUNT_STAR && op <= FO_FIRSTNAN && p.fcode[i].h) return false;  // (tuples carry no per-aggregate NULL mask)
    if (lean_takes_operand(op)) ++fields;
  }
  return after_group && fields <= 2 + (uint32_t)kMaxPartOperands;
}
// The packed form's partition layout; false when the plan or the hint rules the packed form out
static bool packed_layout(const Plan& p, u64 hint, u64 gcap, bool small_tables, PackedLayout& L) {
  L = PackedLayout();
  if (!hint) return false;
  L.row_bits = packed_row_bits(p, &L.key_bits, L.op_bits, &L.n_ops);
  if (!L.row_bits) return false;
  const u64 span = 1ull << L.key_bits;  // packed keys are < 2^key_bits (the column minimum is subtracted)
  uint32_t slots = L.n_ops <= 1 ? 8192u : 4096u;
  const bool dense = span <= std::max<u64>(hint * 4, 1ull << 16);
  u64 parts;
  uint32_t shift = 0;
  if (dense) {
    while (small_tables && slots > 256 && span / slots < 64) slots /= 2;  // (tests: small tables still get several partitions)
    while ((1u << shift) < slots) ++shift;
    parts = (span + slots - 1) / slots;
  } else {
    if (fold_smem_bytes(slots, L.n_ops, false) > 200u * 1024u) slots /= 2;
    while (small_tables && slots > 256 && hint * 2 / slots < 16) slots /= 2;
    parts = next_pow2(std::max<u64>(2, (hint * 2 + slots - 1) / slots));
    uint32_t cap_log2 = 0, bits = 0;
    while ((1ull << cap_log2) < gcap) ++cap_log2;
    while ((1ull << bits) < parts) ++bits;
    if (bits > cap_log2) return false;
    shift = cap_log2 - bits;
  }
  if (parts < 2 || parts > (u64)kMaxPackedPartitions || fold_smem_bytes(slots, L.n_ops, dense) > 200u * 1024u) return false;
  L.parts = (uint32_t)parts;
  L.shift = shift;
  L.slots = slots;
  L.dense = dense ? 1u : 0u;
  return true;
}

// The form policy of a grouped lean plan, for the runtime and for llkv_gpu_debug_plan alike: LEAN_PACKED (layout in L),
// LEAN_PARTITIONED, or LEAN_INTERPRETED when the plan keeps the per-row form.  Partitioning is worth two extra streaming
// passes over the tuples once the group table is far larger than L2 (every row is then a random DRAM read-modify-write);
// it needs the specialised kernel.  direct_global: that of the interpreted geometry (a hint above 128).
static LeanForm partition_form(const Plan& p, int partition_mode, int jit_mode, bool direct_global, u64 hint, u64 gcap, u64 rows,
                               PackedLayout& L) {
  if (!partition_mode || !jit_mode || !direct_global || !partition_eligible(p) || gcap < 64) return LEAN_INTERPRETED;
  const u64 table_bytes = gcap * (8ull + 8ull * p.n_gwords);
  const bool big = table_bytes > (64ull << 20) && rows >= (4ull << 20);
  if (!big && partition_mode < 2) return LEAN_INTERPRETED;
  // Packed form first: one 64-bit tuple per row into partitions of a few thousand groups, each aggregated in shared memory
  // by partition_fold_kernel.
  if (partition_mode != 3 && packed_layout(p, hint, gcap, partition_mode == 2, L)) return LEAN_PACKED;
  return LEAN_PARTITIONED;
}

constexpr u64 kStageBytes = 64u << 10;  // results up to this size travel to page-locked memory behind the scan
static u64 result_bytes(u64 gcap, uint32_t n_gwords, uint32_t n_keys) { return (gcap + 2) * n_gwords * 8 + (n_keys ? gcap * 8 : 0); }

// The step form of a run, for the runtime and for llkv_gpu_debug_plan alike: true when the scan publishes its result itself
// (LeanPlan::publish) and a repeated step is that one kernel.  It needs the lean plan in its per-row form, a result that fits
// the stage, group keys that need no pass over the table on the device (hashed wide keys are verified there), one rank, and
// a run that starts from the initial state (the kernel re-arms it).  Any other run is reset, scan and result copy.
static bool step_publishes(bool per_row_lean, u64 bytes, uint32_t single_wide_key, int n_ranks, bool from_reset) {
  return per_row_lean && bytes <= kStageBytes && single_wide_key != 2 && n_ranks == 1 && from_reset;
}

static int32_t lean_geometry(const LeanTune& tn, const Plan& p, uint64_t row_begin, uint64_t row_end, uint64_t hint, LeanPlan& lp, Geometry& g,
                             uint32_t* ctas_out) {
  memset(&lp, 0, sizeof(lp));
  LeanShape& s = lp.s;
  if (p.n_finstr > (uint32_t)kMaxFastInstr || p.n_lits > (uint32_t)kMaxLits || p.n_fast_words > (uint32_t)kLeanMaxWords)
    return set_error(LLKV_ERR_INTERNAL, "lean plan exceeds its limits");
  s.n_code = p.n_finstr;
  for (uint32_t i = 0; i < p.n_finstr; ++i) s.code[i] = p.fcode[i];
  for (uint32_t i = 0; i < p.n_lits; ++i) lp.lits[i] = (long long)p.lits[i].lo;
  s.n_cols = p.n_cols;
  bool any_bits = p.exists_bits != nullptr;
  for (uint32_t c = 0; c < p.n_cols; ++c) {
    lp.col_base[c] = p.cols[c].base;
    lp.col_valid[c] = p.cols[c].validity;
    s.cols[c].elem_bytes = p.cols[c].elem_bytes;
    s.cols[c].has_valid = p.cols[c].validity ? 1u : 0u;
    any_bits = any_bits || p.cols[c].validity;
  }
  lp.exists_bits = p.exists_bits;
  s.has_exists = p.exists_bits ? 1u : 0u;
  lp.txn_id = p.txn_id;
  lp.snapshot_id = p.snapshot_id;
  // TXN_ID_AUTO_COMMIT (1) is always committed (llkv-transaction/src/mvcc.rs:157-171): never listed for the kernel.
  // Neither are ids above the snapshot: a row created by one fails created_by <= snapshot whether or not the id is
  // listed, and a deletion by one passes deleted_by > snapshot either way.
  lp.n_noncommitted = 0;
  for (uint32_t i = 0; i < p.n_noncommitted; ++i)
    if (p.noncommitted[i] != 1ull && p.noncommitted[i] <= p.snapshot_id) lp.noncommitted[lp.n_noncommitted++] = p.noncommitted[i];
  s.n_keys = p.n_keys;
  s.single_wide_key = p.single_wide_key;
  for (int k = 0; k < kMaxKeys; ++k) {
    s.key_bits[k] = p.key_bits[k];
    s.key_kind[k] = p.key_kind[k];
    s.key_strlen[k] = p.key_strlen[k];
    s.key_col[k] = p.key_col[k];
    s.key_load[k] = p.key_load[k];
    s.key_nullable[k] = p.key_nullable[k];
    lp.key_min[k] = p.key_min[k];
  }
  s.n_words = p.n_fast_words;
  s.n_gwords = p.n_gwords;
  uint32_t thread_bytes = 0;  // accumulator bytes per consumer thread and slot
  for (uint32_t w = 0; w < p.n_fast_words; ++w) {
    s.words[w].kind = p.fast[w].kind;
    s.words[w].width = p.fast[w].kind == FK_SKIP ? 0 : (p.fast[w].lean_width == 4 ? 4 : 8);  // the low half of a 128-bit pair has no thread state
    s.words[w].rowrel = s.words[w].width == 4 ? p.fast[w].lean_rowrel : 0;
    s.words[w].gword = p.fast[w].gword;
    thread_bytes += s.words[w].width;
  }
  uint32_t NC = tn.block ? (uint32_t)tn.block : (tn.packed ? 512u : 128u);
  if (NC > (tn.packed ? 512u : 256u)) NC = tn.packed ? 512u : 256u;
  if (NC < 32) NC = 32;
  NC = NC / 32 * 32;
  // CTA-local group slots: every slot costs thread_bytes per consumer thread
  uint32_t FG = 1;
  if (p.n_keys) {
    if (hint == 0) FG = 8;
    else if (hint <= 16) FG = (uint32_t)std::max<u64>(4, next_pow2(hint));
    else if (hint <= 128) FG = 16;
    else {  // high cardinality: nearly every row goes to the global table anyway
      FG = 1;
      s.direct_global = 1;
    }
    if (tn.partition) {
      FG = 1;
      s.direct_global = 1;
      s.partition = 1;
      s.n_fields = 2;
      for (uint32_t i = 0; i < p.n_finstr; ++i)
        if (lean_takes_operand(p.fcode[i].op)) ++s.n_fields;
      if (tn.packed) {
        s.partition = 2;
        s.pack_key_bits = tn.packed->key_bits;
        s.pack_row_bits = tn.packed->row_bits;
        s.pack_parts = tn.packed->parts;
        for (int j = 0; j < 8; ++j) s.pack_op_bits[j] = tn.packed->op_bits[j];
      }
    }
    while (FG > 4 && (u64)FG * thread_bytes * NC > 64u * 1024u) FG /= 2;
  }
  const uint32_t budget_total = (uint32_t)tn.max_smem;
  uint32_t want_stages = tn.stages ? (uint32_t)tn.stages : 0u;
  if (want_stages == 1) want_stages = 2;
  const uint32_t want_ctas = tn.ctas ? (uint32_t)tn.ctas : 0u;
  uint32_t want_R = tn.rpt ? (uint32_t)tn.rpt : (tn.packed ? 2u : 0u);  // (packed: the shared memory goes to the batch buffer, not to tiles)

  // layout for one candidate geometry; returns the stages that fit (0 = does not fit)
  auto layout = [&](uint32_t R, uint32_t ctas, uint32_t fg, uint32_t nc) -> uint32_t {
    const uint32_t T = nc * R;
    uint32_t stage_bytes = 0, tx = 0;
    if (any_bits && (T % 128u)) return 0;  // bitmap tiles travel as bulk copies of T / 8 bytes: multiples of 16
    for (uint32_t c = 0; c < p.n_cols; ++c) {
      s.cols[c].smem_off = stage_bytes;
      stage_bytes += align_up(T * s.cols[c].elem_bytes, 128);
      tx += T * s.cols[c].elem_bytes;
      if (s.cols[c].has_valid) {
        s.cols[c].vsmem_off = stage_bytes;
        stage_bytes += align_up(T / 8, 128);
        tx += T / 8;
      }
    }
    if (s.has_exists) {
      s.exists_smem_off = stage_bytes;
      stage_bytes += align_up(T / 8, 128);
      tx += T / 8;
    }
    uint32_t woff = 0;
    for (uint32_t w = 0; w < s.n_words; ++w) {
      s.words[w].off = woff;
      woff += s.words[w].width * nc;
    }
    const uint32_t slot_stride = align_up(woff, 128);
    const uint32_t acc_bytes = align_up(fg * slot_stride, 128), tmp_bytes = align_up(p.fast_tmps * T * 8, 128), tbl_bytes = align_up(fg * 16, 128);
    uint32_t part_bytes = s.partition ? align_up(3u * (kMaxPartitions + 1) * 4 + 4 + s.n_fields * T * 8, 128) : 0;
    const uint32_t per_cta = budget_total / ctas - 1024;
    if (s.partition == 2) {  // fill word, counters and reserved bases per partition, then the batch buffer: as large as fits
      uint32_t B = 16384;
      if (const char* e = getenv("LLKV_GPU_PACK_BATCH")) B = (uint32_t)std::max<long>(2 * T, strtol(e, nullptr, 10));  // experiments
      for (; B >= 2 * T; B /= 2) {
        part_bytes = align_up(8u + 2u * s.pack_parts * 4u + B * 8u + B * 2u + 64u * 4u, 128);  // + sorted order (u16) + warp partial sums
        if (per_cta >= 128 + acc_bytes + tmp_bytes + tbl_bytes + part_bytes + 2 * stage_bytes) break;
      }
      if (B < 2 * T) return 0;
      s.pack_batch = B;
    }
    const uint32_t fixed = 128 /* barriers */ + acc_bytes + tmp_bytes + tbl_bytes + part_bytes;
    if (!stage_bytes || per_cta < fixed + 2 * stage_bytes) return 0;
    uint32_t st = (per_cta - fixed) / stage_bytes;
    if (want_stages) {
      if (st < want_stages) return 0;
      st = want_stages;
    } else {
      if (st > 4) st = 4;
      // More than ~160 KB of bulk copies in flight per SM buys nothing and costs DRAM efficiency (Q6 at SF10, tools/sweep_q6.py:
      // 4 CTAs x 3 stages x 16 KB = 192 KB in flight 0.155 ms; 4 x 2 x 16 KB 0.145 ms; 3 x 3 x 16 KB 0.144 ms; 4 x 4 x 8 KB 0.145 ms)
      while (st > 2 && (uint64_t)ctas * st * stage_bytes > 160u * 1024u) --st;
    }
    uint32_t off = 0;
    s.smem_bar_off = off;
    off += 128;
    s.smem_stage_off = off;
    off += stage_bytes * st;
    s.smem_acc_off = off;
    off += acc_bytes;
    s.smem_tmp_off = off;
    off += tmp_bytes;
    s.smem_tbl_off = off;
    off += tbl_bytes;
    s.smem_part_off = off;
    off += part_bytes;
    s.smem_total = off;
    s.nc = nc;
    s.rows_per_thread = R;
    s.fg = fg;
    s.slot_stride = slot_stride;
    s.tile_rows = T;
    s.stages = st;
    s.stage_bytes = stage_bytes;
    s.tx_bytes = tx;
    return st;
  };
  // Candidates: rows per thread x CTAs per SM, each with the deepest pipeline (2..4 stages) that fits.  The kernel is
  // latency-bound when its per-thread state is fat (Q1) and HBM-bound when it is thin (Q6), so the choice maximises
  // resident consumer warps (up to 16 per SM: Q1 still gains from 12 -> 16), then rows per thread (fewer
  // per-tile fixed costs), then stages.  One row per thread only when nothing else fits; then fewer CTA-local groups
  // and consumer threads.  Explicit tuning pins the corresponding dimension.
  uint32_t got_ctas = 0;
  for (uint32_t fg = FG, nc = NC; !got_ctas;) {
    uint32_t best_score = 0, best_R = 0, best_c = 0;
    const uint32_t Rs[4] = {8, 4, 2, 1};
    for (int ri = 0; ri < 4; ++ri) {
      if (want_R ? Rs[ri] != want_R : (Rs[ri] == 1 && best_score)) continue;
      // (packed: one CTA per SM, all of the shared memory for the batch buffer — what counts is the length of the sorted runs
      // a flush writes per partition: 16384 tuples over 1221 partitions measured 2.7 ms per 2^28 rows, 2 CTAs x 4096 5.7 ms)
      for (uint32_t ctas = tn.packed ? 1 : 4; ctas >= 1; --ctas) {
        const uint32_t c = want_ctas ? want_ctas : ctas;
        const uint32_t st = layout(Rs[ri], c, fg, nc);
        if (st >= 2) {
          const uint32_t warps = std::min<uint32_t>(c * (nc / 32), tn.interpreted ? 8 : 16);
          // (partitioned scans: rows per tile first — longer runs per partition, fewer barriers and reservations per row)
          const uint32_t score = tn.partition ? Rs[ri] * 100000u + warps * 1000 + st
                                 : tn.interpreted ? (Rs[ri] >= 4 ? 100000u : 0u) + warps * 1000 + Rs[ri] * 10 + st : warps * 1000 + Rs[ri] * 10 + st;
          if (score > best_score) { best_score = score; best_R = Rs[ri]; best_c = c; }
        }
        if (want_ctas) break;
      }
    }
    if (best_score) {
      layout(best_R, best_c, fg, nc);  // re-establish the winner's layout in `s`
      got_ctas = best_c;
      break;
    }
    // Nothing fits: fewer consumer threads first (their accumulators are the fat part), fewer CTA-local group slots last
    // — a group without a slot sends its rows to the global table one contended atomic at a time (Q1 with two slots for
    // its four groups: 2 ms instead of 0.035 ms per million rows, tools/tune_check.py).
    if (nc > 32) nc = nc > 64 ? (nc / 2 + 31) / 32 * 32 : 32;  // whole warps
    else if (p.n_keys && fg > 2) {
      fg /= 2;
      nc = NC;
    } else break;
  }
  if (got_ctas) {
    const uint32_t T = s.tile_rows;
    lp.row_begin = row_begin;
    lp.row_end = row_end;
    lp.first_tile = row_begin / T;
    lp.n_tiles = row_end > row_begin ? (row_end + T - 1) / T - lp.first_tile : 0;
    g.block = s.nc;
    g.R = s.rows_per_thread;
    g.smem = s.smem_total;
    g.grid = (uint32_t)((u64)tn.sm_count * got_ctas);  // persistent CTAs; a launch uses min(grid, tiles of its row range)
    *ctas_out = got_ctas;
    return LLKV_OK;
  }
  return set_error(LLKV_ERR_INVALID_ARGUMENT, "query state does not fit in shared memory on the lean path");
}

static LeanTune lean_tune(const llkv_gpu_ctx* ctx) {
  LeanTune t;
  t.block = ctx->tune_block;
  t.rpt = ctx->tune_rpt;
  t.stages = ctx->tune_stages;
  t.ctas = ctx->tune_ctas;
  t.max_smem = ctx->max_smem;
  t.sm_count = ctx->sm_count;
  return t;
}

static int32_t build_request(llkv_gpu_ctx* ctx, uint64_t table_id, const llkv_gpu_program* prog, int apply_mvcc, CompileRequest& req,
                             std::vector<llkv_gpu_column*>& handles, uint64_t* table_rows) {
  int32_t rc = collect_columns(ctx, table_id, req.cols, handles, table_rows);
  if (rc) return rc;
  req.prog = prog ? &prog->view : nullptr;
  req.mvcc = MvccView();
  if (apply_mvcc) {
    auto it = ctx->mvcc.find(table_id);
    // missing MVCC columns => every row is visible (llkv-transaction/src/helpers.rs:141-152)
    if (it != ctx->mvcc.end() && it->second.created_by && it->second.deleted_by) {
      const MvccState& m = it->second;
      for (size_t i = 0; i < handles.size(); ++i) {
        if (handles[i] == m.created_by) req.mvcc.created_by = &req.cols[i];
        if (handles[i] == m.deleted_by) req.mvcc.deleted_by = &req.cols[i];
      }
      if (!req.mvcc.created_by || !req.mvcc.deleted_by)
        return set_error(LLKV_ERR_INVALID_ARGUMENT, "MVCC columns of table %llu are not registered under that table id", (unsigned long long)table_id);
      req.mvcc.enabled = true;
      req.mvcc.txn_id = m.txn_id;
      req.mvcc.snapshot_id = m.snapshot_id;
      req.mvcc.noncommitted = m.noncommitted;
    }
  }
  return LLKV_OK;
}

// ------------------------------------------------------------------------------------------------ diagnostics
static const char* fast_op_name(uint32_t op) {
  static const char* names[] = {"END", "LEAF", "MVCC", "SELECT_DONE", "GROUP", "LD_COL", "LD_LIT", "LD_TMP", "ST_TMP", "OP_COL", "OP_LIT",
                                "OP_TMP", "DIVR", "MULP", "I2F", "D2F", "COUNT_STAR", "COUNT", "FIRSTROW", "SUM", "FSUM", "MIN_I", "MAX_I",
                                "MIN_F", "MAX_F", "FIRSTVALID", "FIRSTNAN", "VALID", "MASK_AND", "MASK_OR", "MASK_NOT", "MASK_LIT",
                                "MASK_FILTER", "CMP", "ISNULL"};
  return op < sizeof(names) / sizeof(names[0]) ? names[op] : "?";
}
static std::string lean_listing(const LeanPlan& lp, const Geometry& g, uint32_t ctas) {
  const LeanShape& s = lp.s;
  char b[256];
  std::string o;
  snprintf(b, sizeof(b), "lean plan: %u instr, %u cols, %u words, %u keys | NC=%u R=%u tile=%u stages=%u stage_bytes=%u fg=%u slot_stride=%u smem=%u ctas/SM=%u grid=%u\n",
           s.n_code, s.n_cols, s.n_words, s.n_keys, s.nc, s.rows_per_thread, s.tile_rows, s.stages, s.stage_bytes, s.fg, s.slot_stride, s.smem_total, ctas, g.grid);
  o += b;
  if (s.partition == 2) {
    snprintf(b, sizeof(b), "  partitioned, packed tuples: %u key bits | %u row bits | operands %u %u %u %u; %u partitions, batch of %u tuples at smem+%u\n",
             s.pack_key_bits, s.pack_row_bits, s.pack_op_bits[0], s.pack_op_bits[1], s.pack_op_bits[2], s.pack_op_bits[3], s.pack_parts, s.pack_batch,
             s.smem_part_off);
    o += b;
  } else if (s.partition) {
    snprintf(b, sizeof(b), "  partitioned: %u fields per tuple, staging at smem+%u\n", s.n_fields, s.smem_part_off);
    o += b;
  }
  for (uint32_t c = 0; c < s.n_cols; ++c) {
    snprintf(b, sizeof(b), "  col %u: %u B/row at stage+%u\n", c, s.cols[c].elem_bytes, s.cols[c].smem_off);
    o += b;
  }
  for (uint32_t w = 0; w < s.n_words; ++w) {
    snprintf(b, sizeof(b), "  word %u: kind %u width %u rowrel %u off %u -> gword %u\n", w, s.words[w].kind, s.words[w].width, s.words[w].rowrel, s.words[w].off,
             s.words[w].gword);
    o += b;
  }
  for (uint32_t i = 0; i < s.n_code; ++i) {
    const FInstr& in = s.code[i];
    snprintf(b, sizeof(b), "  %2u %-11s a=%u b=%u c=%u", i, fast_op_name(in.op), in.a, in.b, in.c);
    o += b;
    if (in.d) {
      snprintf(b, sizeof(b), "  [pre: %s %u kind %u]", in.d == 1 ? "lit" : in.d == 2 ? "col" : "tmp", in.e, in.f);
      o += b;
    }
    if (in.op == FO_LEAF) {
      if (in.g == 3) snprintf(b, sizeof(b), "  IN list of %u literals%s", in.f, in.e ? " (pushed)" : "");
      else snprintf(b, sizeof(b), "  range [%lld, %lld]%s%s", lp.lits[in.c], lp.lits[in.c + 1],
                    in.g == 1 ? " unsigned" : in.g == 2 ? " over the ordered image of the float bits" : "", in.e ? " (pushed)" : "");
      o += b;
    }
    if (in.op == FO_OP_LIT || in.op == FO_LD_LIT) {
      snprintf(b, sizeof(b), "  lit %lld", lp.lits[in.op == FO_OP_LIT ? in.c : in.e]);
      o += b;
    }
    o += "\n";
  }
  return o;
}

extern "C" int32_t llkv_gpu_debug_plan(const llkv_debug_column* cols, int32_t n_cols, const llkv_gpu_program* prog, int32_t created_by_col,
                                        int32_t deleted_by_col, uint64_t txn_id, uint64_t snapshot_id, const llkv_agg_spec* specs,
                                        int32_t n_aggs, const llkv_scalar_node* nodes, int32_t n_nodes, const uint64_t* group_key_fields,
                                        int32_t n_keys, int32_t expr_mode, uint64_t cardinality_hint, int32_t block_threads,
                                        int32_t rows_per_thread, int32_t stages, int32_t ctas_per_sm, int32_t jit, const char* cubin_path,
                                        char* out_text, uint64_t out_cap) {
  if (!cols || n_cols <= 0 || n_aggs < 0 || n_keys < 0 || n_keys > kMaxKeys) return set_error(LLKV_ERR_INVALID_ARGUMENT, "bad arguments");
  CompileRequest req;
  uint64_t rows = ~0ull;
  for (int i = 0; i < n_cols; ++i) {
    const llkv_debug_column& d = cols[i];
    ColumnMeta m;
    m.field_id = lfid_field(d.logical_field_id) | ((d.logical_field_id >> 48) << 48);
    m.type = d.prim_type;
    m.precision = d.precision;
    m.scale = d.scale;
    m.nullable = d.nullable != 0;
    if (m.nullable) m.dev_validity = reinterpret_cast<const unsigned char*>((uintptr_t)0x2000);  // never dereferenced here
    m.load_kind = device_load_kind(d.prim_type);
    m.elem_bytes = device_elem_bytes(d.prim_type);
    if (m.elem_bytes == 0) return set_error(LLKV_ERR_INVALID_ARGUMENT, "column type %d does not cross this boundary", d.prim_type);
    m.arrow_bytes = d.prim_type == LLKV_PT_UTF8 ? 4u + d.max_strlen : (uint32_t)prim_type_width(d.prim_type);
    if (d.prim_type == LLKV_PT_DECIMAL128 && d.dec_fits_i64) {  // as sealed: resident i64, or i32 when the statistics allow
      const bool fits32 = d.has_minmax && d.min_value >= (int64_t)INT32_MIN && d.max_value <= (int64_t)INT32_MAX;
      m.load_kind = fits32 ? LK_D32 : LK_D64;
      m.elem_bytes = fits32 ? 4 : 8;
    }
    if (d.prim_type == LLKV_PT_UTF8 && d.max_strlen == 1) {  // as sealed: one byte per row
      m.load_kind = LK_STR8;
      m.elem_bytes = 1;
    }
    m.dev_values = reinterpret_cast<const void*>((uintptr_t)0x1000);  // never dereferenced here
    m.n_rows = d.n_rows;
    m.dec_fits_i64 = d.dec_fits_i64 != 0;
    if (d.has_minmax) {
      m.has_minmax = true;
      m.min_bits = (uint64_t)d.min_value;
      m.max_bits = (uint64_t)d.max_value;
    }
    m.max_strlen = d.max_strlen;
    req.cols.push_back(m);
    rows = std::min<uint64_t>(rows, d.n_rows);
  }
  req.prog = prog ? &prog->view : nullptr;
  if (created_by_col >= 0 && deleted_by_col >= 0) {
    if (created_by_col >= n_cols || deleted_by_col >= n_cols) return set_error(LLKV_ERR_INVALID_ARGUMENT, "MVCC column index out of range");
    req.mvcc.enabled = true;
    req.mvcc.created_by = &req.cols[(size_t)created_by_col];
    req.mvcc.deleted_by = &req.cols[(size_t)deleted_by_col];
    req.mvcc.txn_id = txn_id;
    req.mvcc.snapshot_id = snapshot_id;
  }
  req.specs = specs;
  req.n_aggs = n_aggs;
  req.agg_nodes = nodes;
  req.n_agg_nodes = n_nodes;
  req.key_fields.assign(group_key_fields, group_key_fields + n_keys);
  req.expr_mode = expr_mode;
  CompileResult cr;
  int32_t rc = compile_plan(req, cr);
  if (rc) return set_error(rc, "%s", cr.error.c_str());
  std::string text;
  if (!cr.fast) {
    text = "general interpreter (no lean program)\n";
  } else {
    LeanTune tn;
    tn.block = block_threads;
    tn.rpt = rows_per_thread;
    tn.stages = stages;
    tn.ctas = ctas_per_sm;
    LeanPlan lp;
    Geometry g;
    uint32_t ctas = 1;
    if ((rc = lean_geometry(tn, cr.plan, 0, rows, cardinality_hint, lp, g, &ctas))) return rc;
    // jit bit 1: the partitioned form of a GROUP BY where the runtime would take it under partitioning mode 3; with bit 3,
    // under mode 2 (packed tuples when the plan allows them).  The listing describes the specialised form whether or not
    // bit 0 asks for its cubin.
    PackedLayout L;
    const int partition_mode = !(jit & 2) ? 0 : (jit & 8) ? 2 : 3;
    const LeanForm form = partition_form(cr.plan, partition_mode, 1, lp.s.direct_global, cardinality_hint, group_table_cap(cardinality_hint), rows, L);
    if (form != LEAN_INTERPRETED) {
      tn.partition = true;
      if (form == LEAN_PACKED) tn.packed = &L;
      if ((rc = lean_geometry(tn, cr.plan, 0, rows, cardinality_hint, lp, g, &ctas))) return rc;
    }
    lp.s.use_tile_list = (jit & 4) ? 1u : 0u;  // jit bit 2: the variant that walks a zone-map tile list
    text = lean_listing(lp, g, ctas);
    // jit bit 4: a run that continues from the previous one (no reset in between)
    const u64 gcap = cr.plan.n_keys ? group_table_cap(cardinality_hint) : 1;
    text += step_publishes(form == LEAN_INTERPRETED, result_bytes(gcap, cr.plan.n_gwords, cr.plan.n_keys), cr.plan.single_wide_key, 1, !(jit & 16))
                ? "step: one kernel, the scan publishes the result to page-locked memory and re-arms the state\n"
                : "step: reset, scan, result copy\n";
    if (jit & 1) {
      std::vector<char> cubin;
      std::string log;
      if (jit_compile_cubin(lp.s, (int)ctas, cubin, log) != 0) return set_error(LLKV_ERR_INTERNAL, "specialisation failed: %s", log.c_str());
      char b[128];
      snprintf(b, sizeof(b), "specialised cubin: %zu bytes\n", cubin.size());
      text += b;
      if (!log.empty()) text += "nvrtc log: " + log + "\n";
      if (cubin_path) {
        FILE* f = fopen(cubin_path, "wb");
        if (!f) return set_error(LLKV_ERR_IO, "cannot write %s", cubin_path);
        fwrite(cubin.data(), 1, cubin.size(), f);
        fclose(f);
      }
    }
  }
  if (out_text && out_cap) {
    const size_t n = std::min<size_t>(text.size(), (size_t)out_cap - 1);
    memcpy(out_text, text.data(), n);
    out_text[n] = 0;
  }
  return LLKV_OK;
}

// ------------------------------------------------------------------------------------------------ selection bitmap
extern "C" int32_t llkv_gpu_filter_bitmap(llkv_gpu_ctx* ctx, uint64_t table_id, const llkv_gpu_program* prog, int32_t apply_mvcc,
                                           uint64_t row_begin, uint64_t row_end, uint64_t* out_words, uint64_t n_words,
                                           uint64_t* out_count) {
  if (!ctx) return set_error(LLKV_ERR_INVALID_ARGUMENT, "ctx is NULL");
  if (row_end < row_begin) return set_error(LLKV_ERR_INVALID_ARGUMENT, "row_end < row_begin");
  CTX_LOCK(ctx);
  CUDA_TRY(cudaSetDevice(ctx->device));
  CompileRequest req;
  std::vector<llkv_gpu_column*> handles;
  uint64_t table_rows = 0;
  int32_t rc = build_request(ctx, table_id, prog, apply_mvcc, req, handles, &table_rows);
  if (rc) return rc;
  if (row_end > table_rows) return set_error(LLKV_ERR_INVALID_ARGUMENT, "row_end %llu beyond the table's %llu rows", (unsigned long long)row_end, (unsigned long long)table_rows);
  const uint64_t need_words = (row_end - row_begin + 63) / 64;
  if (out_words && n_words < need_words) return set_error(LLKV_ERR_INVALID_ARGUMENT, "bitmap buffer too small");
  req.bitmap_mode = true;
  req.force_wide = ctx->tune_force_wide == 1;
  const unsigned char* exists_bits = nullptr;
  if ((rc = table_exists_bits(ctx, table_id, handles, table_rows, &exists_bits))) return rc;
  u64* d_bits = nullptr;
  Plan* d_plan = nullptr;
  uint32_t* d_flags = nullptr;
  const uint64_t alloc_words = need_words + 2;
  CUDA_TRY(cudaMalloc((void**)&d_bits, (alloc_words + 1) * 8));
  CUDA_TRY(cudaMalloc((void**)&d_plan, sizeof(Plan)));
  CUDA_TRY(cudaMalloc((void**)&d_flags, 4));
  int32_t result = LLKV_OK;
  for (int pass = 0; pass < 2; ++pass) {
    CompileResult cr;
    if ((rc = compile_plan(req, cr))) { result = set_error(rc, "%s", cr.error.c_str()); break; }
    Geometry g;
    if ((rc = plan_geometry(ctx, cr.plan, cr.wide, row_begin, row_end, 0, g))) { result = rc; break; }
    cr.plan.exists_bits = exists_bits;
    cr.plan.out_bitmap = d_bits;
    cr.plan.out_count = d_bits + alloc_words;
    cr.plan.flags = d_flags;
    cr.plan.gcap = 1;
    cudaError_t e = cudaMemsetAsync(d_bits, 0, (alloc_words + 1) * 8, ctx->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(d_flags, 0, 4, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_plan, &cr.plan, sizeof(Plan), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess && cr.plan.n_tiles) e = launch_scan(d_plan, cr.wide, (int)g.R, g.grid, g.block, g.smem, ctx->stream);
    uint32_t flags = 0;
    if (e == cudaSuccess) e = cudaMemcpyAsync(&flags, d_flags, 4, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) { result = set_error(LLKV_ERR_IO, "CUDA error %s in filter_bitmap", cudaGetErrorString(e)); break; }
    if ((flags & FLAG_NARROW_FAIL) && !cr.wide) {
      req.force_wide = true;
      continue;
    }
    if (flags & FLAG_BAD_PLAN) { result = set_error(LLKV_ERR_INTERNAL, "device interpreter met an unknown instruction"); break; }
    if (flags & FLAG_DIV_ZERO) { result = set_error(LLKV_ERR_INTERNAL, "Divide by zero error"); break; }
    if (flags & FLAG_ARITH_OVERFLOW) { result = set_error(LLKV_ERR_INTERNAL, "Arithmetic overflow: Overflow happened in a predicate expression"); break; }
    if (flags & FLAG_EXACT_OVERFLOW) { result = set_error(LLKV_ERR_INVALID_ARGUMENT, "Decimal overflow in a predicate expression"); break; }
    if (out_words && need_words) {
      e = cudaMemcpy(out_words, d_bits, need_words * 8, cudaMemcpyDeviceToHost);
      if (e != cudaSuccess) { result = set_error(LLKV_ERR_IO, "CUDA error %s reading the bitmap", cudaGetErrorString(e)); break; }
    }
    if (out_count) {
      e = cudaMemcpy(out_count, d_bits + alloc_words, 8, cudaMemcpyDeviceToHost);
      if (e != cudaSuccess) { result = set_error(LLKV_ERR_IO, "CUDA error %s reading the count", cudaGetErrorString(e)); break; }
    }
    break;
  }
  cudaFree(d_bits);
  cudaFree(d_plan);
  cudaFree(d_flags);
  return result;
}

// ------------------------------------------------------------------------------------------------ aggregates
extern "C" int32_t llkv_gpu_agg_create(llkv_gpu_ctx* ctx, uint64_t table_id, const llkv_agg_spec* specs, int32_t n_aggs,
                                        const llkv_scalar_node* nodes, int32_t n_nodes, const uint64_t* group_key_fields,
                                        int32_t n_keys, int32_t expr_mode, uint64_t cardinality_hint, llkv_gpu_agg** out) {
  if (!ctx || !out) return set_error(LLKV_ERR_INVALID_ARGUMENT, "NULL argument");
  *out = nullptr;
  if (n_aggs < 0 || n_nodes < 0 || n_keys < 0 || (n_aggs && !specs) || (n_nodes && !nodes) || (n_keys && !group_key_fields))
    return set_error(LLKV_ERR_INVALID_ARGUMENT, "bad aggregate arguments");
  if (n_keys > kMaxKeys) return set_error(LLKV_ERR_INVALID_ARGUMENT, "too many GROUP BY keys (max %d)", kMaxKeys);
  if (expr_mode != LLKV_EXPR_ARROW && expr_mode != LLKV_EXPR_EXACT) return set_error(LLKV_ERR_INVALID_ARGUMENT, "bad expr_mode %d", expr_mode);
  int n_distinct = 0;
  uint64_t distinct_field = 0;
  for (int i = 0; i < n_aggs; ++i) {
    if (specs[i].expr_root >= n_nodes) return set_error(LLKV_ERR_INVALID_ARGUMENT, "aggregate %d: expression root out of range", i);
    if (specs[i].expr_root < 0 && specs[i].kind != LLKV_AGG_COUNT) return set_error(LLKV_ERR_INVALID_ARGUMENT, "aggregate %d needs an argument", i);
    if (!specs[i].distinct) continue;
    // DISTINCT (llkv-aggregate/src/lib.rs:103-204: CountDistinctColumn, Sum/Total/AvgDistinctInt64): ungrouped, over one bare
    // integer column, every aggregate of the query DISTINCT over that column
    const llkv_scalar_node* arg = specs[i].expr_root >= 0 ? &nodes[specs[i].expr_root] : nullptr;
    if (n_keys || !arg || arg->tag != LLKV_SE_COLUMN || (n_distinct && arg->field_id != distinct_field) ||
        !(specs[i].kind == LLKV_AGG_COUNT || specs[i].kind == LLKV_AGG_SUM || specs[i].kind == LLKV_AGG_TOTAL || specs[i].kind == LLKV_AGG_AVG))
      return set_error(LLKV_ERR_INVALID_ARGUMENT, "DISTINCT aggregates on this path: ungrouped COUNT / SUM / TOTAL / AVG over one integer column");
    distinct_field = arg->field_id;
    ++n_distinct;
  }
  if (n_distinct && n_distinct != n_aggs) return set_error(LLKV_ERR_INVALID_ARGUMENT, "DISTINCT and plain aggregates cannot share one fused scan on this path");
  CTX_LOCK(ctx);
  CUDA_TRY(cudaSetDevice(ctx->device));
  llkv_gpu_agg* a = new llkv_gpu_agg();
  a->ctx = ctx;
  a->table_id = table_id;
  a->specs.assign(specs, specs + n_aggs);
  a->nodes.assign(nodes, nodes + n_nodes);
  for (llkv_scalar_node& nd : a->nodes)
    if (nd.tag == LLKV_SE_LITERAL) own_string_literal(nd.literal, a->strings);
  a->keys.assign(group_key_fields, group_key_fields + n_keys);
  a->expr_mode = expr_mode;
  a->hint = cardinality_hint;
  memset(&a->info, 0, sizeof(a->info));
  cudaError_t e = cudaMalloc((void**)&a->d_flags, 8);  // [status word, ticket of a publishing scan]
  if (e == cudaSuccess) e = cudaMemset(a->d_flags, 0, 8);
  if (e == cudaSuccess) e = cudaMalloc((void**)&a->d_plan, sizeof(Plan));
  if (e == cudaSuccess) e = cudaHostAlloc((void**)&a->h_plan, sizeof(Plan), cudaHostAllocDefault);
  if (e == cudaSuccess) e = cudaHostAlloc((void**)&a->h_flags, 4, cudaHostAllocDefault);
  if (e != cudaSuccess) {
    llkv_gpu_agg_destroy(a);
    return set_error(LLKV_ERR_IO, "CUDA error %s allocating aggregate state", cudaGetErrorString(e));
  }
  *a->h_flags = 0;
  if (n_distinct) {  // the set of distinct values = the groups of GROUP BY <column> (COUNT(*) per value keeps the table's layout simple)
    llkv_agg_spec count_star;
    memset(&count_star, 0, sizeof(count_star));
    count_star.kind = LLKV_AGG_COUNT;
    count_star.expr_root = -1;
    count_star.data_type = LLKV_PT_INT64;
    const int32_t rc = llkv_gpu_agg_create(ctx, table_id, &count_star, 1, nullptr, 0, &distinct_field, 1, LLKV_EXPR_EXACT,
                                           cardinality_hint ? cardinality_hint : 1024, &a->inner);
    if (rc) {
      llkv_gpu_agg_destroy(a);
      return rc;
    }
  }
  *out = a;
  return LLKV_OK;
}

extern "C" int32_t llkv_gpu_agg_set_output(llkv_gpu_agg* a, const llkv_having_term* having, int32_t n_having, const llkv_order_key* order,
                                            int32_t n_order, uint64_t offset, uint64_t limit) {
  if (!a || n_having < 0 || n_order < 0 || (n_having && !having) || (n_order && !order)) return set_error(LLKV_ERR_INVALID_ARGUMENT, "bad output arguments");
  CTX_LOCK(a->ctx);
  const int32_t n_aggs = (int32_t)a->specs.size(), n_keys = (int32_t)a->keys.size();
  for (int i = 0; i < n_having; ++i)
    if (having[i].index < 0 || having[i].index >= (having[i].is_aggregate ? n_aggs : n_keys) || having[i].cmp_op < LLKV_CMP_EQ || having[i].cmp_op > LLKV_CMP_GE)
      return set_error(LLKV_ERR_INVALID_ARGUMENT, "HAVING term %d refers to output column %d", i, having[i].index);
  for (int i = 0; i < n_order; ++i)
    if (order[i].index < 0 || order[i].index >= (order[i].is_aggregate ? n_aggs : n_keys))
      return set_error(LLKV_ERR_INVALID_ARGUMENT, "ORDER BY key %d refers to output column %d", i, order[i].index);
  a->having.assign(having, having + n_having);
  for (llkv_having_term& t : a->having) own_string_literal(t.literal, a->strings);
  a->order.assign(order, order + n_order);
  a->out_offset = offset;
  a->out_limit = limit;
  return LLKV_OK;
}

extern "C" void llkv_gpu_agg_destroy(llkv_gpu_agg* a) {
  if (!a) return;
  CTX_LOCK(a->ctx);
  if (a->inner) llkv_gpu_agg_destroy(a->inner);
  a->inner = nullptr;
  cudaSetDevice(a->ctx->device);
  cudaStreamSynchronize(a->ctx->stream);
  if (a->d_gclass) cudaFree(a->d_gclass);
  if (a->gkeys) cudaFree(a->gkeys);
  if (a->gwords) cudaFree(a->gwords);
  if (a->bk_keys) cudaFree(a->bk_keys);
  if (a->bk_words) cudaFree(a->bk_words);
  if (a->mg_keys) cudaFree(a->mg_keys);
  if (a->mg_words) cudaFree(a->mg_words);
  if (a->mg_cap) cudaFree(a->mg_cap);
  if (a->mg_stats) cudaFree(a->mg_stats);
  if (a->part_out) cudaFree(a->part_out);
  if (a->part_cursor) cudaFree(a->part_cursor);
  if (a->d_tile_list) cudaFree(a->d_tile_list);
  if (a->stage_ev) cudaEventDestroy(a->stage_ev);
  if (a->graph_exec) cudaGraphExecDestroy(a->graph_exec);
  if (a->d_flags) cudaFree(a->d_flags);
  if (a->d_plan) cudaFree(a->d_plan);
  if (a->h_plan) cudaFreeHost(a->h_plan);
  if (a->h_flags) cudaFreeHost(a->h_flags);
  if (a->h_stage) cudaFreeHost(a->h_stage);
  if (a->h_pub) cudaFreeHost(a->h_pub);
  delete a;
}

static int32_t agg_alloc_table(llkv_gpu_agg* a, u64 gcap) {
  llkv_gpu_ctx* ctx = a->ctx;
  ++a->plan_epoch;
  const u64 rows = gcap + 2;
  CUDA_TRY(cudaMalloc((void**)&a->gkeys, gcap * 8));
  CUDA_TRY(cudaMalloc((void**)&a->gwords, rows * a->n_gwords * 8));
  a->gcap = gcap;
  CUDA_TRY(launch_init_table(a->gkeys, a->gwords, rows, a->n_gwords, a->d_gclass, ctx->stream));
  return LLKV_OK;
}

static int32_t agg_freeze_layout(llkv_gpu_agg* a, const CompileResult& cr) {
  const Plan& p = cr.plan;
  u64 cap = p.n_keys ? group_table_cap(a->hint) : 1;
  if (a->frozen) {
    if (p.n_gwords == a->n_gwords && memcmp(p.gword_class, a->gclass.data(), a->n_gwords) == 0) return LLKV_OK;
    // The layout follows facts of the request as well as the aggregates: a COUNT over a column that cannot hold NULLs is
    // the row count and has no word of its own, and appended or deleted rows can give a column NULLs.  A state that holds
    // nothing yet (armed: a reset or a new step) takes the new layout; a run cannot continue a state of the old one.
    if (!a->armed || a->in_capture)
      return set_error(LLKV_ERR_INVALID_ARGUMENT, "accumulator layout changed since the aggregate's state was started (a column gained "
                       "NULLs?): reset the aggregate before running over the changed table");
    llkv_gpu_ctx* ctx = a->ctx;
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));  // (queued launches may still read the old table or classes)
    CUDA_TRY(cudaFree(a->gkeys));
    CUDA_TRY(cudaFree(a->gwords));
    CUDA_TRY(cudaFree(a->d_gclass));
    if (a->bk_keys) CUDA_TRY(cudaFree(a->bk_keys));
    if (a->bk_words) CUDA_TRY(cudaFree(a->bk_words));
    a->gkeys = a->gwords = a->bk_keys = a->bk_words = nullptr;
    a->d_gclass = nullptr;
    a->bk_cap = 0;
    cap = a->gcap;  // (a table grown for this aggregate's groups keeps its size)
  }
  a->n_gwords = p.n_gwords;
  a->gclass.assign(p.gword_class, p.gword_class + p.n_gwords);
  CUDA_TRY(cudaMalloc((void**)&a->d_gclass, a->n_gwords ? a->n_gwords : 1));
  CUDA_TRY(cudaMemcpy(a->d_gclass, a->gclass.data(), a->n_gwords, cudaMemcpyHostToDevice));
  int32_t rc = agg_alloc_table(a, cap);
  if (rc) return rc;
  a->frozen = true;
  return LLKV_OK;
}

static int32_t agg_backup(llkv_gpu_agg* a) {
  llkv_gpu_ctx* ctx = a->ctx;
  if (a->bk_cap != a->gcap) {
    if (a->bk_keys) CUDA_TRY(cudaFree(a->bk_keys));
    if (a->bk_words) CUDA_TRY(cudaFree(a->bk_words));
    a->bk_keys = a->bk_words = nullptr;
    CUDA_TRY(cudaMalloc((void**)&a->bk_keys, a->gcap * 8));
    CUDA_TRY(cudaMalloc((void**)&a->bk_words, (a->gcap + 2) * a->n_gwords * 8));
    a->bk_cap = a->gcap;
  }
  CUDA_TRY(cudaMemcpyAsync(a->bk_keys, a->gkeys, a->gcap * 8, cudaMemcpyDeviceToDevice, ctx->stream));
  CUDA_TRY(cudaMemcpyAsync(a->bk_words, a->gwords, (a->gcap + 2) * a->n_gwords * 8, cudaMemcpyDeviceToDevice, ctx->stream));
  return LLKV_OK;
}
static int32_t agg_restore(llkv_gpu_agg* a) {
  llkv_gpu_ctx* ctx = a->ctx;
  a->armed = false;
  CUDA_TRY(cudaMemcpyAsync(a->gkeys, a->bk_keys, a->gcap * 8, cudaMemcpyDeviceToDevice, ctx->stream));
  CUDA_TRY(cudaMemcpyAsync(a->gwords, a->bk_words, (a->gcap + 2) * a->n_gwords * 8, cudaMemcpyDeviceToDevice, ctx->stream));
  return LLKV_OK;
}

// grows the global group table (x4) and rehashes the current contents into it
static int32_t agg_grow_table(llkv_gpu_agg* a) {
  llkv_gpu_ctx* ctx = a->ctx;
  u64* old_keys = a->gkeys;
  u64* old_words = a->gwords;
  const u64 old_cap = a->gcap;
  a->armed = false;
  a->gkeys = nullptr;
  a->gwords = nullptr;
  int32_t rc = agg_alloc_table(a, old_cap * 4);
  if (rc) return rc;
  Plan mp = a->cr.plan;
  mp.gkeys = a->gkeys;
  mp.gwords = a->gwords;
  mp.gcap = a->gcap;
  mp.flags = a->d_flags;
  CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  memcpy(a->h_plan, &mp, sizeof(Plan));
  CUDA_TRY(cudaMemcpyAsync(a->d_plan, a->h_plan, sizeof(Plan), cudaMemcpyHostToDevice, ctx->stream));
  CUDA_TRY(launch_merge_table(a->d_plan, old_keys, old_words, old_cap, ctx->stream));
  CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  CUDA_TRY(cudaFree(old_keys));
  CUDA_TRY(cudaFree(old_words));
  return LLKV_OK;
}

// Everything the compiled plan of a run depends on, folded into one word: the columns as the compiler sees them (device
// pointers, row counts, statistics), the predicate program, the snapshot, tuning.  A prepared aggregate that runs again
// over unchanged inputs reuses its lean plan instead of recompiling (the compile is ~20 us, a Q6 scan of SF10 240 us).
static uint64_t request_signature(const llkv_gpu_ctx* ctx, const CompileRequest& req, const llkv_gpu_program* prog, bool force_wide,
                                  const unsigned char* exists_bits) {
  uint64_t h = 0xcbf29ce484222325ull;
  h = fnv_pod(h, exists_bits);
  for (const ColumnMeta& c : req.cols) {
    h = fnv_pod(h, c.field_id);
    h = fnv_pod(h, c.type);
    h = fnv_pod(h, c.precision);
    h = fnv_pod(h, c.scale);
    h = fnv_pod(h, c.nullable);
    h = fnv_pod(h, c.load_kind);
    h = fnv_pod(h, c.elem_bytes);
    h = fnv_pod(h, c.dev_values);
    h = fnv_pod(h, c.dev_validity);
    h = fnv_pod(h, c.n_rows);
    h = fnv_pod(h, c.dec_fits_i64);
    h = fnv_pod(h, c.has_minmax);
    h = fnv_pod(h, c.min_bits);
    h = fnv_pod(h, c.max_bits);
    h = fnv_pod(h, c.max_strlen);
    h = fnv_pod(h, c.str_non_ascii);
    h = fnv_pod(h, c.dict_epoch);
    h = fnv_pod(h, (uint64_t)(c.dict_sorted ? c.dict_sorted->size() + 1 : 0));
  }
  if (prog) {
    h = fnv1a(h, prog->ops.data(), prog->ops.size() * sizeof(llkv_eval_op));
    h = fnv1a(h, prog->literals.data(), prog->literals.size() * sizeof(llkv_literal));
    if (prog->strings)  // (literals by reference hash as addresses above: their bytes decide)
      for (const std::string& x : *prog->strings) h = fnv1a(fnv_pod(h, x.size()), x.data(), x.size());
    h = fnv1a(h, prog->nodes.data(), prog->nodes.size() * sizeof(llkv_scalar_node));
    h = fnv1a(h, prog->list_roots.data(), prog->list_roots.size() * sizeof(int32_t));
  }
  h = fnv_pod(h, (int)(prog != nullptr));
  h = fnv_pod(h, req.mvcc.enabled);
  if (req.mvcc.enabled) {
    h = fnv_pod(h, (size_t)(req.mvcc.created_by - req.cols.data()));
    h = fnv_pod(h, (size_t)(req.mvcc.deleted_by - req.cols.data()));
    h = fnv_pod(h, req.mvcc.txn_id);
    h = fnv_pod(h, req.mvcc.snapshot_id);
    h = fnv1a(h, req.mvcc.noncommitted.data(), req.mvcc.noncommitted.size() * 8);
  }
  const int tune[6] = {ctx->tune_ctas, ctx->tune_block, ctx->tune_stages, ctx->tune_rpt, ctx->tune_force_wide, (int)force_wide};
  h = fnv1a(h, tune, sizeof(tune));
  return h ? h : 1;
}

// Multi-GPU GROUP BY over Utf8 keys: dictionary codes only merge if every rank codes alike.  When any rank holds a key
// column in dictionary form, every rank switches that column to dictionary form, the ranks exchange their entries
// (all-gather), intern what they did not have and re-rank (dict_seal): equal sets of strings give equal ranks everywhere.
// Collective; skipped (by all ranks alike) while nothing a plan depends on has changed since the last agreement.
static int32_t agree_dictionaries(llkv_gpu_ctx* ctx, llkv_gpu_agg* a, const std::vector<llkv_gpu_column*>& handles, bool* changed) {
  *changed = false;
  std::vector<llkv_gpu_column*> cols;
  for (uint64_t f : a->keys)
    for (llkv_gpu_column* h : handles)
      if (lfid_field(h->lfid) == f && h->type == LLKV_PT_UTF8) cols.push_back(h);
  if (cols.empty() || a->in_rerun || a->dict_agreed_epoch == ctx->state_epoch) return LLKV_OK;
  const int N = ctx->n_ranks;
  cudaStream_t s = ctx->stream;
  std::vector<u64> v(cols.size());
  u64* d_v = nullptr;
  CUDA_TRY(cudaMalloc((void**)&d_v, v.size() * 8));
  auto all_max = [&]() -> int32_t {
    CUDA_TRY(cudaMemcpyAsync(d_v, v.data(), v.size() * 8, cudaMemcpyHostToDevice, s));
    NCCL_TRY(g_nccl.all_reduce(d_v, d_v, v.size(), 5 /* ncclUint64 */, 2 /* ncclMax */, ctx->nccl_comm, s));
    CUDA_TRY(cudaMemcpyAsync(v.data(), d_v, v.size() * 8, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    return LLKV_OK;
  };
  int32_t rc = LLKV_OK;
  for (size_t i = 0; i < cols.size(); ++i) v[i] = cols[i]->dict ? 1 : 0;
  if ((rc = all_max())) { cudaFree(d_v); return rc; }
  std::vector<char> coded(cols.size());
  bool any = false;
  for (size_t i = 0; i < cols.size() && !rc; ++i) {
    coded[i] = v[i] != 0;
    if (!coded[i]) continue;
    any = true;
    llkv_gpu_column* col = cols[i];
    if (!col->dict) {  // this rank's shard has short strings only: into dictionary form like the others
      if ((rc = column_flush(col))) break;
      if (col->load_kind == LK_STR8 && (rc = widen_str8(col))) break;
      if ((rc = enter_dict_mode(col))) break;
      *changed = true;
    }
  }
  if (!rc && any) {
    // entries as [u32 length][bytes]..., padded to the longest rank's size
    std::vector<std::string> blob(cols.size());
    for (size_t i = 0; i < cols.size(); ++i) {
      v[i] = 0;
      if (!coded[i]) continue;
      for (const std::string& e : cols[i]->dict->strings) {
        const uint32_t len = (uint32_t)e.size();
        blob[i].append(reinterpret_cast<const char*>(&len), 4);
        blob[i].append(e);
      }
      v[i] = blob[i].size();
    }
    rc = all_max();
    for (size_t i = 0; i < cols.size() && !rc; ++i) {
      if (!coded[i]) continue;
      const size_t slot = (size_t)((v[i] + 8 + 7) / 8 * 8);  // [u64 bytes][entries...]
      std::vector<char> mine(slot, 0), all(slot * (size_t)N);
      const u64 bytes = blob[i].size();
      memcpy(mine.data(), &bytes, 8);
      memcpy(mine.data() + 8, blob[i].data(), blob[i].size());
      char *d_mine = nullptr, *d_all = nullptr;
      CUDA_TRY(cudaMalloc((void**)&d_mine, slot));
      CUDA_TRY(cudaMalloc((void**)&d_all, slot * (size_t)N));
      CUDA_TRY(cudaMemcpyAsync(d_mine, mine.data(), slot, cudaMemcpyHostToDevice, s));
      NCCL_TRY(g_nccl.all_gather(d_mine, d_all, slot, 0 /* ncclInt8 */, ctx->nccl_comm, s));
      CUDA_TRY(cudaMemcpyAsync(all.data(), d_all, slot * (size_t)N, cudaMemcpyDeviceToHost, s));
      CUDA_TRY(cudaStreamSynchronize(s));
      CUDA_TRY(cudaFree(d_mine));
      CUDA_TRY(cudaFree(d_all));
      StrDict& d = *cols[i]->dict;
      const size_t before = d.strings.size();
      for (int r = 0; r < N; ++r) {
        const char* p = all.data() + slot * (size_t)r;
        u64 n;
        memcpy(&n, p, 8);
        for (u64 at = 0; at + 4 <= n;) {
          uint32_t len;
          memcpy(&len, p + 8 + at, 4);
          d.intern(p + 8 + at + 4, len);
          at += 4 + len;
        }
      }
      if (d.strings.size() > kMaxDictEntries) rc = set_error(LLKV_ERR_INVALID_ARGUMENT, "more than %zu distinct strings in a dictionary-coded column", kMaxDictEntries);
      if (!rc && (d.strings.size() != before || d.strings.size() != d.sealed)) {
        rc = dict_seal(cols[i]);
        ++cols[i]->version;
        ++ctx->state_epoch;
        *changed = true;
      }
    }
  }
  cudaFree(d_v);
  if (any) a->agreed_epoch = ~0ull;  // every rank agrees the key statistics again (a rank-invariant decision: `any` is)
  if (!rc) a->dict_agreed_epoch = ctx->state_epoch;
  return rc;
}

static int32_t agree_key_stats(llkv_gpu_ctx* ctx, llkv_gpu_agg* a, CompileRequest& req) {
  const size_t nk = a->keys.size();
  std::vector<u64> v(nk * 4);
  std::vector<int> col_of(nk, -1);
  const u64 sign = 0x8000000000000000ull;
  for (size_t k = 0; k < nk; ++k) {
    for (size_t i = 0; i < req.cols.size(); ++i)
      if (req.cols[i].field_id == a->keys[k]) col_of[k] = (int)i;
    if (col_of[k] < 0) return set_error(LLKV_ERR_NOT_FOUND, "unknown GROUP BY field %llu", (unsigned long long)a->keys[k]);
    const ColumnMeta& c = req.cols[(size_t)col_of[k]];
    const bool is_signed = c.type == LLKV_PT_INT8 || c.type == LLKV_PT_INT16 || c.type == LLKV_PT_INT32 || c.type == LLKV_PT_INT64 ||
                           c.type == LLKV_PT_DATE32 || c.type == LLKV_PT_DATE64;
    const u64 flip = is_signed ? sign : 0;
    // all four lanes reduce with MIN: maxima and lengths travel complemented
    v[4 * k + 0] = c.has_minmax ? (c.min_bits ^ flip) : ~0ull;
    v[4 * k + 1] = c.has_minmax ? ~(c.max_bits ^ flip) : ~0ull;
    v[4 * k + 2] = ~(u64)c.max_strlen;
    v[4 * k + 3] = (c.has_minmax || c.n_rows == 0) ? 1 : 0;  // an empty shard does not veto the statistics of the others
  }
  if ((a->in_rerun || a->agreed_epoch == ctx->state_epoch) && a->agreed_stats.size() == v.size()) {
    // a rerun (wider interpreter, larger table) is this rank's own business: no collective, the agreed values again.
    // Likewise when nothing a plan depends on has changed since the ranks last agreed (ranks issue the same calls on
    // their handles, so they all skip the collective together).
    v = a->agreed_stats;
  } else {
  if (a->mg_stats_elems < v.size()) {
    if (a->mg_stats) CUDA_TRY(cudaFree(a->mg_stats));
    CUDA_TRY(cudaMalloc((void**)&a->mg_stats, v.size() * 8));
    a->mg_stats_elems = v.size();
  }
  CUDA_TRY(cudaMemcpyAsync(a->mg_stats, v.data(), v.size() * 8, cudaMemcpyHostToDevice, ctx->stream));
  NCCL_TRY(g_nccl.all_reduce(a->mg_stats, a->mg_stats, v.size(), 5 /* ncclUint64 */, 3 /* ncclMin */, ctx->nccl_comm, ctx->stream));
  CUDA_TRY(cudaMemcpyAsync(v.data(), a->mg_stats, v.size() * 8, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  a->agreed_stats = v;
  a->agreed_epoch = ctx->state_epoch;
  }
  for (size_t k = 0; k < nk; ++k) {
    ColumnMeta& c = req.cols[(size_t)col_of[k]];
    const bool is_signed = c.type == LLKV_PT_INT8 || c.type == LLKV_PT_INT16 || c.type == LLKV_PT_INT32 || c.type == LLKV_PT_INT64 ||
                           c.type == LLKV_PT_DATE32 || c.type == LLKV_PT_DATE64;
    const u64 flip = is_signed ? sign : 0;
    const bool all_have = v[4 * k + 3] != 0 && v[4 * k + 0] != ~0ull;
    if (all_have) {
      c.has_minmax = true;
      c.min_bits = v[4 * k + 0] ^ flip;
      c.max_bits = (~v[4 * k + 1]) ^ flip;
    } else {
      c.has_minmax = false;
    }
    c.max_strlen = (uint8_t)(~v[4 * k + 2]);
  }
  return LLKV_OK;
}

// Queues, behind whatever the stream holds, the copy of the device status word and — for small tables (an ungrouped state
// row, Q1's 32 rows) — of the table itself into page-locked memory: finalize then needs the one synchronisation that
// settles the run and no copy of its own.  Called after the scan and again after a merge that was queued behind it.
static int32_t agg_queue_result_copy(llkv_gpu_agg* a) {
  llkv_gpu_ctx* ctx = a->ctx;
  CUDA_TRY(cudaMemcpyAsync(a->h_flags, a->d_flags, 4, cudaMemcpyDeviceToHost, ctx->stream));
  a->prefetched = false;
  const size_t wbytes = (size_t)(a->gcap + 2) * a->n_gwords * 8, kbytes = a->cr.plan.n_keys ? (size_t)a->gcap * 8 : 0;
  if (wbytes + kbytes > kStageBytes) return LLKV_OK;
  if (a->h_stage_bytes < wbytes + kbytes) {
    if (a->h_stage) CUDA_TRY(cudaFreeHost(a->h_stage));
    a->h_stage = nullptr;
    a->h_stage_bytes = 0;
    CUDA_TRY(cudaHostAlloc((void**)&a->h_stage, kStageBytes, cudaHostAllocDefault));
    a->h_stage_bytes = kStageBytes;
  }
  CUDA_TRY(cudaMemcpyAsync(a->h_stage, a->gwords, wbytes, cudaMemcpyDeviceToHost, ctx->stream));
  if (kbytes) CUDA_TRY(cudaMemcpyAsync(a->h_stage + wbytes, a->gkeys, kbytes, cudaMemcpyDeviceToHost, ctx->stream));
  if (!a->stage_ev) CUDA_TRY(cudaEventCreateWithFlags(&a->stage_ev, cudaEventDisableTiming));
  CUDA_TRY(cudaEventRecord(a->stage_ev, ctx->stream));
  a->stage_ev_valid = true;
  a->prefetched = true;
  return LLKV_OK;
}

// What agg_launch settles for one run before its launch loop
struct RunLaunches {
  Geometry g;
  uint32_t lean_ctas = 1;
  bool use_jit = false;
  u64 max_rows = 0;    // rows per launch
  PartPlan pp;         // partitioned form: the partition_apply pass behind every scan launch
  FoldPlan fp;         // packed form: the partition_fold pass behind every scan launch
  uint32_t part_grid = 0;
  bool use_tile_list = false;
  bool publish = false;  // step_publishes: the last launch publishes the result and re-arms the state
};

// Compiles the request and freezes the accumulator layout, unless the lean plan of the previous run still applies
// (request_signature() unchanged).  A plan for the general interpreter gets its geometry here.
static int32_t agg_compile(llkv_gpu_agg* a, CompileRequest& req, uint64_t sig, bool force_wide, uint64_t row_begin, uint64_t row_end,
                           Geometry& g) {
  llkv_gpu_ctx* ctx = a->ctx;
  if (a->lean_sig == sig && a->cr.fast && a->frozen) return LLKV_OK;
  a->lean_sig = 0;
  a->lean_jit_runs = 0;
  a->forget_forms();
  req.specs = a->specs.data();
  req.n_aggs = (int32_t)a->specs.size();
  req.agg_nodes = a->nodes.data();
  req.n_agg_nodes = (int32_t)a->nodes.size();
  req.key_fields = a->keys;
  req.expr_mode = a->expr_mode;
  req.force_wide = force_wide || ctx->tune_force_wide == 1;
  req.no_fast = ctx->tune_force_wide != 0;
  int32_t rc;
  if ((rc = compile_plan(req, a->cr))) return set_error(rc, "%s", a->cr.error.c_str());
  if ((rc = agg_freeze_layout(a, a->cr))) return rc;
  if (a->cr.fast) a->lean_sig = sig;
  else if ((rc = plan_geometry(ctx, a->cr.plan, a->cr.wide, row_begin, row_end, a->hint, g))) return rc;
  return LLKV_OK;
}

// The geometry of one form of the current lean plan, computed the first time a run asks for it
static int32_t agg_form_geometry(llkv_gpu_agg* a, LeanForm form, uint64_t row_begin, uint64_t row_end) {
  LeanFormGeometry& f = a->forms[form];
  if (f.have) return LLKV_OK;
  LeanTune tn = lean_tune(a->ctx);
  tn.interpreted = form == LEAN_INTERPRETED;
  tn.partition = form >= LEAN_PARTITIONED;
  if (form == LEAN_PACKED) tn.packed = &a->packed;
  Geometry g;
  // (a hint below the number of groups already seen would leave groups without a CTA-local slot: every row of such a
  // group is a contended atomic on the global table)
  const uint64_t hint_eff = a->hint && a->observed_groups > a->hint ? a->observed_groups : a->hint;
  int32_t rc = lean_geometry(tn, a->cr.plan, row_begin, row_end, hint_eff, f.plan, g, &f.ctas);
  if (rc) return rc;
  f.grid = g.grid;
  f.have = true;
  return LLKV_OK;
}

// Chooses the form the lean plan runs in and leaves it in a->lean.  A shape is specialised once it repeats (jit_mode 1),
// always (2) or never (0); runs are counted on the interpreted shape.  A partitioned form (partition_form) is taken when its
// specialised kernel is ready, the packed one first.
static int32_t agg_choose_form(llkv_gpu_agg* a, uint64_t row_begin, uint64_t row_end, RunLaunches& r) {
  llkv_gpu_ctx* ctx = a->ctx;
  int32_t rc;
  if ((rc = agg_form_geometry(a, LEAN_INTERPRETED, row_begin, row_end))) return rc;
  if (ctx->jit_mode == 2) r.use_jit = true;
  else if (ctx->jit_mode == 1) {
    if (a->lean_jit_runs < 2) {
      const std::string key(reinterpret_cast<const char*>(&a->forms[LEAN_INTERPRETED].plan.s), sizeof(LeanShape));
      a->lean_jit_runs = ++ctx->shape_runs[key];
    }
    r.use_jit = a->lean_jit_runs >= 2;
  }
  LeanForm form = r.use_jit ? LEAN_SPECIALISED : LEAN_INTERPRETED;
  PackedLayout L;
  const LeanForm part = partition_form(a->cr.plan, ctx->partition_mode, ctx->jit_mode, a->forms[LEAN_INTERPRETED].plan.s.direct_global,
                                       a->hint, a->gcap, row_end - row_begin, L);
  auto ready = [&](LeanForm f) { return jit_ready(ctx->device, a->forms[f].plan, (int)a->forms[f].ctas); };
  if (part == LEAN_PACKED) {
    if (memcmp(&a->packed, &L, sizeof(L)) != 0) a->forms[LEAN_PACKED].have = false;
    a->packed = L;
    if (agg_form_geometry(a, LEAN_PACKED, row_begin, row_end) == LLKV_OK && ready(LEAN_PACKED)) form = LEAN_PACKED;
  }
  if (part != LEAN_INTERPRETED && form != LEAN_PACKED) {
    if ((rc = agg_form_geometry(a, LEAN_PARTITIONED, row_begin, row_end))) return rc;
    if (ready(LEAN_PARTITIONED)) form = LEAN_PARTITIONED;
  }
  if (form >= LEAN_PARTITIONED) r.use_jit = true;
  if ((rc = agg_form_geometry(a, form, row_begin, row_end))) return rc;
  const LeanFormGeometry& f = a->forms[form];
  LeanPlan& lean = a->lean;
  lean = f.plan;
  r.lean_ctas = f.ctas;
  r.g.grid = f.grid;
  r.g.block = lean.s.nc;
  r.g.R = lean.s.rows_per_thread;
  r.g.smem = lean.s.smem_total;
  Plan& p = a->cr.plan;
  p.tile_rows = lean.s.tile_rows;
  p.stages = lean.s.stages;
  p.fast_groups = lean.s.fg;
  return LLKV_OK;
}

// Points the run's plan at the aggregate's table and status word.  First-row words hold row ids (position + the row id of
// position 0), so shards of one table uploaded with their own row_id_base merge into the table's first-appearance order.
static int32_t agg_bind_state(llkv_gpu_agg* a, const std::vector<llkv_gpu_column*>& handles) {
  uint64_t row_origin = 0;
  for (size_t i = 0; i < handles.size(); ++i) {
    if (!handles[i]->has_origin) continue;
    if (i && handles[0]->has_origin && handles[i]->row_id_origin != handles[0]->row_id_origin)
      return set_error(LLKV_ERR_INVALID_ARGUMENT, "columns of table %llu start at different row ids (%llu vs %llu)", (unsigned long long)a->table_id,
                       (unsigned long long)handles[i]->row_id_origin, (unsigned long long)handles[0]->row_id_origin);
    row_origin = handles[i]->row_id_origin;
  }
  Plan& p = a->cr.plan;
  LeanPlan& lean = a->lean;
  p.row_origin = row_origin;
  lean.row_origin = row_origin;
  p.gkeys = a->gkeys;
  p.gwords = a->gwords;
  p.gcap = a->gcap;
  p.flags = a->d_flags;
  lean.gkeys = a->gkeys;
  lean.gwords = a->gwords;
  lean.gcap = a->gcap;
  lean.flags = a->d_flags;
  return LLKV_OK;
}

// The tuple partitions of a partitioned scan, in either form: sizes the launches (max_rows), and the capacity of a partition
// as the uniform share of a launch's rows over `share` partitions + 25 %, of which `words` x part_cap fill part_out.
// batch_rows: the longest launch.  LLKV_GPU_PART_BATCH_ROWS (tests: several launches on small tables) caps it when
// env_caps, else replaces it.
static int32_t agg_part_buffers(llkv_gpu_agg* a, u64 batch_rows, bool env_caps, u64 share, u64 words, u64 rows, u64& max_rows) {
  const u64 T = a->cr.plan.tile_rows;
  if (const char* e = getenv("LLKV_GPU_PART_BATCH_ROWS")) {
    const u64 v = std::max<u64>(T, strtoull(e, nullptr, 10));
    batch_rows = env_caps ? std::min<u64>(batch_rows, v) : v;
  }
  const u64 dense_max_rows = max_rows;
  u64 part_cap = 0;
  for (;;) {  // the tuple buffer of one launch; when HBM is short the launches get smaller instead
    max_rows = std::max<u64>(T, std::min<u64>(dense_max_rows, batch_rows) / T * T);
    const u64 launch_rows = std::min<u64>(rows + T, max_rows);
    part_cap = (launch_rows / share + launch_rows / (4 * share) + 1024 + 15) / 16 * 16;
    const size_t elems = (size_t)(words * part_cap);
    if (a->part_out_elems >= elems) break;
    if (a->part_out) CUDA_TRY(cudaFree(a->part_out));
    a->part_out = nullptr;
    a->part_out_elems = 0;
    if (cudaMalloc((void**)&a->part_out, elems * 8) == cudaSuccess) {
      a->part_out_elems = elems;
      break;
    }
    cudaGetLastError();
    a->part_out = nullptr;
    if (batch_rows <= (1ull << 22)) return set_error(LLKV_ERR_IO, "out of device memory for the tuple partitions of a GROUP BY (%zu bytes)", elems * 8);
    batch_rows >>= 1;
  }
  if (!a->part_cursor) CUDA_TRY(cudaMalloc((void**)&a->part_cursor, kMaxPackedPartitions * 4));
  a->lean.part_out = a->part_out;
  a->lean.part_cursor = a->part_cursor;
  a->lean.part_cap = part_cap;
  return LLKV_OK;
}

// The fold pass of the packed form
static FoldPlan fold_plan(const llkv_gpu_agg* a) {
  const LeanPlan& lean = a->lean;
  FoldPlan fp{};
  fp.tuples = a->part_out;
  fp.cursor = a->part_cursor;
  fp.part_cap = lean.part_cap;
  fp.gkeys = a->gkeys;
  fp.gwords = a->gwords;
  fp.gcap = a->gcap;
  fp.flags = a->d_flags;
  fp.n_parts = a->packed.parts;
  fp.n_gwords = lean.s.n_gwords;
  fp.n_keys = lean.s.n_keys;
  fp.key_bits = a->packed.key_bits;
  fp.row_bits = a->packed.row_bits;
  fp.dense = a->packed.dense;
  fp.part_shift = a->packed.shift;
  fp.slots = a->packed.slots;
  fp.first_gword = ~0u;
  for (uint32_t i = 0; i < lean.s.n_code; ++i) {  // operands in the order of the aggregates (lean_field_index)
    const FInstr& in = lean.s.code[i];
    if (in.op == FO_COUNT_STAR || in.op == FO_COUNT) fp.count_gword[fp.n_counts++] = in.c;
    else if (in.op == FO_FIRSTROW) fp.first_gword = in.c;
    else if (in.op == FO_SUM) {
      fp.op_bits[fp.n_ops] = in.g;
      fp.op_gword[fp.n_ops] = in.c;
      fp.op_wide[fp.n_ops] = (in.a & 0x80) ? 1u : 0u;
      ++fp.n_ops;
    }
  }
  return fp;
}

// The apply pass of the partitioned form (multi-field tuples)
static PartPlan part_plan(const llkv_gpu_agg* a, uint32_t n_parts) {
  const LeanPlan& lean = a->lean;
  PartPlan pp{};
  pp.tuples = a->part_out;
  pp.cursor = a->part_cursor;
  pp.part_cap = lean.part_cap;
  pp.gkeys = a->gkeys;
  pp.gwords = a->gwords;
  pp.gcap = a->gcap;
  pp.flags = a->d_flags;
  pp.n_parts = n_parts;
  pp.n_fields = lean.s.n_fields;
  pp.n_keys = lean.s.n_keys;
  pp.n_gwords = lean.s.n_gwords;
  pp.chunk = 2048;
  pp.chunks_per_part = (uint32_t)((lean.part_cap + pp.chunk - 1) / pp.chunk);
  for (uint32_t i = 0; i < lean.s.n_code; ++i) {  // operand fields follow the order of the aggregates (lean_field_index)
    const FInstr& in = lean.s.code[i];
    if (in.op < FO_COUNT_STAR || in.op > FO_FIRSTNAN) continue;
    PartOp& o = lean_takes_operand(in.op) ? pp.vops[pp.n_vops++] : pp.nops[pp.n_nops++];
    o.op = in.op;
    o.flags = in.a;
    o.gword = in.c;
  }
  return pp;
}

// Partitioned GROUP BY: the tuple partitions and the second pass of the chosen form.  Packed tuples go to partitions of a
// few thousand groups (PackedLayout).  Multi-field tuples go to 2^bits hash partitions, each a contiguous slice of the table
// of about 24 MB (keys + words) so a slice and the tuple stream share L2 comfortably.  A launch covers at most 2^28 rows
// so the tuple buffers stay bounded; a partition that fills up (skewed keys) hands its surplus rows to the per-row path
// inside the scan, so no rerun is ever needed.
static int32_t agg_partitions(llkv_gpu_agg* a, const CompileRequest& req, uint64_t row_begin, uint64_t row_end, RunLaunches& r) {
  llkv_gpu_ctx* ctx = a->ctx;
  const Plan& p = a->cr.plan;
  LeanPlan& lean = a->lean;
  const uint32_t partition = a->cr.fast ? lean.s.partition : 0;
  a->info.partitions = 0;
  a->info.packed_tuples = 0;
  int32_t rc;
  if (partition == 2) {
    // partitions that can hold keys: all of them for hash ranges; for key ranges those below the largest packed key
    u64 used = a->packed.parts;
    if (a->packed.dense && p.n_keys == 1 && p.key_kind[0] == KK_INT) {
      for (const ColumnMeta& c : req.cols)
        if (c.field_id == a->keys[0] && c.has_minmax) {
          const u64 kmax = c.max_bits - c.min_bits;  // (two's complement difference: also right for signed columns)
          used = std::min<u64>(used, (kmax >> a->packed.shift) + 1);
        }
    }
    if ((rc = agg_part_buffers(a, 1ull << a->packed.row_bits, true, used, a->packed.parts, row_end - row_begin, r.max_rows))) return rc;
    lean.part_bits = 0;
    lean.part_shift = a->packed.shift;
    lean.part_dense = a->packed.dense;
    r.fp = fold_plan(a);
    r.part_grid = (uint32_t)std::min<u64>((u64)ctx->sm_count, used);
    a->info.partitions = (uint32_t)used;
    a->info.packed_tuples = 1 + a->packed.dense;
  } else if (partition) {
    const u64 table_bytes = a->gcap * (8ull + 8ull * a->n_gwords);
    uint32_t cap_log2 = 0;
    while ((1ull << cap_log2) < a->gcap) ++cap_log2;
    uint32_t bits = 1;
    u64 slice_mb = 24;
    if (const char* e = getenv("LLKV_GPU_PART_SLICE_MB")) slice_mb = std::max<u64>(1, strtoull(e, nullptr, 10));  // experiments
    while (bits < 8 && (table_bytes >> bits) > (slice_mb << 20)) ++bits;
    if (bits + 3 > cap_log2) bits = cap_log2 > 3 ? cap_log2 - 3 : 1;
    const u64 P = 1ull << bits;
    if ((rc = agg_part_buffers(a, 1ull << 28, false, P, P * lean.s.n_fields, row_end - row_begin, r.max_rows))) return rc;
    lean.part_bits = bits;
    lean.part_shift = cap_log2 - bits;
    r.pp = part_plan(a, (uint32_t)P);
    r.part_grid = (uint32_t)ctx->sm_count;  // launch_partition_apply multiplies by the kernel's resident CTAs per SM
    a->info.partitions = (uint32_t)P;
  }
  return LLKV_OK;
}

// Zone-map pruning (lean path): every FO_LEAF of the program is a conjunct (`selected &= lo <= v <= hi`), so a tile none
// of whose zones can satisfy some leaf holds no selected row.  The surviving tiles are listed on the host from the
// columns' zone maps and the launch walks the list instead of the dense tile range.  *use_tile_list: the run walks it.
static int32_t agg_tile_list(llkv_gpu_agg* a, uint64_t sig, const std::vector<llkv_gpu_column*>& handles, uint64_t table_rows,
                             uint64_t row_begin, uint64_t row_end, bool* use_tile_list) {
  llkv_gpu_ctx* ctx = a->ctx;
  const Plan& p = a->cr.plan;
  const LeanPlan& lean = a->lean;
  a->info.tiles_pruned = 0;
  bool use = false;
  if (a->cr.fast && ctx->prune_mode && row_end > row_begin) {
    struct PruneLeaf { llkv_gpu_column* col; i64 lo, hi; bool uns; };
    std::vector<PruneLeaf> leaves;
    uint64_t key = fnv_pod(fnv_pod(fnv_pod(fnv_pod(sig, p.tile_rows), row_begin), row_end), ctx->prune_mode);
    for (uint32_t i = 0; i < lean.s.n_code; ++i) {
      const FInstr& in = lean.s.code[i];
      if (in.op != FO_LEAF || in.e) continue;  // (a leaf inside an OR / NOT tree is no conjunct)
      if (in.g >= 2) continue;                 // (float images and IN lists are not ranges of the zone order)
      llkv_gpu_column* col = nullptr;
      for (llkv_gpu_column* h : handles)
        if (h->values == lean.col_base[in.a]) col = h;
      if (!col) continue;
      const bool col_unsigned64 = col->type == LLKV_PT_UINT64;
      if (col_unsigned64 != (in.g != 0)) continue;  // the zone order must be the leaf's compare order
      leaves.push_back(PruneLeaf{col, (i64)lean.lits[in.c], (i64)lean.lits[in.c + 1], in.g != 0});
      key = fnv_pod(fnv_pod(key, col->version), (uint64_t)(uintptr_t)col);
    }
    bool wanted = !leaves.empty();
    if (wanted && ctx->prune_mode == 1) {  // only columns that are scanned again without having changed
      bool settled = true;
      for (PruneLeaf& L : leaves) settled = settled && L.col->scans_unchanged >= 1;
      for (PruneLeaf& L : leaves) ++L.col->scans_unchanged;
      wanted = settled;
    }
    if (wanted && a->tile_list_key == key) {
      use = a->tile_list_use;
    } else if (wanted) {
      const u64 T = p.tile_rows;
      const u64 n_zones = (table_rows + kZoneRows - 1) / kZoneRows;
      std::vector<uint8_t> zone_ok(n_zones, 1);
      bool any_map = false;
      for (PruneLeaf& L : leaves) {
        bool ok = false;
        int32_t rc = ensure_zones(L.col, &ok);
        if (rc) return rc;
        if (!ok || L.col->h_zones.size() != 2 * n_zones) continue;
        any_map = true;
        const u64* z = L.col->h_zones.data();
        for (u64 q = 0; q < n_zones; ++q) {
          const bool disjoint = L.uns ? ((u64)L.hi < z[2 * q] || (u64)L.lo > z[2 * q + 1]) : (L.hi < (i64)z[2 * q] || L.lo > (i64)z[2 * q + 1]);
          const bool empty = L.uns ? (u64)L.hi < (u64)L.lo : L.hi < L.lo;
          if (disjoint || empty) zone_ok[q] = 0;
        }
      }
      const u64 t0 = row_begin / T, t1 = (row_end + T - 1) / T;
      a->h_tile_list.clear();
      if (any_map) {
        for (u64 t = t0; t < t1; ++t) {
          const u64 z0 = t * T / kZoneRows, z1 = std::min<u64>((t + 1) * T - 1, table_rows - 1) / kZoneRows;
          bool keep = false;
          for (u64 q = z0; q <= z1 && !keep; ++q) keep = zone_ok[q] != 0;
          if (keep) a->h_tile_list.push_back((uint32_t)t);
        }
      }
      const u64 total = t1 - t0, kept = any_map ? a->h_tile_list.size() : total;
      a->tile_list_total = total;
      a->tile_list_use = any_map && kept < total && (ctx->prune_mode == 2 || (total - kept) * 8 >= total) && t1 <= 0xffffffffull;
      a->tile_list_key = key;
      if (a->tile_list_use && kept) {
        if (a->tile_list_cap < kept) {
          if (a->d_tile_list) CUDA_TRY(cudaFree(a->d_tile_list));
          a->d_tile_list = nullptr;
          a->tile_list_cap = 0;
          CUDA_TRY(cudaMalloc((void**)&a->d_tile_list, kept * 4));
          a->tile_list_cap = kept;
        }
        CUDA_TRY(cudaMemcpyAsync(a->d_tile_list, a->h_tile_list.data(), kept * 4, cudaMemcpyHostToDevice, ctx->stream));
        CUDA_TRY(cudaStreamSynchronize(ctx->stream));  // (h_tile_list is pageable; once per list)
      }
      use = a->tile_list_use;
    }
    if (use) a->info.tiles_pruned = (uint32_t)(a->tile_list_total - a->h_tile_list.size());
  }
  *use_tile_list = use;
  return LLKV_OK;
}

// The launches of a run: dense row ranges, or runs of the tile list (bounded in tiles, and in the rows they span:
// launch-relative row indices are 32-bit).  A partitioned scan launch is followed by the second pass of its form.
static int32_t agg_run_launches(llkv_gpu_agg* a, uint64_t row_begin, uint64_t row_end, RunLaunches& r, uint32_t* launches_out) {
  llkv_gpu_ctx* ctx = a->ctx;
  const Plan& p = a->cr.plan;
  LeanPlan& lean = a->lean;
  const bool partitioned = a->cr.fast && lean.s.partition != 0;
  const bool packed = a->cr.fast && lean.s.partition == 2;
  a->pending.timed = ctx->timing;
  if (ctx->timing) CUDA_TRY(cudaEventRecord(ctx->ev0, ctx->stream));
  uint32_t launches = 0;
  a->info.used_jit_kernel = 0;
  a->published = false;
  lean.tile_list = nullptr;
  lean.s.use_tile_list = r.use_tile_list ? 1u : 0u;
  const u64 list_n = r.use_tile_list ? a->h_tile_list.size() : 0;
  const u64 tiles_per_launch = std::max<u64>(1, r.max_rows / p.tile_rows);
  u64 list_pos = 0;
  for (u64 rb = row_begin; r.use_tile_list || rb < row_end || (rb == row_begin && launches == 0); rb += r.max_rows) {
    u64 re = std::min<u64>(row_end, rb + r.max_rows);
    u64 first_tile = rb / p.tile_rows;
    u64 n_tiles = re > rb ? (re + p.tile_rows - 1) / p.tile_rows - first_tile : 0;
    if (r.use_tile_list) {
      if (list_pos >= list_n) break;
      first_tile = a->h_tile_list[list_pos];
      n_tiles = 1;
      while (list_pos + n_tiles < list_n && n_tiles < tiles_per_launch &&
             ((u64)a->h_tile_list[list_pos + n_tiles] - first_tile + 1) * p.tile_rows < 0xf0000000ull)
        ++n_tiles;
      const u64 last_tile = a->h_tile_list[list_pos + n_tiles - 1];
      rb = std::max<u64>(row_begin, first_tile * p.tile_rows);
      re = std::min<u64>(row_end, (last_tile + 1) * p.tile_rows);
      lean.tile_list = a->d_tile_list + list_pos;
      list_pos += n_tiles;
    }
    if (n_tiles == 0) break;
    const u64 grid = std::min<u64>(r.g.grid, n_tiles);
    if (!launches) a->info.grid = (uint32_t)grid;
    const bool last = r.use_tile_list ? list_pos >= list_n : re >= row_end;
    a->armed = false;
    if (a->cr.fast) {
      lean.row_begin = rb;
      lean.row_end = re;
      lean.first_tile = first_tile;
      lean.n_tiles = n_tiles;
      if (r.publish && last) {
        lean.publish = a->d_pub;
        lean.ticket = a->d_flags + 1;
        lean.gclass = a->d_gclass;
        a->armed = a->published = true;
        ++a->info.published_steps;
      }
      bool jitted = false;
      if (partitioned) CUDA_TRY(cudaMemsetAsync(a->part_cursor, 0, kMaxPackedPartitions * 4, ctx->stream));
      if (r.use_jit) CUDA_TRY(jit_launch(ctx->device, lean, (int)r.lean_ctas, (uint32_t)grid, ctx->stream, &jitted, nullptr));
      if (partitioned) {
        if (!jitted) return set_error(LLKV_ERR_INTERNAL, "the partitioned scan needs its specialised kernel");
        if (packed) {
          r.fp.row_base = lean.row_origin + first_tile * (u64)p.tile_rows;  // launch-relative row 0
          CUDA_TRY(launch_partition_fold(r.fp, r.part_grid, ctx->stream));
        } else {
          CUDA_TRY(launch_partition_apply(r.pp, r.part_grid, ctx->stream));
        }
        ++launches;
      }
      if (!jitted) CUDA_TRY(launch_lean(lean, (uint32_t)grid, ctx->stream));
      a->info.used_jit_kernel = jitted ? 1 : 0;
    } else {
      Plan lp = p;
      lp.row_begin = rb;
      lp.row_end = re;
      lp.first_tile = first_tile;
      lp.n_tiles = n_tiles;
      if (launches) CUDA_TRY(cudaStreamSynchronize(ctx->stream));  // h_plan is reused
      memcpy(a->h_plan, &lp, sizeof(Plan));
      CUDA_TRY(cudaMemcpyAsync(a->d_plan, a->h_plan, sizeof(Plan), cudaMemcpyHostToDevice, ctx->stream));
      CUDA_TRY(launch_scan(a->d_plan, a->cr.wide, (int)r.g.R, (uint32_t)grid, r.g.block, r.g.smem, ctx->stream));
    }
    ++launches;
    if (last) break;
  }
  lean.publish = nullptr;
  if (ctx->timing) CUDA_TRY(cudaEventRecord(ctx->ev1, ctx->stream));
  *launches_out = launches;
  return LLKV_OK;
}

static int32_t agg_launch(llkv_gpu_agg* a, const llkv_gpu_program* prog, int apply_mvcc, uint64_t row_begin, uint64_t row_end,
                          bool force_wide) {
  llkv_gpu_ctx* ctx = a->ctx;
  CompileRequest req;
  std::vector<llkv_gpu_column*> handles;
  uint64_t table_rows = 0;
  int32_t rc = build_request(ctx, a->table_id, prog, apply_mvcc, req, handles, &table_rows);
  if (rc) return rc;
  if (row_end > table_rows) return set_error(LLKV_ERR_INVALID_ARGUMENT, "row_end %llu beyond the table's %llu rows", (unsigned long long)row_end, (unsigned long long)table_rows);
  // Multi-GPU GROUP BY: the packed key layout (bits, minimum, string length per key) comes from column statistics, and
  // partial tables can only be merged key by key if every rank packs alike.  The ranks agree on the statistics of the
  // key columns (min of minima, max of maxima / string lengths) with one small all-reduce before compiling.
  if (ctx->nccl_comm && ctx->n_ranks > 1 && !a->keys.empty()) {
    bool changed = false;
    if ((rc = agree_dictionaries(ctx, a, handles, &changed))) return rc;
    if (changed) {  // columns were re-coded: their descriptions again
      req = CompileRequest();
      handles.clear();
      if ((rc = build_request(ctx, a->table_id, prog, apply_mvcc, req, handles, &table_rows))) return rc;
    }
    if ((rc = agree_key_stats(ctx, a, req))) return rc;
  }
  const unsigned char* exists_bits = nullptr;
  if ((rc = table_exists_bits(ctx, a->table_id, handles, table_rows, &exists_bits))) return rc;
  const uint64_t sig = request_signature(ctx, req, prog, force_wide, exists_bits);
  RunLaunches r;
  if ((rc = agg_compile(a, req, sig, force_wide, row_begin, row_end, r.g))) return rc;
  a->cr.plan.exists_bits = exists_bits;
  if (a->cr.fast && (rc = agg_choose_form(a, row_begin, row_end, r))) return rc;
  if ((rc = agg_bind_state(a, handles))) return rc;
  // a run from the initial state needs no backup: a rerun starts again from the initial state
  const bool from_reset = a->armed;
  const bool need_backup = !from_reset && (a->cr.can_narrow_fail || a->cr.plan.n_keys != 0);
  if (need_backup && (rc = agg_backup(a))) return rc;
  a->pending.has_backup = need_backup;
  a->pending.from_reset = from_reset;
  r.publish = step_publishes(a->cr.fast && a->lean.s.partition == 0, result_bytes(a->gcap, a->n_gwords, a->cr.plan.n_keys), a->cr.plan.single_wide_key,
                             ctx->n_ranks, from_reset);
  if (r.publish && !a->h_pub) {
    if (a->in_capture) r.publish = false;  // (no allocation inside a stream capture: this step keeps the copy)
    else {
      CUDA_TRY(cudaHostAlloc((void**)&a->h_pub, 8 + kStageBytes, cudaHostAllocMapped));
      CUDA_TRY(cudaHostGetDevicePointer((void**)&a->d_pub, a->h_pub, 0));
    }
  }
  // thread-private partial sums stay exact while a thread folds a bounded number of rows per launch: split very long scans
  // (general interpreter: < 2^15 rows per thread; lean kernel: 2^kLeanRowsPerThreadLog2 rows per consumer thread, and
  // launch-relative row indices must fit 32 bits)
  const uint32_t T = a->cr.plan.tile_rows;
  r.max_rows = (u64)r.g.grid * r.g.block * 32000ull;
  if (a->cr.fast) r.max_rows = std::min<u64>(r.max_rows, 0xf0000000ull) / T * T;
  if ((rc = agg_partitions(a, req, row_begin, row_end, r))) return rc;
  if ((rc = agg_tile_list(a, sig, handles, table_rows, row_begin, row_end, &r.use_tile_list))) return rc;
  uint32_t launches = 0;
  if ((rc = agg_run_launches(a, row_begin, row_end, r, &launches))) return rc;
  if (!a->published && !a->skip_scan_copy && (rc = agg_queue_result_copy(a))) return rc;
  a->info.rows = row_end - row_begin;
  a->info.kernel_launches = launches;
  a->info.used_wide_path = a->cr.wide ? 1 : 0;
  a->info.used_fast_kernel = a->cr.fast ? 1 : 0;
  a->info.algorithmic_bytes_per_row = a->cr.algorithmic_bytes_per_row;
  a->info.physical_bytes_per_row = a->cr.physical_bytes_per_row;
  a->info.block = r.g.block;
  a->info.rows_per_tile = T;
  a->info.stages = a->cr.plan.stages;
  a->info.smem_bytes = r.g.smem;
  a->info.fast_groups = a->cr.plan.fast_groups;
  return LLKV_OK;
}

static int32_t agg_fail(llkv_gpu_agg* a, int32_t code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  a->err_code = code;
  a->err_msg = buf;
  return set_error(code, "%s", buf);
}

// llkv_gpu_agg_reset only marks the state; the status word and the table are cleared here, in stream order, right before
// whatever uses them next (so a reset and the scan that follows it are one run of launches — and one captured graph)
// Puts the status word and the table back to their initial values, in stream order (nothing while the state is armed)
static int32_t agg_rearm(llkv_gpu_agg* a) {
  if (a->armed) return LLKV_OK;
  llkv_gpu_ctx* ctx = a->ctx;
  CUDA_TRY(cudaMemsetAsync(a->d_flags, 0, 4, ctx->stream));
  if (a->frozen) CUDA_TRY(launch_init_table(a->gkeys, a->gwords, a->gcap + 2, a->n_gwords, a->d_gclass, ctx->stream));
  a->armed = a->frozen;
  return LLKV_OK;
}
static int32_t agg_apply_reset(llkv_gpu_agg* a) {
  if (!a->reset_pending) return LLKV_OK;
  a->reset_pending = false;
  a->published = false;  // (the published result is dropped; the scan that published it re-armed the state)
  return agg_rearm(a);
}

// Something continues from the published result (a run without a reset, a merge): the table goes back onto the device
static int32_t agg_unpublish(llkv_gpu_agg* a) {
  if (!a->published) return LLKV_OK;
  llkv_gpu_ctx* ctx = a->ctx;
  a->published = false;
  a->armed = false;
  const u64 n_words = (a->gcap + 2) * a->n_gwords;
  CUDA_TRY(cudaMemcpyAsync(a->gwords, a->h_pub + 1, n_words * 8, cudaMemcpyHostToDevice, ctx->stream));
  if (a->cr.plan.n_keys) CUDA_TRY(cudaMemcpyAsync(a->gkeys, a->h_pub + 1 + n_words, a->gcap * 8, cudaMemcpyHostToDevice, ctx->stream));
  return LLKV_OK;
}

// waits for the outstanding run and settles it: reruns on the 128-bit interpreter / a larger group table when the
// device asked for it, and turns device error flags into the reference's errors
static int32_t agg_merge_impl(llkv_gpu_agg* a);
static int32_t agg_resolve(llkv_gpu_agg* a) {
  llkv_gpu_ctx* ctx = a->ctx;
  if (!a->pending.active) return agg_apply_reset(a);
  for (int guard = 0; guard < 24; ++guard) {
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    if (a->pending.timed) {
      float ms = 0;
      if (cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1) == cudaSuccess) a->info.last_kernel_ms = ms;
      else cudaGetLastError();
    }
    if (a->pending.timed_merge) {
      float ms = 0;
      if (cudaEventElapsedTime(&ms, ctx->ev2, ctx->ev3) == cudaSuccess) a->info.last_merge_ms = ms;
      else cudaGetLastError();
    }
    const uint32_t flags = a->published ? (uint32_t)a->h_pub[0] : *a->h_flags;
    if (flags == 0) break;
    a->prefetched = false;  // the run is repeated or failed: what travelled behind it is not the result
    a->published = false;   // (the scan that published it re-armed the state)
    CUDA_TRY(cudaMemsetAsync(a->d_flags, 0, 4, ctx->stream));
    *a->h_flags = 0;
    const bool narrow_fail = (flags & FLAG_NARROW_FAIL) && !a->pending.wide;
    const bool table_full = (flags & FLAG_TABLE_FULL) != 0;
    const bool merge_retry = a->pending.is_merge && (flags & FLAG_MERGE_RETRY);
    auto merge_again = [&](bool exchange) -> int32_t {  // (a retry is a new exchange on every rank: they all saw the flag)
      CUDA_TRY(launch_merge_grouped_p2p(a->gkeys, a->gwords, a->gcap, a->n_gwords, a->d_gclass, a->d_flags, ctx->peer_gbox, kGroupSlotWords, ctx->n_ranks,
                                        ctx->rank, ctx->d_epoch, exchange, ctx->stream));
      return agg_queue_result_copy(a);
    };
    if (a->pending.is_merge && !merge_retry && table_full && !(flags & ~(uint32_t)FLAG_TABLE_FULL)) {
      // the union of the ranks' groups outgrew this rank's table while folding: a larger, empty table, and fold again
      // (the received tables are still in the mailbox)
      const u64 cap = a->gcap;
      CUDA_TRY(cudaFree(a->gkeys));
      CUDA_TRY(cudaFree(a->gwords));
      a->gkeys = a->gwords = nullptr;
      int32_t rc = agg_alloc_table(a, cap * 4);
      if (!rc) rc = merge_again(false);
      if (rc) {
        a->pending.active = false;
        return rc;
      }
      continue;
    }
    if (a->pending.is_merge && flags == FLAG_MERGE_OVERSIZE) {
      // some rank's table does not fit a mailbox slot (a cardinality hint far below the truth): every rank saw the marker
      // and kept its table, and they all merge over NCCL instead, now and from here on
      a->p2p_group_disabled = true;
      a->pending.is_merge = false;
      a->pending.active = false;
      ++a->plan_epoch;
      return agg_merge_impl(a);
    }
    if (merge_retry && !(narrow_fail || table_full)) {  // another rank repeats its scan: this rank's table is untouched
      int32_t rc = merge_again(true);
      if (rc) {
        a->pending.active = false;
        return rc;
      }
      continue;
    }
    if (narrow_fail || table_full) {
      if (!a->pending.from_reset && !a->pending.has_backup) return agg_fail(a, LLKV_ERR_INTERNAL, "device asked for a rerun without a saved state");
      int32_t rc = a->pending.from_reset ? agg_rearm(a) : agg_restore(a);
      if (rc) return rc;
      if (table_full && (rc = agg_grow_table(a))) return rc;
      if (narrow_fail) a->pending.wide = true;
      a->in_rerun = true;
      rc = agg_launch(a, a->pending.has_prog ? &a->pending.prog : nullptr, a->pending.apply_mvcc, a->pending.row_begin,
                      a->pending.row_end, a->pending.wide);
      a->in_rerun = false;
      if (!rc && merge_retry) rc = merge_again(true);
      if (rc) {
        a->pending.active = false;
        return rc;
      }
      continue;
    }
    a->pending.active = false;
    if (flags & FLAG_BAD_PLAN) return agg_fail(a, LLKV_ERR_INTERNAL, "device interpreter met an unknown instruction");
    if (flags & FLAG_MERGE_TIMEOUT) return agg_fail(a, LLKV_ERR_IO, "multi-GPU merge: a peer's partial state did not arrive within 120 s");
    if (flags & FLAG_TYPE_ERROR) {
      for (const AggLayout& L : a->cr.aggs)
        if (L.raise_code) return agg_fail(a, L.raise_code, "%s", L.raise_message.c_str());
      return agg_fail(a, LLKV_ERR_INTERNAL, "aggregate argument type error");
    }
    if (flags & FLAG_DIV_ZERO) return agg_fail(a, LLKV_ERR_INTERNAL, "Divide by zero error");
    if (flags & FLAG_ARITH_OVERFLOW) return agg_fail(a, LLKV_ERR_INTERNAL, "Arithmetic overflow: Overflow happened in an arrow-arith kernel");
    if (flags & FLAG_EXACT_OVERFLOW) return agg_fail(a, LLKV_ERR_INVALID_ARGUMENT, "Decimal or integer overflow in an exact aggregate expression");
    if (flags & FLAG_MERGE_OVERSIZE) return agg_fail(a, LLKV_ERR_INVALID_ARGUMENT, "multi-GPU merge: a rank's group table outgrew the peer mailbox (the cardinality hint is far too low)");
    if (flags & FLAG_MERGE_PEER_FAILED) return agg_fail(a, LLKV_ERR_INTERNAL, "multi-GPU merge: the scan of another rank failed");
    return agg_fail(a, LLKV_ERR_INTERNAL, "unexpected device status %u", flags);
  }
  a->pending.active = false;
  return LLKV_OK;
}

extern "C" int32_t llkv_gpu_agg_reset(llkv_gpu_agg* a) {
  if (!a) return set_error(LLKV_ERR_INVALID_ARGUMENT, "agg is NULL");
  if (a->inner) return llkv_gpu_agg_reset(a->inner);
  llkv_gpu_ctx* ctx = a->ctx;
  CTX_LOCK(ctx);
  CUDA_TRY(cudaSetDevice(ctx->device));
  if (a->pending.active) {
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    a->pending.active = false;
  }
  a->err_code = 0;
  a->err_msg.clear();
  a->prefetched = false;
  *a->h_flags = 0;
  a->reset_pending = true;
  return LLKV_OK;
}

static int32_t agg_run_impl(llkv_gpu_agg* a, const llkv_gpu_program* prog, int32_t apply_mvcc, uint64_t row_begin, uint64_t row_end) {
  if (a->inner) return agg_run_impl(a->inner, prog, apply_mvcc, row_begin, row_end);
  if (a->err_code) return set_error(a->err_code, "%s", a->err_msg.c_str());
  int32_t rc = agg_resolve(a);
  if (rc) return rc;
  if ((rc = agg_unpublish(a))) return rc;
  a->pending.has_prog = prog != nullptr;
  if (prog && a->pending.prog.serial != prog->serial) {
    a->pending.prog.ops = prog->ops;
    a->pending.prog.literals = prog->literals;
    a->pending.prog.nodes = prog->nodes;
    a->pending.prog.list_roots = prog->list_roots;
    a->pending.prog.serial = prog->serial;
    a->pending.prog.bind();
  }
  a->pending.apply_mvcc = apply_mvcc;
  a->pending.row_begin = row_begin;
  a->pending.row_end = row_end;
  a->pending.wide = false;
  a->pending.is_merge = false;
  a->pending.timed_merge = false;
  rc = agg_launch(a, prog, apply_mvcc, row_begin, row_end, false);
  if (rc) return rc;
  a->pending.wide = a->cr.wide;
  a->pending.active = true;
  ++a->runs_done;
  return LLKV_OK;
}

extern "C" int32_t llkv_gpu_agg_run(llkv_gpu_agg* a, const llkv_gpu_program* prog, int32_t apply_mvcc, uint64_t row_begin,
                                     uint64_t row_end) {
  if (!a) return set_error(LLKV_ERR_INVALID_ARGUMENT, "agg is NULL");
  if (row_end < row_begin) return set_error(LLKV_ERR_INVALID_ARGUMENT, "row_end < row_begin");
  CTX_LOCK(a->ctx);
  CUDA_TRY(cudaSetDevice(a->ctx->device));
  return agg_run_impl(a, prog, apply_mvcc, row_begin, row_end);
}

extern "C" int32_t llkv_gpu_agg_run_info(const llkv_gpu_agg* a, llkv_run_info* out) {
  if (!a || !out) return set_error(LLKV_ERR_INVALID_ARGUMENT, "NULL argument");
  if (a->inner) a = a->inner;
  *out = a->info;
  return LLKV_OK;
}

// ---- finalize -----------------------------------------------------------------------------------------------
static void val_i64(llkv_agg_value* o, i64 v, int valid) {
  memset(o, 0, sizeof(*o));
  o->type = LLKV_PT_INT64;
  o->lo = valid ? (uint64_t)v : 0;
  o->valid = (uint8_t)valid;
}
static void val_f64(llkv_agg_value* o, double v, int valid) {
  memset(o, 0, sizeof(*o));
  o->type = LLKV_PT_FLOAT64;
  if (valid) memcpy(&o->lo, &v, 8);
  o->valid = (uint8_t)valid;
}
static void val_dec(llkv_agg_value* o, i128 v, int p, int s, int valid) {
  memset(o, 0, sizeof(*o));
  o->type = LLKV_PT_DECIMAL128;
  o->precision = (uint8_t)p;
  o->scale = (int8_t)s;
  o->valid = (uint8_t)valid;
  if (valid) {
    o->lo = (uint64_t)(u128)v;
    o->hi = (uint64_t)((u128)v >> 64);
  }
}
static double dec_f64_bits(u64 e) {  // inverse of enc_f64
  const u64 b = (e >> 63) ? (e & 0x7fffffffffffffffull) : ~e;
  double d;
  memcpy(&d, &b, 8);
  return d;
}
// exact value of a limb-split integer sum; false when it does not fit in i128
static bool limbs_value(const u64* w, int n_limbs, i128* out) {
  if (n_limbs == 2) {
    *out = (i128)(u128)w[0] + (((i128)(i64)w[1]) << 32);
    return true;
  }
  u128 d0 = w[0];
  u128 d1 = (u128)w[1] + (d0 >> 32);
  d0 &= 0xffffffffull;
  u128 d2 = (u128)w[2] + (d1 >> 32);
  d1 &= 0xffffffffull;
  const i128 top = (i128)(i64)w[3] + (i128)(d2 >> 32);
  d2 &= 0xffffffffull;
  if (top < -((i128)1 << 31) || top >= ((i128)1 << 31)) return false;
  *out = (i128)(((u128)top << 96) | (d2 << 64) | (d1 << 32) | d0);
  return true;
}

static int32_t finalize_group(llkv_gpu_agg* a, const u64* w, llkv_agg_value* out) {
  const std::vector<AggLayout>& aggs = a->cr.aggs;
  const u64 rows = w[0];
  for (size_t i = 0; i < aggs.size(); ++i) {
    const AggLayout& L = aggs[i];
    llkv_agg_value* o = &out[i];
    const u64 count = L.dead ? 0 : (L.w_count >= 0 ? w[L.w_count] : 0);
    i128 total = 0;
    if (L.all_null_group_is_error && rows > 0 && count == 0) return agg_fail(a, LLKV_ERR_INVALID_ARGUMENT, "Expected Decimal128 array");
    switch (L.acc) {
      case ACC_COUNT_STAR: val_i64(o, (i64)rows, 1); break;
      case ACC_COUNT_COL: val_i64(o, (i64)count, 1); break;
      case ACC_COUNT_NULLS: val_i64(o, (i64)(rows - count), 1); break;
      case ACC_SUM_I64:
        if (L.dead || count == 0) { val_i64(o, 0, 0); break; }
        limbs_value(&w[L.w_val], 2, &total);
        if (total < (i128)INT64_MIN || total > (i128)INT64_MAX) return agg_fail(a, LLKV_ERR_INVALID_ARGUMENT, "integer overflow");
        val_i64(o, (i64)total, 1);
        break;
      case ACC_AVG_I64:
        if (L.dead || count == 0) { val_f64(o, 0, 0); break; }
        limbs_value(&w[L.w_val], 2, &total);
        if (total < (i128)INT64_MIN || total > (i128)INT64_MAX) return agg_fail(a, LLKV_ERR_INVALID_ARGUMENT, "AVG aggregate sum exceeds i64 range");
        val_f64(o, (double)(i64)total / (double)(i64)count, 1);
        break;
      case ACC_TOTAL_I64: case ACC_TOTAL_F64: {
        double f = 0.0;
        if (!L.dead) memcpy(&f, &w[L.w_val], 8);
        val_f64(o, f, 1);
        break;
      }
      case ACC_SUM_F64: {
        double f = 0.0;
        if (!L.dead) memcpy(&f, &w[L.w_val], 8);
        val_f64(o, f, !L.dead && count > 0);
        break;
      }
      case ACC_AVG_F64: {
        double f = 0.0;
        if (!L.dead) memcpy(&f, &w[L.w_val], 8);
        val_f64(o, count > 0 ? f / (double)(i64)count : 0.0, !L.dead && count > 0);
        break;
      }
      case ACC_MIN_I64: case ACC_MAX_I64:
        if (L.dead || count == 0) val_i64(o, 0, 0);
        else val_i64(o, (i64)(w[L.w_val] ^ 0x8000000000000000ull), 1);
        break;
      case ACC_MIN_F64: case ACC_MAX_F64: {
        if (L.dead || w[L.w_first_valid] == ~0ull) { val_f64(o, 0, 0); break; }
        // a leading NaN sticks: nothing compares Less/Greater than it (llkv-aggregate/src/lib.rs:1309-1331,1377-1399)
        if (w[L.w_first_nan] == w[L.w_first_valid]) {
          const u64 qnan = 0x7ff8000000000000ull;
          double d;
          memcpy(&d, &qnan, 8);
          val_f64(o, d, 1);
        } else {
          val_f64(o, dec_f64_bits(w[L.w_val]), 1);
        }
        break;
      }
      case ACC_SUM_DEC: case ACC_TOTAL_DEC:
        if (L.dead) { val_dec(o, 0, L.precision, L.scale, 1); break; }
        if (!limbs_value(&w[L.w_val], 4, &total))
          return agg_fail(a, LLKV_ERR_INVALID_ARGUMENT, L.acc == ACC_TOTAL_DEC ? "Decimal128 total overflow" : "Decimal128 sum overflow");
        val_dec(o, total, L.precision, L.scale, 1);  // always a value: 0 when no rows (lib.rs:1567-1582)
        break;
      case ACC_AVG_DEC: {
        if (L.dead || count == 0) { val_dec(o, 0, L.precision, L.scale, 0); break; }
        if (!limbs_value(&w[L.w_val], 4, &total)) return agg_fail(a, LLKV_ERR_INVALID_ARGUMENT, "Decimal128 sum overflow");
        const i128 c = (i128)count;
        i128 avg = total / c;
        const i128 rem = total % c;
        const i128 ar = rem < 0 ? -rem : rem;
        if (ar * 2 >= c) {  // round half away from zero (lib.rs:1731-1742)
          if (total > 0) avg += 1;
          else avg -= 1;
        }
        val_dec(o, avg, L.precision, L.scale, 1);
        break;
      }
      case ACC_MIN_DEC: case ACC_MAX_DEC:
        if (L.dead || count == 0) val_dec(o, 0, L.precision, L.scale, 0);
        else {
          const u64 hi = w[L.w_val] ^ 0x8000000000000000ull, lo = w[L.w_val + 1];
          val_dec(o, (i128)(((u128)hi << 64) | lo), L.precision, L.scale, 1);
        }
        break;
      default: return agg_fail(a, LLKV_ERR_INTERNAL, "unknown accumulator %d", L.acc);
    }
  }
  return LLKV_OK;
}

static void decode_keys(const llkv_gpu_agg* a, u64 K, bool null_slot, llkv_group_key* out) {
  const std::vector<KeyLayout>& keys = a->cr.keys;
  const Plan& p = a->cr.plan;
  int shift = 0;
  for (size_t k = 0; k < keys.size(); ++k) {
    const KeyLayout& kl = keys[k];
    llkv_group_key* o = &out[k];
    memset(o, 0, sizeof(*o));
    o->type = kl.type;
    if (p.single_wide_key == 1) {
      o->valid = null_slot ? 0 : 1;
      o->bits = null_slot ? 0 : K;
      if (kl.type == LLKV_PT_BOOLEAN && o->valid) o->bits = o->bits != 0;
      continue;
    }
    const u64 field = kl.bits == 64 ? (K >> shift) : ((K >> shift) & ((1ull << kl.bits) - 1));
    shift += kl.bits;
    bool isnull = false;
    if (kl.nullable) {
      isnull = (K >> shift) & 1;
      shift += 1;
    }
    o->valid = isnull ? 0 : 1;
    if (isnull) continue;
    o->dict = kl.dict ? 1 : 0;
    if (kl.kind == KK_STR) {
      const int L = kl.strlen;
      const u64 len = field & 7, bytes = field >> 3;
      o->bits = (L ? (bytes << (64 - 8 * L)) : 0ull) | len;
    } else {
      u64 v = field + kl.min;
      // without statistics the field holds the low bits of the sign-extended value
      if (kl.min == 0 && kl.is_signed && kl.bits < 64 && kl.bits == 8 * prim_type_width(kl.type) && ((v >> (kl.bits - 1)) & 1))
        v |= ~0ull << kl.bits;
      o->bits = kl.type == LLKV_PT_BOOLEAN ? (u64)(v != 0) : v;
    }
  }
}

struct GroupRef {
  u64 slot, first_row;
};

static bool wide_key_cols(const llkv_gpu_agg* a, WideKeyCols* out, u64* n_rows, u64* origin) {
  memset(out, 0, sizeof(*out));
  const std::vector<KeyLayout>& keys = a->cr.keys;
  out->n_keys = (uint32_t)keys.size();
  *n_rows = ~0ull;
  *origin = 0;
  for (size_t k = 0; k < keys.size(); ++k) {
    llkv_gpu_column* col = nullptr;
    for (auto& kv : a->ctx->columns)
      if (lfid_table(kv.second->lfid) == (a->table_id & 0xffffull) && lfid_field(kv.second->lfid) == keys[k].field_id) col = kv.second;
    if (!col) return false;
    out->values[k] = col->values;
    out->validity[k] = col->validity;
    out->load_kind[k] = col->load_kind;
    *n_rows = std::min<u64>(*n_rows, col->n_rows);
    if (col->has_origin) *origin = col->row_id_origin;
  }
  return true;
}

// Hashed wide keys: proves once per run that no two different keys share a group, then reads every group's key values
// from the columns at the group's first row.
static int32_t wide_keys_fetch(llkv_gpu_agg* a, const std::vector<GroupRef>& groups, std::vector<llkv_group_key>& out) {
  llkv_gpu_ctx* ctx = a->ctx;
  const std::vector<KeyLayout>& keys = a->cr.keys;
  const size_t nk = keys.size(), ng = groups.size();
  out.assign(ng * nk, llkv_group_key());
  if (ng == 0) return LLKV_OK;
  WideKeyCols cols;
  u64 n_rows, origin;
  if (!wide_key_cols(a, &cols, &n_rows, &origin)) return set_error(LLKV_ERR_INTERNAL, "a GROUP BY key column is gone");
  cudaStream_t s = ctx->stream;
  if (a->wide_verified != a->runs_done) {
    unsigned int* d_flag = nullptr;
    CUDA_TRY(cudaMalloc((void**)&d_flag, 4));
    CUDA_TRY(cudaMemsetAsync(d_flag, 0, 4, s));
    wide_key_verify_kernel<<<1184, 256, 0, s>>>(cols, n_rows, origin, a->gkeys, a->gwords, a->gcap, a->n_gwords, d_flag);
    CUDA_TRY(cudaGetLastError());
    unsigned int flag = 0;
    CUDA_TRY(cudaMemcpyAsync(&flag, d_flag, 4, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    CUDA_TRY(cudaFree(d_flag));
    if (flag) return agg_fail(a, LLKV_ERR_INTERNAL, "two different GROUP BY keys share a 64-bit hash (FLAG_KEY_COLLISION): this query cannot run on this path");
    a->wide_verified = a->runs_done;
  }
  std::vector<u64> pos(ng);
  for (size_t g = 0; g < ng; ++g) pos[g] = groups[g].first_row - origin;
  u64 *d_pos = nullptr, *d_bits = nullptr;
  unsigned char* d_null = nullptr;
  CUDA_TRY(cudaMalloc((void**)&d_pos, ng * 8));
  cudaError_t e = cudaMalloc((void**)&d_bits, ng * nk * 8);
  if (e == cudaSuccess) e = cudaMalloc((void**)&d_null, ng * nk);
  std::vector<u64> bits(ng * nk);
  std::vector<unsigned char> nul(ng * nk);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_pos, pos.data(), ng * 8, cudaMemcpyHostToDevice, s);
  if (e == cudaSuccess) {
    wide_key_gather_kernel<<<(unsigned)std::min<u64>((ng + 255) / 256, 1184), 256, 0, s>>>(cols, d_pos, ng, n_rows, d_bits, d_null);
    e = cudaGetLastError();
  }
  if (e == cudaSuccess) e = cudaMemcpyAsync(bits.data(), d_bits, ng * nk * 8, cudaMemcpyDeviceToHost, s);
  if (e == cudaSuccess) e = cudaMemcpyAsync(nul.data(), d_null, ng * nk, cudaMemcpyDeviceToHost, s);
  if (e == cudaSuccess) e = cudaStreamSynchronize(s);
  cudaFree(d_pos);
  if (d_bits) cudaFree(d_bits);
  if (d_null) cudaFree(d_null);
  if (e != cudaSuccess) return set_error(LLKV_ERR_IO, "CUDA error %s reading GROUP BY keys", cudaGetErrorString(e));
  for (size_t g = 0; g < ng; ++g)
    for (size_t k = 0; k < nk; ++k) {
      llkv_group_key* o = &out[g * nk + k];
      o->type = keys[k].type;
      o->valid = nul[g * nk + k] ? 0 : 1;
      if (!o->valid) continue;
      o->dict = keys[k].dict ? 1 : 0;
      o->bits = keys[k].type == LLKV_PT_BOOLEAN ? (u64)(bits[g * nk + k] != 0) : bits[g * nk + k];
    }
  return LLKV_OK;
}

static int32_t agg_collect(llkv_gpu_agg* a, std::vector<u64>& hk, std::vector<u64>& hw, std::vector<GroupRef>& groups) {
  llkv_gpu_ctx* ctx = a->ctx;
  const u64 rows = a->gcap + 2;
  hk.resize(a->gcap);
  hw.resize(rows * a->n_gwords);
  const size_t wbytes = hw.size() * 8, kbytes = a->cr.plan.n_keys ? hk.size() * 8 : 0;
  if (a->published) {  // the scan put it there (agg_resolve waited for it)
    memcpy(hw.data(), a->h_pub + 1, wbytes);
    if (kbytes) memcpy(hk.data(), a->h_pub + 1 + hw.size(), kbytes);
  } else if (a->prefetched && a->h_stage_bytes >= wbytes + kbytes) {  // already on its way (agg_queue_result_copy)
    // usually complete: agg_resolve waited for the run.  Not when the copy was queued with no run pending (a merge behind
    // a run that had to be settled first).
    if (a->stage_ev_valid) CUDA_TRY(cudaEventSynchronize(a->stage_ev));
    else CUDA_TRY(cudaStreamSynchronize(ctx->stream));  // (replayed from a graph: the event belongs to the capture)
    memcpy(hw.data(), a->h_stage, wbytes);
    if (kbytes) memcpy(hk.data(), a->h_stage + wbytes, kbytes);
  } else if (wbytes + kbytes <= (4u << 20)) {  // small tables land in a page-locked buffer (one DMA each, no pageable staging)
    if (a->h_stage_bytes < wbytes + kbytes) {
      if (a->h_stage) CUDA_TRY(cudaFreeHost(a->h_stage));
      a->h_stage = nullptr;
      CUDA_TRY(cudaHostAlloc((void**)&a->h_stage, wbytes + kbytes, cudaHostAllocDefault));
      a->h_stage_bytes = wbytes + kbytes;
    }
    CUDA_TRY(cudaMemcpyAsync(a->h_stage, a->gwords, wbytes, cudaMemcpyDeviceToHost, ctx->stream));
    if (kbytes) CUDA_TRY(cudaMemcpyAsync(a->h_stage + wbytes, a->gkeys, kbytes, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    memcpy(hw.data(), a->h_stage, wbytes);
    if (kbytes) memcpy(hk.data(), a->h_stage + wbytes, kbytes);
  } else {
    CUDA_TRY(cudaMemcpyAsync(hw.data(), a->gwords, wbytes, cudaMemcpyDeviceToHost, ctx->stream));
    if (kbytes) CUDA_TRY(cudaMemcpyAsync(hk.data(), a->gkeys, kbytes, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  }
  groups.clear();
  if (a->cr.plan.n_keys == 0) {
    groups.push_back(GroupRef{0, 0});
    return LLKV_OK;
  }
  for (u64 s = 0; s < rows; ++s) {
    const bool occupied = s < a->gcap ? hk[s] != kEmptyKey : hw[s * a->n_gwords] != 0;
    if (!occupied) continue;
    groups.push_back(GroupRef{s, hw[s * a->n_gwords + 1]});
  }
  // first-appearance order of the groups (llkv-executor/src/lib.rs:5064-5089)
  std::sort(groups.begin(), groups.end(), [](const GroupRef& x, const GroupRef& y) { return x.first_row < y.first_row; });
  if (a->hint && a->hint <= 128 && groups.size() > a->hint && groups.size() > a->observed_groups) {
    a->observed_groups = groups.size();  // the caller's hint was low: later runs of this aggregate get more CTA-local slots
    a->forget_forms();
    ++a->plan_epoch;
  }
  return LLKV_OK;
}

static int32_t agg_ensure_layout(llkv_gpu_agg* a) {
  if (a->frozen) return LLKV_OK;
  // finalize before any run: compile against the table to learn the layout, with an empty scan
  int32_t rc = agg_launch(a, nullptr, 0, 0, 0, false);
  if (rc) return rc;
  CUDA_TRY(cudaStreamSynchronize(a->ctx->stream));
  return LLKV_OK;
}

extern "C" int32_t llkv_gpu_agg_group_count(llkv_gpu_agg* a, uint64_t* out_groups) {
  if (!a || !out_groups) return set_error(LLKV_ERR_INVALID_ARGUMENT, "NULL argument");
  if (a->inner) {  // DISTINCT aggregates are ungrouped: one row
    *out_groups = 1;
    return LLKV_OK;
  }
  CTX_LOCK(a->ctx);
  CUDA_TRY(cudaSetDevice(a->ctx->device));
  if (a->err_code) return set_error(a->err_code, "%s", a->err_msg.c_str());
  int32_t rc = agg_resolve(a);
  if (rc) return rc;
  if ((rc = agg_ensure_layout(a))) return rc;
  std::vector<u64> hk, hw;
  std::vector<GroupRef> groups;
  if ((rc = agg_collect(a, hk, hw, groups))) return rc;
  *out_groups = groups.size();
  return LLKV_OK;
}

// ---- output shaping: HAVING / ORDER BY / OFFSET / LIMIT over the finalized rows (llkv-executor/src/lib.rs:5306-5348) -----
static i128 cell_i128(const llkv_agg_value& v) { return (i128)(((u128)v.hi << 64) | (u128)v.lo); }
static double cell_f64(const llkv_agg_value& v) {
  double d;
  memcpy(&d, &v.lo, 8);
  return d;
}
// three-way compare of two cells of one output column (same type); NaN sorts above every number, like arrow's sort
static int compare_values(const llkv_agg_value& x, const llkv_agg_value& y) {
  if (x.type == LLKV_PT_FLOAT64) {
    const double a = cell_f64(x), b = cell_f64(y);
    const bool an = a != a, bn = b != b;
    if (an || bn) return an == bn ? 0 : (an ? 1 : -1);
    return a < b ? -1 : (a > b ? 1 : 0);
  }
  const i128 a = x.type == LLKV_PT_DECIMAL128 ? cell_i128(x) : (i128)(i64)x.lo, b = y.type == LLKV_PT_DECIMAL128 ? cell_i128(y) : (i128)(i64)y.lo;
  return a < b ? -1 : (a > b ? 1 : 0);
}
static int compare_keys(const llkv_group_key& x, const llkv_group_key& y) {
  const bool uns = x.type == LLKV_PT_UTF8 || x.type == LLKV_PT_UINT64 || x.type == LLKV_PT_UINT32 || x.type == LLKV_PT_UINT16 || x.type == LLKV_PT_UINT8 ||
                   x.type == LLKV_PT_BOOLEAN;  // (strings: bytes from the top byte, length in the low one: byte order)
  if (uns) return x.bits < y.bits ? -1 : (x.bits > y.bits ? 1 : 0);
  return (i64)x.bits < (i64)y.bits ? -1 : ((i64)x.bits > (i64)y.bits ? 1 : 0);
}
// TRUE / FALSE of `cell cmp literal`; a NULL cell is neither (HAVING keeps rows that evaluate to TRUE only)
// the dictionary behind key `index` of an aggregate whose key column is dictionary-coded, else null
static const StrDict* key_dict(const llkv_gpu_agg* a, size_t index) {
  if (index >= a->cr.keys.size() || !a->cr.keys[index].dict) return nullptr;
  for (auto& kv : a->ctx->columns)
    if (lfid_table(kv.second->lfid) == (a->table_id & 0xffffull) && lfid_field(kv.second->lfid) == a->cr.keys[index].field_id) return kv.second->dict.get();
  return nullptr;
}

static bool having_holds(const llkv_having_term& t, const llkv_agg_value* v, const llkv_group_key* k, const StrDict* dict = nullptr) {
  int c;
  if (t.is_aggregate) {
    if (!v->valid) return false;
    if (v->type == LLKV_PT_FLOAT64 || t.literal.kind == LLKV_LIT_FLOAT64) {
      double lit;
      if (t.literal.kind == LLKV_LIT_FLOAT64) memcpy(&lit, &t.literal.lo, 8);
      else lit = (double)(i128)(((u128)t.literal.hi << 64) | t.literal.lo) / pow(10.0, t.literal.kind == LLKV_LIT_DECIMAL128 ? t.literal.scale : 0);
      const double x = v->type == LLKV_PT_FLOAT64 ? cell_f64(*v) : (double)(v->type == LLKV_PT_DECIMAL128 ? cell_i128(*v) : (i128)(i64)v->lo) /
                                                                       pow(10.0, v->type == LLKV_PT_DECIMAL128 ? v->scale : 0);
      c = x < lit ? -1 : (x > lit ? 1 : 0);
    } else {  // exact: both sides as integers at the larger scale
      i128 x = v->type == LLKV_PT_DECIMAL128 ? cell_i128(*v) : (i128)(i64)v->lo, lit = (i128)(((u128)t.literal.hi << 64) | t.literal.lo);
      int sx = v->type == LLKV_PT_DECIMAL128 ? v->scale : 0, sl = t.literal.kind == LLKV_LIT_DECIMAL128 ? t.literal.scale : 0;
      for (; sx < sl; ++sx) x *= 10;
      for (; sl < sx; ++sl) lit *= 10;
      c = x < lit ? -1 : (x > lit ? 1 : 0);
    }
  } else {
    if (!k->valid) return false;
    llkv_group_key lit = *k;
    if (k->dict) {  // a dictionary code: compare the entry's bytes with the literal's (str: Ord)
      if (!dict || t.literal.kind != LLKV_LIT_STRING || k->bits >= dict->sorted.size()) return false;
      const char* bytes;
      size_t len;
      literal_bytes(t.literal, &bytes, &len);
      c = dict->sorted[(size_t)k->bits].compare(std::string(bytes, len));
      c = c < 0 ? -1 : (c > 0 ? 1 : 0);
    } else if (t.literal.kind == LLKV_LIT_STRING) {  // literal bytes (little endian in lo/hi) -> the key's packed form
      uint64_t bits = 0;
      const char* bytes;
      size_t len;
      literal_bytes(t.literal, &bytes, &len);
      if (len > 7) return false;
      for (size_t i = 0; i < len; ++i) bits |= (uint64_t)(unsigned char)bytes[i] << (56 - 8 * i);
      lit.bits = bits | len;
    } else {
      lit.bits = t.literal.lo;
    }
    if (!k->dict) c = compare_keys(*k, lit);
  }
  switch (t.cmp_op) {
    case LLKV_CMP_EQ: return c == 0;
    case LLKV_CMP_NE: return c != 0;
    case LLKV_CMP_LT: return c < 0;
    case LLKV_CMP_LE: return c <= 0;
    case LLKV_CMP_GT: return c > 0;
    default: return c >= 0;
  }
}

// DISTINCT aggregates from the inner aggregation's groups (one per distinct value; the NULL group does not count)
static int32_t finalize_distinct(llkv_gpu_agg* a, llkv_agg_value* out) {
  llkv_gpu_agg* in = a->inner;
  int32_t rc = agg_resolve(in);
  if (rc) return rc;
  if ((rc = agg_ensure_layout(in))) return rc;
  std::vector<u64> hk, hw;
  std::vector<GroupRef> groups;
  if ((rc = agg_collect(in, hk, hw, groups))) return rc;
  i128 sum = 0;
  u64 count = 0;
  for (const GroupRef& g : groups) {
    if (g.slot == in->gcap + 1) continue;  // NULL key
    llkv_group_key k;
    decode_keys(in, g.slot < in->gcap ? hk[g.slot] : kEmptyKey, false, &k);
    if (!k.valid) continue;  // (a nullable key packs its NULL flag into the key)
    if (k.type == LLKV_PT_UTF8 || k.type == LLKV_PT_BOOLEAN) return agg_fail(a, LLKV_ERR_INVALID_ARGUMENT, "DISTINCT aggregates on this path take integer columns");
    const bool uns = k.type == LLKV_PT_UINT64;
    sum += uns ? (i128)k.bits : (i128)(i64)k.bits;
    ++count;
  }
  for (size_t i = 0; i < a->specs.size(); ++i) {
    llkv_agg_value* o = &out[i];
    switch (a->specs[i].kind) {
      case LLKV_AGG_COUNT: val_i64(o, (i64)count, 1); break;
      case LLKV_AGG_SUM:
        if (!count) { val_i64(o, 0, 0); break; }
        if (sum < (i128)INT64_MIN || sum > (i128)INT64_MAX) return agg_fail(a, LLKV_ERR_INVALID_ARGUMENT, "integer overflow");
        val_i64(o, (i64)sum, 1);
        break;
      case LLKV_AGG_TOTAL: val_f64(o, (double)sum, 1); break;
      default:  // AVG
        if (!count) { val_f64(o, 0, 0); break; }
        val_f64(o, (double)sum / (double)count, 1);
        break;
    }
  }
  return LLKV_OK;
}

extern "C" int32_t llkv_gpu_agg_finalize(llkv_gpu_agg* a, llkv_agg_value* out_values, llkv_group_key* out_keys, uint64_t group_capacity,
                                          uint64_t* out_groups) {
  if (!a) return set_error(LLKV_ERR_INVALID_ARGUMENT, "agg is NULL");
  CTX_LOCK(a->ctx);
  CUDA_TRY(cudaSetDevice(a->ctx->device));
  if (a->inner) {
    if (group_capacity < 1 || !out_values) return set_error(LLKV_ERR_INVALID_ARGUMENT, "output buffer too small");
    const int32_t drc = finalize_distinct(a, out_values);
    if (drc) return drc;
    if (out_groups) *out_groups = 1;
    return LLKV_OK;
  }
  if (a->err_code) return set_error(a->err_code, "%s", a->err_msg.c_str());
  int32_t rc = agg_resolve(a);
  if (rc) return rc;
  if ((rc = agg_ensure_layout(a))) return rc;
  std::vector<u64> hk, hw;
  std::vector<GroupRef> groups;
  if ((rc = agg_collect(a, hk, hw, groups))) return rc;
  const size_t n_aggs = a->specs.size(), n_keys = a->keys.size();
  const bool shaped = !a->having.empty() || !a->order.empty() || a->out_offset || a->out_limit;
  const bool hashed = n_keys && a->cr.plan.single_wide_key == 2;
  std::vector<llkv_group_key> wide;
  if (hashed && (rc = wide_keys_fetch(a, groups, wide))) return rc;
  if (!shaped) {
    if (groups.size() > group_capacity)
      return set_error(LLKV_ERR_INVALID_ARGUMENT, "group capacity %llu < %llu groups", (unsigned long long)group_capacity, (unsigned long long)groups.size());
    if ((n_aggs && !out_values) || (n_keys && !out_keys)) return set_error(LLKV_ERR_INVALID_ARGUMENT, "output buffer is NULL");
    for (size_t gi = 0; gi < groups.size(); ++gi) {
      const u64 s = groups[gi].slot;
      if ((rc = finalize_group(a, &hw[s * a->n_gwords], out_values + gi * n_aggs))) return rc;
      if (hashed) {
        memcpy(out_keys + gi * n_keys, wide.data() + gi * n_keys, n_keys * sizeof(llkv_group_key));
      } else if (n_keys) {
        const bool null_slot = s == a->gcap + 1;
        const u64 K = s < a->gcap ? hk[s] : kEmptyKey;
        decode_keys(a, K, null_slot, out_keys + gi * n_keys);
      }
    }
    if (out_groups) *out_groups = groups.size();
    return LLKV_OK;
  }
  // every group first (first-appearance order), then HAVING, ORDER BY (stable), OFFSET / LIMIT
  std::vector<llkv_agg_value> vals(groups.size() * std::max<size_t>(1, n_aggs));
  std::vector<llkv_group_key> keys(groups.size() * std::max<size_t>(1, n_keys));
  for (size_t gi = 0; gi < groups.size(); ++gi) {
    const u64 s = groups[gi].slot;
    if ((rc = finalize_group(a, &hw[s * a->n_gwords], vals.data() + gi * n_aggs))) return rc;
    if (hashed) memcpy(keys.data() + gi * n_keys, wide.data() + gi * n_keys, n_keys * sizeof(llkv_group_key));
    else if (n_keys) decode_keys(a, s < a->gcap ? hk[s] : kEmptyKey, s == a->gcap + 1, keys.data() + gi * n_keys);
  }
  std::vector<size_t> rows;
  for (size_t gi = 0; gi < groups.size(); ++gi) {
    bool keep = true;
    for (const llkv_having_term& t : a->having)
      keep = keep && having_holds(t, t.is_aggregate ? &vals[gi * n_aggs + (size_t)t.index] : nullptr, t.is_aggregate ? nullptr : &keys[gi * n_keys + (size_t)t.index],
                                  t.is_aggregate ? nullptr : key_dict(a, (size_t)t.index));
    if (keep) rows.push_back(gi);
  }
  if (!a->order.empty())
    std::stable_sort(rows.begin(), rows.end(), [&](size_t x, size_t y) {
      for (const llkv_order_key& o : a->order) {
        bool xv, yv;
        int c;
        if (o.is_aggregate) {
          const llkv_agg_value &vx = vals[x * n_aggs + (size_t)o.index], &vy = vals[y * n_aggs + (size_t)o.index];
          xv = vx.valid;
          yv = vy.valid;
          c = xv && yv ? compare_values(vx, vy) : 0;
        } else {
          const llkv_group_key &kx = keys[x * n_keys + (size_t)o.index], &ky = keys[y * n_keys + (size_t)o.index];
          xv = kx.valid;
          yv = ky.valid;
          c = xv && yv ? compare_keys(kx, ky) : 0;
        }
        if (xv != yv) return o.nulls_first ? !xv : xv;  // NULLs go where nulls_first says, whatever the direction
        if (c) return o.descending ? c > 0 : c < 0;
      }
      return false;
    });
  const size_t begin = std::min<size_t>(rows.size(), (size_t)a->out_offset);
  const size_t end = a->out_limit ? std::min<size_t>(rows.size(), begin + (size_t)a->out_limit) : rows.size();
  if (end - begin > group_capacity)
    return set_error(LLKV_ERR_INVALID_ARGUMENT, "group capacity %llu < %llu groups", (unsigned long long)group_capacity, (unsigned long long)(end - begin));
  if ((n_aggs && !out_values) || (n_keys && !out_keys)) return set_error(LLKV_ERR_INVALID_ARGUMENT, "output buffer is NULL");
  for (size_t i = begin; i < end; ++i) {
    if (n_aggs) memcpy(out_values + (i - begin) * n_aggs, vals.data() + rows[i] * n_aggs, n_aggs * sizeof(llkv_agg_value));
    if (n_keys) memcpy(out_keys + (i - begin) * n_keys, keys.data() + rows[i] * n_keys, n_keys * sizeof(llkv_group_key));
  }
  if (out_groups) *out_groups = end - begin;
  return LLKV_OK;
}

// ------------------------------------------------------------------------------------------------ multi-GPU
extern "C" int32_t llkv_gpu_comm_unique_id(uint8_t out_id[LLKV_GPU_UNIQUE_ID_BYTES]) {
  if (!out_id) return set_error(LLKV_ERR_INVALID_ARGUMENT, "out_id is NULL");
  int32_t rc = load_nccl();
  if (rc) return rc;
  NCCL_TRY(g_nccl.get_unique_id(out_id));
  return LLKV_OK;
}

static void comm_teardown_p2p(llkv_gpu_ctx* ctx);
// Maps every rank's mailbox into every other rank (CUDA IPC over NVLink peer access).  The handles travel through the
// NCCL communicator that was just created; the peer-memory path is used only when every rank managed to map every peer
// (agreed with an all-reduce), otherwise the merge stays on NCCL.  LLKV_GPU_NO_P2P_MERGE=1 forces the NCCL path.
static void comm_setup_p2p(llkv_gpu_ctx* ctx) {
  const int N = ctx->n_ranks;
  ctx->p2p_merge = false;
  const char* off = getenv("LLKV_GPU_NO_P2P_MERGE");
  if (N < 2 || N > 8 || (off && off[0] && off[0] != '0')) return;
  const int nccl_u8 = 1 /* ncclUint8 */, nccl_u64 = 5 /* ncclUint64 */, nccl_min = 3 /* ncclMin */;
  const size_t box_bytes = (size_t)N * 2 * (kUngroupedSlotWords + kGroupSlotWords) * 8;
  u64 ok = 1;
  cudaIpcMemHandle_t mine;
  memset(&mine, 0, sizeof(mine));
  if (cudaMalloc((void**)&ctx->d_epoch, 8) != cudaSuccess || cudaMemset(ctx->d_epoch, 0, 8) != cudaSuccess) ok = 0;
  if (cudaMalloc((void**)&ctx->mbox, box_bytes) != cudaSuccess || cudaMemset(ctx->mbox, 0, box_bytes) != cudaSuccess ||
      cudaIpcGetMemHandle(&mine, ctx->mbox) != cudaSuccess)
    ok = 0;
  cudaGetLastError();
  unsigned char* d_handles = nullptr;
  u64* d_ok = nullptr;
  std::vector<cudaIpcMemHandle_t> all((size_t)N);
  if (cudaMalloc((void**)&d_handles, sizeof(mine) * (size_t)(N + 1)) != cudaSuccess || cudaMalloc((void**)&d_ok, 8) != cudaSuccess) {
    // without scratch memory the collectives below cannot run: every rank would need to know; give up on the whole setup
    if (d_handles) cudaFree(d_handles);
    comm_teardown_p2p(ctx);
    cudaGetLastError();
    return;
  }
  // all-gather the handles (the collective runs on every rank whatever `ok` says, so the ranks stay in step)
  cudaMemcpyAsync(d_handles + sizeof(mine) * (size_t)N, &mine, sizeof(mine), cudaMemcpyHostToDevice, ctx->stream);
  int nrc = g_nccl.all_gather(d_handles + sizeof(mine) * (size_t)N, d_handles, sizeof(mine), nccl_u8, ctx->nccl_comm, ctx->stream);
  cudaMemcpyAsync(all.data(), d_handles, sizeof(mine) * (size_t)N, cudaMemcpyDeviceToHost, ctx->stream);
  if (cudaStreamSynchronize(ctx->stream) != cudaSuccess || nrc != 0) ok = 0;
  if (ok) {
    for (int r = 0; r < N; ++r) {
      if (r == ctx->rank) {
        ctx->peer_mbox[r] = ctx->mbox;
        continue;
      }
      void* p = nullptr;
      if (cudaIpcOpenMemHandle(&p, all[(size_t)r], cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
        ok = 0;
        cudaGetLastError();
        break;
      }
      ctx->peer_mbox[r] = (u64*)p;
    }
  }
  // every rank or none
  cudaMemcpyAsync(d_ok, &ok, 8, cudaMemcpyHostToDevice, ctx->stream);
  nrc = g_nccl.all_reduce(d_ok, d_ok, 1, nccl_u64, nccl_min, ctx->nccl_comm, ctx->stream);
  u64 all_ok = 0;
  cudaMemcpyAsync(&all_ok, d_ok, 8, cudaMemcpyDeviceToHost, ctx->stream);
  if (cudaStreamSynchronize(ctx->stream) != cudaSuccess || nrc != 0) all_ok = 0;
  cudaFree(d_handles);
  cudaFree(d_ok);
  cudaGetLastError();
  if (all_ok) {
    ctx->p2p_merge = true;
    for (int r = 0; r < N; ++r) ctx->peer_gbox[r] = ctx->peer_mbox[r] + (size_t)N * 2 * kUngroupedSlotWords;
  } else comm_teardown_p2p(ctx);
  if (getenv("LLKV_GPU_VERBOSE"))
    fprintf(stderr, "[llkv] rank %d/%d: ungrouped merge over %s\n", ctx->rank, N, ctx->p2p_merge ? "NVLink peer mailboxes (CUDA IPC)" : "NCCL all-gather");
}

extern "C" int32_t llkv_gpu_comm_init(llkv_gpu_ctx* ctx, const uint8_t id[LLKV_GPU_UNIQUE_ID_BYTES], int32_t n_ranks, int32_t rank) {
  if (!ctx || !id) return set_error(LLKV_ERR_INVALID_ARGUMENT, "NULL argument");
  if (n_ranks < 1 || rank < 0 || rank >= n_ranks) return set_error(LLKV_ERR_INVALID_ARGUMENT, "bad rank %d of %d", rank, n_ranks);
  int32_t rc = load_nccl();
  if (rc) return rc;
  CTX_LOCK(ctx);
  CUDA_TRY(cudaSetDevice(ctx->device));
  if (ctx->nccl_comm) {
    g_nccl.comm_destroy(ctx->nccl_comm);
    ctx->nccl_comm = nullptr;
  }
  NcclIdByValue v;
  memcpy(v.internal, id, 128);
  NCCL_TRY(g_nccl.comm_init_rank(&ctx->nccl_comm, n_ranks, v, rank));
  ctx->n_ranks = n_ranks;
  ctx->rank = rank;
  ++ctx->state_epoch;
  comm_setup_p2p(ctx);
  return LLKV_OK;
}

static void comm_teardown_p2p(llkv_gpu_ctx* ctx) {
  for (int r = 0; r < 8; ++r) {
    if (ctx->peer_mbox[r] && r != ctx->rank) cudaIpcCloseMemHandle(ctx->peer_mbox[r]);
    ctx->peer_mbox[r] = nullptr;
    ctx->peer_gbox[r] = nullptr;
  }
  if (ctx->mbox) cudaFree(ctx->mbox);
  ctx->mbox = nullptr;
  ctx->p2p_merge = false;
  if (ctx->d_epoch) cudaFree(ctx->d_epoch);
  ctx->d_epoch = nullptr;
  cudaGetLastError();
}

extern "C" int32_t llkv_gpu_comm_destroy(llkv_gpu_ctx* ctx) {
  if (!ctx) return set_error(LLKV_ERR_INVALID_ARGUMENT, "ctx is NULL");
  CTX_LOCK(ctx);
  if (ctx->nccl_comm && g_nccl.comm_destroy) {
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    comm_teardown_p2p(ctx);
    g_nccl.comm_destroy(ctx->nccl_comm);
  }
  ctx->nccl_comm = nullptr;
  ctx->n_ranks = 1;
  ctx->rank = 0;
  ++ctx->state_epoch;
  return LLKV_OK;
}

// Every rank gathers every rank's partial table (allgather over NVLink) and folds them in rank order into a fresh
// table, so all ranks end with bit-identical states (f64 sums included).
// true when llkv_gpu_agg_merge of this aggregate is one kernel over the peer mailboxes (no collective, no host wait)
static bool merge_is_p2p(const llkv_gpu_agg* a) {
  const llkv_gpu_ctx* ctx = a->ctx;
  if (!a->frozen || !ctx->nccl_comm || ctx->n_ranks < 2 || !ctx->p2p_merge) return false;
  if (a->cr.plan.n_keys == 0) return !a->cr.can_narrow_fail && a->n_gwords < 127;
  if (!a->hint || a->p2p_group_disabled) return false;
  const u64 cap0 = group_table_cap(a->hint) * 4;
  return 2 + cap0 + (cap0 + 2) * (a->n_gwords + 1) <= kGroupSlotWords;
}

static int32_t agg_merge_impl(llkv_gpu_agg* a) {
  if (a->inner) return agg_merge_impl(a->inner);
  llkv_gpu_ctx* ctx = a->ctx;
  if (a->err_code) return set_error(a->err_code, "%s", a->err_msg.c_str());
  if (ctx->n_ranks > 1 && a->cr.plan.single_wide_key == 2)
    return set_error(LLKV_ERR_INVALID_ARGUMENT, "GROUP BY keys wider than 64 bits do not merge across GPUs: a group's key values are read from the shard that holds its first row");
  int32_t rc;
  if (!a->pending.active && (rc = agg_apply_reset(a))) return rc;
  if (ctx->nccl_comm && ctx->n_ranks > 1) {  // the merge works on the table on the device
    if (a->published && ((rc = agg_resolve(a)) || (rc = agg_unpublish(a)))) return rc;
    a->armed = false;
  }
  a->prefetched = false;  // the merge rewrites the table
  const int N = ctx->n_ranks;
  const int nccl_u64 = 5 /* ncclUint64 */, nccl_max = 2 /* ncclMax */;
  // Ungrouped state: the merge is queued behind the scan on the same stream without waiting for it (there is no table
  // to fill): peer-memory mailboxes over NVLink, or an all-gather of the one state row and one kernel.
  // (Every rank must take the same branch here: the condition only uses properties of the plan that do not depend on
  // the rank's data.  Whether the 64-bit run of THIS rank may still ask for a rerun does depend on its statistics, so
  // that is settled locally first.)
  if (a->frozen && a->cr.plan.n_keys == 0 && ctx->nccl_comm && N > 1) {
    if (a->cr.can_narrow_fail && (rc = agg_resolve(a))) return rc;
    if (!a->pending.active) {  // nothing left to settle from the run: the merge itself still has a status to report
      a->pending.active = true;
      a->pending.timed = false;
      a->pending.has_backup = false;
    }
    a->info.merged_p2p = ctx->p2p_merge && a->n_gwords < 127 ? 1 : 0;
    if (ctx->p2p_merge && a->n_gwords < 127) {  // NVLink peer stores + flags, no collective library on the path
      a->pending.timed_merge = ctx->timing;
      if (ctx->timing) CUDA_TRY(cudaEventRecord(ctx->ev2, ctx->stream));
      CUDA_TRY(launch_merge_ungrouped_p2p(a->gwords, ctx->peer_mbox, N, ctx->rank, a->n_gwords, ctx->d_epoch, a->d_gclass, a->d_flags,
                                          ctx->stream));
      if (ctx->timing) CUDA_TRY(cudaEventRecord(ctx->ev3, ctx->stream));
      return agg_queue_result_copy(a);  // (also the status word again: the merge kernel reports a peer that never arrives)
    }
    const size_t word_elems = (size_t)(3 * a->n_gwords);
    if (a->mg_word_elems < word_elems * (size_t)N) {
      if (a->mg_words) CUDA_TRY(cudaFree(a->mg_words));
      CUDA_TRY(cudaMalloc((void**)&a->mg_words, word_elems * 8 * (size_t)N));
      a->mg_word_elems = word_elems * (size_t)N;
    }
    NCCL_TRY(g_nccl.all_gather(a->gwords, a->mg_words, word_elems, nccl_u64, ctx->nccl_comm, ctx->stream));
    CUDA_TRY(launch_merge_ungrouped(a->gwords, a->mg_words, N, a->n_gwords, word_elems, a->d_gclass, ctx->stream));
    return agg_queue_result_copy(a);
  }
  // Small group tables (a cardinality hint that keeps the table within a mailbox slot even after growing x4): the same
  // peer-mailbox exchange, one kernel queued behind the scan, no collective, no host synchronisation.  The condition only
  // uses the hint and the accumulator layout, which every rank shares.
  if (a->frozen && a->cr.plan.n_keys != 0 && ctx->nccl_comm && N > 1 && ctx->p2p_merge && a->hint && !a->p2p_group_disabled) {
    const u64 cap0 = group_table_cap(a->hint) * 4;
    if (2 + cap0 + (cap0 + 2) * (a->n_gwords + 1) <= kGroupSlotWords) {
      if (!a->pending.active) {
        a->pending.active = true;
        a->pending.timed = false;
        a->pending.has_backup = false;
      }
      a->pending.is_merge = true;
      a->info.merged_p2p = 1;
      a->pending.timed_merge = ctx->timing;
      if (ctx->timing) CUDA_TRY(cudaEventRecord(ctx->ev2, ctx->stream));
      CUDA_TRY(launch_merge_grouped_p2p(a->gkeys, a->gwords, a->gcap, a->n_gwords, a->d_gclass, a->d_flags, ctx->peer_gbox, kGroupSlotWords, N, ctx->rank,
                                        ctx->d_epoch, true, ctx->stream));
      if (ctx->timing) CUDA_TRY(cudaEventRecord(ctx->ev3, ctx->stream));
      return agg_queue_result_copy(a);
    }
  }
  rc = agg_resolve(a);
  if (rc) return rc;
  if ((rc = agg_ensure_layout(a))) return rc;
  if (!ctx->nccl_comm || ctx->n_ranks == 1) return LLKV_OK;
  a->info.merged_p2p = 0;
  const bool grouped = a->cr.plan.n_keys != 0;
  if (grouped) {
    // all ranks must use one table size: agree on the largest
    if (!a->mg_cap) CUDA_TRY(cudaMalloc((void**)&a->mg_cap, 8));
    u64 cap = a->gcap;
    CUDA_TRY(cudaMemcpyAsync(a->mg_cap, &cap, 8, cudaMemcpyHostToDevice, ctx->stream));
    NCCL_TRY(g_nccl.all_reduce(a->mg_cap, a->mg_cap, 1, nccl_u64, nccl_max, ctx->nccl_comm, ctx->stream));
    CUDA_TRY(cudaMemcpyAsync(&cap, a->mg_cap, 8, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    while (a->gcap < cap)
      if ((rc = agg_grow_table(a))) return rc;
  }
  const u64 rows = a->gcap + 2;
  const size_t key_elems = (size_t)a->gcap, word_elems = (size_t)(rows * a->n_gwords);
  if (a->mg_key_elems < key_elems * (size_t)N) {
    if (a->mg_keys) CUDA_TRY(cudaFree(a->mg_keys));
    CUDA_TRY(cudaMalloc((void**)&a->mg_keys, key_elems * 8 * (size_t)N));
    a->mg_key_elems = key_elems * (size_t)N;
  }
  if (a->mg_word_elems < word_elems * (size_t)N) {
    if (a->mg_words) CUDA_TRY(cudaFree(a->mg_words));
    CUDA_TRY(cudaMalloc((void**)&a->mg_words, word_elems * 8 * (size_t)N));
    a->mg_word_elems = word_elems * (size_t)N;
  }
  u64* all_keys = a->mg_keys;
  u64* all_words = a->mg_words;
  if (grouped) NCCL_TRY(g_nccl.all_gather(a->gkeys, all_keys, key_elems, nccl_u64, ctx->nccl_comm, ctx->stream));
  NCCL_TRY(g_nccl.all_gather(a->gwords, all_words, word_elems, nccl_u64, ctx->nccl_comm, ctx->stream));
  CUDA_TRY(launch_init_table(a->gkeys, a->gwords, rows, a->n_gwords, a->d_gclass, ctx->stream));
  Plan mp = a->cr.plan;
  mp.gkeys = a->gkeys;
  mp.gwords = a->gwords;
  mp.gcap = a->gcap;
  mp.flags = a->d_flags;
  memcpy(a->h_plan, &mp, sizeof(Plan));  // the stream is idle here: agg_resolve synchronised it and nothing reads h_plan since
  CUDA_TRY(cudaMemcpyAsync(a->d_plan, a->h_plan, sizeof(Plan), cudaMemcpyHostToDevice, ctx->stream));
  const u64 src_cap = a->gcap;
  for (int attempt = 0; attempt < 16; ++attempt) {
    for (int r = 0; r < N; ++r)
      CUDA_TRY(launch_merge_table(a->d_plan, all_keys + (size_t)r * key_elems, all_words + (size_t)r * word_elems, src_cap, ctx->stream));
    CUDA_TRY(cudaMemcpyAsync(a->h_flags, a->d_flags, 4, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    if (!(*a->h_flags & FLAG_TABLE_FULL)) break;
    // the union of the ranks' groups outgrew the table: a larger, empty one, and fold everything again
    *a->h_flags = 0;
    CUDA_TRY(cudaMemsetAsync(a->d_flags, 0, 4, ctx->stream));
    CUDA_TRY(cudaFree(a->gkeys));
    CUDA_TRY(cudaFree(a->gwords));
    a->gkeys = a->gwords = nullptr;
    if ((rc = agg_alloc_table(a, a->gcap * 4))) return rc;
    mp.gkeys = a->gkeys;
    mp.gwords = a->gwords;
    mp.gcap = a->gcap;
    memcpy(a->h_plan, &mp, sizeof(Plan));
    CUDA_TRY(cudaMemcpyAsync(a->d_plan, a->h_plan, sizeof(Plan), cudaMemcpyHostToDevice, ctx->stream));
  }
  if ((rc = agg_queue_result_copy(a))) return rc;
  CUDA_TRY(cudaStreamSynchronize(ctx->stream));  // (no run is pending here: nothing else would wait for the copy)
  return LLKV_OK;
}

extern "C" int32_t llkv_gpu_agg_merge(llkv_gpu_agg* a) {
  if (!a) return set_error(LLKV_ERR_INVALID_ARGUMENT, "agg is NULL");
  CTX_LOCK(a->ctx);
  CUDA_TRY(cudaSetDevice(a->ctx->device));
  return agg_merge_impl(a);
}

// One step of a prepared aggregate: fresh accumulators -> fused scan of rows [row_begin, row_end) -> (merge != 0 and the
// context has peers) merge of the ranks' partial states -> result on its way to page-locked memory.  The same launches as
// reset + run + merge; once a step repeats with nothing changed (same columns, program, snapshot, row range, knobs; the
// previous steps came back clean) it is captured as a CUDA graph and replayed with a single launch call.
extern "C" int32_t llkv_gpu_agg_execute(llkv_gpu_agg* a, const llkv_gpu_program* prog, int32_t apply_mvcc, uint64_t row_begin, uint64_t row_end,
                                         int32_t merge) {
  if (!a) return set_error(LLKV_ERR_INVALID_ARGUMENT, "agg is NULL");
  if (row_end < row_begin) return set_error(LLKV_ERR_INVALID_ARGUMENT, "row_end < row_begin");
  if (a->inner) return llkv_gpu_agg_execute(a->inner, prog, apply_mvcc, row_begin, row_end, merge);
  llkv_gpu_ctx* ctx = a->ctx;
  CTX_LOCK(ctx);
  CUDA_TRY(cudaSetDevice(ctx->device));
  // reset: an unfinished step is dropped, its errors with it
  bool prev_clean = a->err_code == 0;
  if (a->pending.active) {
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    a->pending.active = false;
    prev_clean = false;  // never settled: whether it came back clean is unknown
  }
  a->err_code = 0;
  a->err_msg.clear();
  a->prefetched = false;
  *a->h_flags = 0;
  a->reset_pending = true;
  const bool do_merge = merge != 0 && ctx->nccl_comm && ctx->n_ranks > 1;
  uint64_t key = 0xcbf29ce484222325ull;
  {
    const uint64_t parts[8] = {ctx->state_epoch, a->plan_epoch, prog ? prog->serial : 0, (uint64_t)apply_mvcc, row_begin, row_end, (uint64_t)do_merge,
                               (uint64_t)ctx->timing};
    key = fnv1a(key, parts, sizeof(parts));
    if (!key) key = 1;
  }
  if (a->graph_exec && a->graph_key == key && prev_clean && (!a->graph_from_armed || a->armed)) {
    const PendingRun& gp = a->graph_pending;  // (the program copy of the captured step is still in a->pending.prog)
    a->pending.has_prog = gp.has_prog;
    a->pending.apply_mvcc = gp.apply_mvcc;
    a->pending.row_begin = gp.row_begin;
    a->pending.row_end = gp.row_end;
    a->pending.wide = gp.wide;
    a->pending.has_backup = gp.has_backup;
    a->pending.timed = gp.timed;
    a->pending.is_merge = gp.is_merge;
    a->pending.timed_merge = gp.timed_merge;
    a->reset_pending = false;  // part of the graph
    CUDA_TRY(cudaGraphLaunch(a->graph_exec, ctx->stream));
    ++a->info.graph_replays;
    if (a->graph_published) ++a->info.published_steps;
    a->prefetched = a->graph_prefetched;
    a->published = a->graph_published;
    a->armed = a->graph_armed_after;
    a->stage_ev_valid = false;
    a->pending.active = true;
    a->info.kernel_launches = a->graph_launches;
    return LLKV_OK;
  }
  if (a->exec_key == key && prev_clean) ++a->exec_same;
  else a->exec_same = 0;
  a->exec_key = key;
  // capture on the third unchanged step: by then the plan is compiled and specialised, statistics, zone maps and tile
  // lists are settled and every buffer is allocated, so the step is launches and asynchronous copies only
  const bool capture = ctx->graph_mode && a->exec_same >= 2 && a->capture_failures < 2 && a->frozen && a->cr.fast && (!do_merge || merge_is_p2p(a));
  if (capture) {
    if (a->graph_exec) {
      cudaGraphExecDestroy(a->graph_exec);
      a->graph_exec = nullptr;
      a->graph_key = 0;
    }
    a->in_capture = true;
    const bool armed_before = a->armed;
    const uint32_t published_before = a->info.published_steps;
    cudaError_t e = cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeThreadLocal);
    int32_t rc = LLKV_OK;
    if (e == cudaSuccess) {
      a->skip_scan_copy = do_merge;  // (capturing implies merge_is_p2p: the merge queues the copies)
      rc = agg_run_impl(a, prog, apply_mvcc, row_begin, row_end);
      a->skip_scan_copy = false;
      if (!rc && do_merge) rc = agg_merge_impl(a);
      cudaGraph_t graph = nullptr;
      e = cudaStreamEndCapture(ctx->stream, &graph);
      if (e == cudaSuccess && !rc && graph) {
        e = cudaGraphInstantiate(&a->graph_exec, graph, 0);
        if (e == cudaSuccess) e = cudaGraphLaunch(a->graph_exec, ctx->stream);  // (capturing executed nothing)
      } else if (e == cudaSuccess && rc) {
        e = cudaErrorUnknown;
      }
      if (graph) cudaGraphDestroy(graph);
    }
    a->in_capture = false;
    if (e == cudaSuccess && !rc) {
      a->graph_key = key;
      a->graph_pending = a->pending;
      a->graph_pending.prog = llkv_gpu_program();
      a->graph_prefetched = a->prefetched;
      a->graph_from_armed = armed_before;
      a->graph_published = a->published;
      a->graph_armed_after = a->armed;
      a->graph_launches = a->info.kernel_launches;
      a->stage_ev_valid = false;
      return LLKV_OK;
    }
    // the step is not capturable as it is (something in it waits for the device): run it the plain way, from scratch
    if (getenv("LLKV_GPU_VERBOSE"))
      fprintf(stderr, "[llkv] rank %d: step not captured as a CUDA graph: %s (rc %d: %s)\n", ctx->rank, cudaGetErrorString(e), rc, rc ? g_last_error.c_str() : "-");
    cudaGetLastError();
    if (a->graph_exec) cudaGraphExecDestroy(a->graph_exec);
    a->graph_exec = nullptr;
    a->graph_key = 0;
    ++a->capture_failures;
    a->pending.active = false;
    a->prefetched = false;
    a->published = false;
    a->info.published_steps = published_before;  // (the captured scan never ran; the plain run below counts the step)
    a->armed = false;  // (the captured resets never ran)
    a->reset_pending = true;
    cudaStreamSynchronize(ctx->stream);
    cudaGetLastError();
  }
  a->skip_scan_copy = do_merge && merge_is_p2p(a);
  int32_t rc = agg_run_impl(a, prog, apply_mvcc, row_begin, row_end);
  a->skip_scan_copy = false;
  if (!rc && do_merge) rc = agg_merge_impl(a);
  return rc;
}

extern "C" int32_t llkv_gpu_ctx_set_graphs(llkv_gpu_ctx* c, int32_t mode) {
  if (!c) return set_error(LLKV_ERR_INVALID_ARGUMENT, "ctx is NULL");
  if (mode < 0 || mode > 1) return set_error(LLKV_ERR_INVALID_ARGUMENT, "graph mode must be 0 or 1");
  CTX_LOCK(c);
  c->graph_mode = mode;
  return LLKV_OK;
}

// common.cuh -- shared device/host helpers for the arrow_b200 kernels.
//
// Layout rules every kernel follows (Arrow columnar format, as consumed by the
// reference through ArraySpan, cpp/src/arrow/array/data.h:525-690):
//   * validity and boolean data are LSB-first bitmaps addressed in BITS with the
//     array's `offset`; they may start at any bit of any byte,
//   * fixed-width values start at data + offset * width,
//   * bits/bytes past `length` in an output buffer are written as zero.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/arrow_b200.h"

namespace b2 {

constexpr int kBlock = 256;          // threads per CTA for the streaming kernels
constexpr int kWarpsPerBlock = kBlock / 32;
constexpr int kSMs = 148;            // B200: 2 dies x 74 SMs

// ---------------------------------------------------------------------------
// Bitmap reader: logical bit i of the array lives at absolute bit (bit0 + i) of
// an 8-byte aligned base.  word(w) returns logical bits [64w, 64w+64) with bits at
// or past nbits cleared.  A NULL bitmap reads as all-valid.  Only aligned 64-bit
// words that contain at least one addressed byte are ever dereferenced.
// ---------------------------------------------------------------------------
struct BitmapReader {
  const uint64_t* base;
  int64_t bit0;
  int64_t nbits;

  __host__ __device__ BitmapReader() : base(nullptr), bit0(0), nbits(0) {}
  __host__ __device__ BitmapReader(const void* bits, int64_t offset, int64_t length) {
    if (bits == nullptr) {
      base = nullptr;
      bit0 = 0;
    } else {
      uintptr_t p = reinterpret_cast<uintptr_t>(bits);
      // offset may be large: fold whole bytes into the pointer first
      p += static_cast<uintptr_t>(offset >> 3);
      int64_t bit = offset & 7;
      uintptr_t aligned = p & ~static_cast<uintptr_t>(7);
      bit += static_cast<int64_t>(p - aligned) * 8;
      base = reinterpret_cast<const uint64_t*>(aligned);
      bit0 = bit;  // 0..63
    }
    nbits = length;
  }
  __device__ __forceinline__ bool present() const { return base != nullptr; }

  __device__ __forceinline__ uint64_t word(int64_t w) const {
    int64_t rem = nbits - (w << 6);
    if (rem <= 0) return 0;
    uint64_t r;
    if (base == nullptr) {
      r = ~0ull;
    } else {
      int64_t start = bit0 + (w << 6);
      int64_t i = start >> 6;
      int sh = static_cast<int>(start & 63);
      uint64_t lo = __ldg(base + i);
      if (sh == 0) {
        r = lo;
      } else {
        r = lo >> sh;
        // bits available from lo: 64 - sh; need the next word only if rem exceeds that
        if (rem > 64 - sh) r |= __ldg(base + i + 1) << (64 - sh);
      }
    }
    if (rem < 64) r &= (1ull << rem) - 1ull;
    return r;
  }
  // 32-bit logical word v: bits [32v, 32v+32)
  __device__ __forceinline__ uint32_t word32(int64_t v) const {
    uint64_t w = word(v >> 1);
    return static_cast<uint32_t>((v & 1) ? (w >> 32) : w);
  }
  __device__ __forceinline__ bool bit(int64_t i) const {
    if (base == nullptr) return true;
    int64_t a = bit0 + i;
    return (__ldg(reinterpret_cast<const uint8_t*>(base) + (a >> 3)) >> (a & 7)) & 1;
  }
  // random-access variant: the byte load carries an L2 cache policy (see l2_policy_*)
  __device__ __forceinline__ bool bit_hint(int64_t i, uint64_t policy) const {
    if (base == nullptr) return true;
    int64_t a = bit0 + i;
    uint32_t v;
    asm volatile("ld.global.nc.L2::cache_hint.u8 %0, [%1], %2;"
                 : "=r"(v)
                 : "l"(reinterpret_cast<const uint8_t*>(base) + (a >> 3)), "l"(policy));
    return (v >> (a & 7)) & 1;
  }
};

__host__ __device__ inline int64_t bitmap_bytes(int64_t nbits) { return (nbits + 7) >> 3; }
__host__ __device__ inline int64_t bitmap_words64(int64_t nbits) { return (nbits + 63) >> 6; }
// output bitmaps are allocated in whole 64-bit words so kernels can store words
__host__ __device__ inline int64_t bitmap_alloc_bytes(int64_t nbits) {
  return bitmap_words64(nbits) * 8 + 8;
}

__host__ __device__ inline int type_width(int t) {
  switch (t) {
    case B2_UINT8: case B2_INT8: return 1;
    case B2_UINT16: case B2_INT16: case B2_HALF_FLOAT: return 2;
    case B2_UINT32: case B2_INT32: case B2_FLOAT: return 4;
    case B2_UINT64: case B2_INT64: case B2_DOUBLE: return 8;
    default: return 0;
  }
}
__host__ __device__ inline bool type_is_numeric(int t) {
  return t >= B2_UINT8 && t <= B2_DOUBLE && t != B2_HALF_FLOAT;
}
__host__ __device__ inline bool type_is_binary_like(int t) {
  return t == B2_STRING || t == B2_BINARY || t == B2_LARGE_STRING || t == B2_LARGE_BINARY;
}
__host__ __device__ inline int offset_width(int t) {
  return (t == B2_LARGE_STRING || t == B2_LARGE_BINARY) ? 8 : 4;
}

// ---------------------------------------------------------------------------
// streaming loads/stores: these columns are read or written exactly once, so
// keep them out of L1 (ld.global.nc.L1::no_allocate) -- guide, Guideline 13.
// ---------------------------------------------------------------------------
template <typename T>
__device__ __forceinline__ T ld_stream(const T* p) {
  return __ldcs(p);
}
template <typename T>
__device__ __forceinline__ void st_stream(T* p, T v) {
  __stcs(p, v);
}

// ---------------------------------------------------------------------------
// L2 residency hints for random-access kernels (gather, hash tables): the big,
// touched-once structure is loaded evict-first and the small hot one (a validity
// bitmap, a hash-table slot array) evict-last, so the 126 MB L2 keeps the latter.
// ---------------------------------------------------------------------------
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
  uint64_t p;
  asm("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
  uint64_t p;
  asm("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ uint32_t ld_hint_u8(const uint8_t* p, uint64_t pol) {
  uint32_t v;
  asm volatile("ld.global.nc.L2::cache_hint.u8 %0, [%1], %2;" : "=r"(v) : "l"(p), "l"(pol));
  return v;
}
template <typename T>
__device__ __forceinline__ T ld_hint(const T* p, uint64_t pol) {
  T out;
  if constexpr (sizeof(T) == 1) {
    uint32_t v;
    asm volatile("ld.global.nc.L2::cache_hint.u8 %0, [%1], %2;" : "=r"(v) : "l"(p), "l"(pol));
    uint8_t b = static_cast<uint8_t>(v);
    memcpy(&out, &b, 1);
  } else if constexpr (sizeof(T) == 2) {
    uint16_t v;
    asm volatile("ld.global.nc.L2::cache_hint.u16 %0, [%1], %2;" : "=h"(v) : "l"(p), "l"(pol));
    memcpy(&out, &v, 2);
  } else if constexpr (sizeof(T) == 4) {
    uint32_t v;
    asm volatile("ld.global.nc.L2::cache_hint.u32 %0, [%1], %2;" : "=r"(v) : "l"(p), "l"(pol));
    memcpy(&out, &v, 4);
  } else if constexpr (sizeof(T) == 8) {
    uint64_t v;
    asm volatile("ld.global.nc.L2::cache_hint.u64 %0, [%1], %2;" : "=l"(v) : "l"(p), "l"(pol));
    memcpy(&out, &v, 8);
  } else {
    uint4 v;
    asm volatile("ld.global.nc.L2::cache_hint.v4.u32 {%0,%1,%2,%3}, [%4], %5;"
                 : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p), "l"(pol));
    memcpy(&out, &v, 16);
  }
  return out;
}

// nbytes (1..8) bytes at p, little-endian, zero-extended; funnel-shifts two aligned 8-byte loads, and only aligned
// words holding an addressed byte are dereferenced, so it never reads past the word holding a buffer's last byte
__device__ __forceinline__ uint64_t load_bytes8(const uint8_t* p, int nbytes) {
  const uintptr_t u = reinterpret_cast<uintptr_t>(p);
  const uint64_t* a = reinterpret_cast<const uint64_t*>(u & ~uintptr_t(7));
  const int skip = static_cast<int>(u & 7);
  uint64_t v = __ldg(a) >> (skip * 8);
  if (skip && 8 - skip < nbytes) v |= __ldg(a + 1) << (64 - skip * 8);
  if (nbytes < 8) v &= (1ull << (8 * nbytes)) - 1ull;
  return v;
}

__device__ __forceinline__ unsigned lane_id() { return threadIdx.x & 31; }
__device__ __forceinline__ unsigned lanemask_lt() {
  unsigned m;
  asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
  return m;
}

// block-wide sum of an int64 (all threads must call); result valid in thread 0
template <int BLOCK>
__device__ __forceinline__ int64_t block_sum(int64_t v) {
  __shared__ int64_t warp_sums[BLOCK / 32];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  if (lane_id() == 0) warp_sums[threadIdx.x >> 5] = v;
  __syncthreads();
  int64_t r = 0;
  if (threadIdx.x < 32) {
    r = threadIdx.x < BLOCK / 32 ? warp_sums[threadIdx.x] : 0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) r += __shfl_down_sync(0xffffffffu, r, o);
  }
  return r;
}

inline bool aligned_to(const void* p, size_t a) { return (reinterpret_cast<uintptr_t>(p) % a) == 0; }

// grid sizing: enough CTAs for `resident` CTAs on each of the 148 SMs and a whole
// number of waves when the work is large (guide, Guideline 11).
inline int grid_for(int64_t work_items, int64_t items_per_block, int max_waves_blocks) {
  int64_t b = (work_items + items_per_block - 1) / items_per_block;
  if (b < 1) b = 1;
  if (b > max_waves_blocks) b = max_waves_blocks;
  return static_cast<int>(b);
}

// Decoupled look-back over one column of a [tile][stride] table of 32-bit cells
// (bits 31:30 = 0 not published / 1 tile aggregate / 2 inclusive prefix, bits 29:0 = count):
// returns the exclusive prefix of `tile`.  Four predecessor cells are requested per step so
// the walk costs one L2 round trip per four tiles instead of one per tile.
__device__ __forceinline__ uint32_t lookback_exclusive(const volatile uint32_t* col, int64_t tile, size_t stride) {
  uint32_t excl = 0;
  int64_t t = tile - 1;
  while (t >= 0) {
    uint32_t c[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) c[k] = (t - k >= 0) ? col[static_cast<size_t>(t - k) * stride] : (2u << 30);
    bool done = false;
    int used = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const uint32_t f = c[k] >> 30;
      if (!done && used == k && f != 0) {
        excl += c[k] & 0x3fffffffu;
        ++used;
        done = f == 2;
      }
    }
    if (done) break;
    t -= used;  // poll again from the first cell that was not published yet
  }
  return excl;
}

// 64-bit-cell variant for columns of 2^30 rows or more (bits 63:62 = flag, bits 61:0 = count)
__device__ __forceinline__ unsigned long long lookback_exclusive64(const volatile unsigned long long* col, int64_t tile, size_t stride) {
  unsigned long long excl = 0;
  int64_t t = tile - 1;
  while (t >= 0) {
    unsigned long long c[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) c[k] = (t - k >= 0) ? col[static_cast<size_t>(t - k) * stride] : (2ull << 62);
    bool done = false;
    int used = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const unsigned f = static_cast<unsigned>(c[k] >> 62);
      if (!done && used == k && f != 0) {
        excl += c[k] & 0x3fffffffffffffffull;
        ++used;
        done = f == 2;
      }
    }
    if (done) break;
    t -= used;
  }
  return excl;
}

}  // namespace b2

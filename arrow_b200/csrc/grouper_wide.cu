// grouper_wide.cu -- Grouper over utf8 / binary key columns and over keys wider than 64 bits.
//
// Replaces, for those key shapes, what GrouperFastImpl does with its row encoding
// (compute/row/grouper.cc:555-963; compute/row/encode_internal.cc: fixed-width columns packed into a row,
// var-length columns appended behind an offset table; Hashing32 over the encoded row, key_hash.cc) and what
// GrouperImpl does for the types the fast path refuses (row/grouper.cc:300-553: a std::string per row).
// Semantics kept: one dense uint32 id per row, a null key value is a value of its own, keys group by BYTES,
// uniques grow by appending, Lookup never inserts and yields null for unknown keys.  As in grouper.cu the ids are
// assigned in first-occurrence row order.
//
// B200 design: no row encoding and no per-row key tuple ever exists in HBM.  The key columns are cut into PARTS --
// runs of fixed-width columns whose packed encoding fits 64 bits, and single utf8/binary columns -- and every part
// is reduced to dense 32-bit ids on its own:
//   * a fixed-width part is the 64-bit grouper of grouper.cu (16-byte slots, one sector per probe);
//   * a string part hashes every value to 64 bits (aligned 8-byte loads, funnel-shifted), groups the HASHES with
//     the same 64-bit grouper (which also reports the rows where new groups first occur -- its own first-occurrence
//     flags), appends those first occurrences to a string store (b2_take), and then VERIFIES
//     every row of the batch against the store entry of its id, byte for byte.  A verified batch is exact; a
//     mismatch (two different strings with one 64-bit hash) rolls the batch back, re-seeds the hash, rebuilds the
//     part from its store and repeats -- results never depend on the hash.
// Parts are then folded left to right: (ids so far, ids of the next part) packed into one uint64 is itself a
// 64-bit key without nulls, so the fold is again the kernel of grouper.cu.  Because each level is a bijection
// between key tuples and ids, the final ids are exactly those a single wide table would have produced, in the
// same first-occurrence order.  GetUniques unfolds the levels with b2_take.
#include <cstdlib>
#include <vector>

#include "bitmap.h"
#include "common.cuh"
#include "context.h"

namespace b2 {

void grouper_never_direct(B2Grouper* g);  // grouper.cu
int grouper_consume_new_rows(B2Grouper* g, const B2Array* keys, B2Array* out_ids, B2Array* out_new_rows, cudaStream_t s);

namespace {

// a C-ABI output whose buffers go back to the pool unless released
struct Owned {
  B2Context* ctx;
  cudaStream_t s;
  B2Array a{};
  Owned(B2Context* c, cudaStream_t st) : ctx(c), s(st) {}
  Owned(const Owned&) = delete;
  Owned& operator=(const Owned&) = delete;
  ~Owned() { reset(); }
  void reset() {
    if (a.validity) ctx->free(const_cast<void*>(a.validity), s);
    if (a.data) ctx->free(const_cast<void*>(a.data), s);
    if (a.data2) ctx->free(const_cast<void*>(a.data2), s);
    a = B2Array{};
  }
  void give(B2Array* out) {
    *out = a;
    a = B2Array{};
  }
};

__device__ __forceinline__ uint64_t mix64(uint64_t h) {
  h ^= h >> 30;
  h *= 0xbf58476d1ce4e5b9ull;
  h ^= h >> 27;
  h *= 0x94d049bb133111ebull;
  h ^= h >> 31;
  return h;
}

__device__ __forceinline__ uint64_t hash_bytes(const uint8_t* p, int64_t len, uint64_t seed) {
  uint64_t h = seed ^ (static_cast<uint64_t>(len) * 0xff51afd7ed558ccdull);
  for (int64_t o = 0; o < len; o += 8) {
    const int nb = len - o >= 8 ? 8 : static_cast<int>(len - o);
    h = (h ^ load_bytes8(p + o, nb)) * 0x9e3779b97f4a7c15ull;
    h ^= h >> 29;
  }
  return mix64(h);
}

__device__ __forceinline__ bool bytes_equal(const uint8_t* a, const uint8_t* b, int64_t len) {
  for (int64_t o = 0; o < len; o += 8) {
    const int nb = len - o >= 8 ? 8 : static_cast<int>(len - o);
    if (load_bytes8(a + o, nb) != load_bytes8(b + o, nb)) return false;
  }
  return true;
}

constexpr uint64_t kNullHash = 0x6e756c6c6b657921ull;

// hash of every value; a null value hashes to a constant (verification keeps real strings apart from it).
// null_bytes (store rows) overrides the validity bitmap (batch rows).
template <typename OffT>
__global__ void __launch_bounds__(kBlock) hash_strings_kernel(const OffT* __restrict__ offs, const uint8_t* __restrict__ bytes,
                                                              BitmapReader valid, const uint8_t* __restrict__ null_bytes,
                                                              int64_t n, uint64_t seed, uint64_t mask, uint64_t* __restrict__ out) {
  for (int64_t i = blockIdx.x * (int64_t)kBlock + threadIdx.x; i < n; i += (int64_t)gridDim.x * kBlock) {
    const bool is_null = null_bytes ? null_bytes[i] != 0 : !valid.bit(i);
    uint64_t h;
    if (is_null) {
      h = mix64(kNullHash ^ seed);
    } else {
      const int64_t o0 = static_cast<int64_t>(offs[i]);
      h = hash_bytes(bytes + o0, static_cast<int64_t>(offs[i + 1]) - o0, seed);
    }
    out[i] = h & mask;
  }
}

// One 32-byte record per stored value = ONE L2 sector per verification: word 0 = length (bit 31: the null value), then the
// first 28 bytes zero-padded.  The verify pass is bound by random L2 requests (211 G/s measured, bench_micro/gather_probe),
// and {null flag, two offsets, the bytes} were four to five of them per row; values longer than 28 bytes fetch their
// tail from the byte store.
constexpr int kRecBytes = 28;
constexpr uint32_t kRecNull = 0x80000000u;

// append the taken first occurrences (offsets start at taken_off[0]) behind group `base`
template <typename OffT>
__global__ void __launch_bounds__(kBlock) store_append_kernel(const OffT* __restrict__ taken_off, const uint8_t* __restrict__ taken_bytes,
                                                              BitmapReader taken_valid, int64_t n_new, int64_t byte_base, int64_t* store_off,
                                                              uint8_t* store_null, uint4* store_rec, uint32_t base) {
  const int64_t o0 = static_cast<int64_t>(taken_off[0]);
  for (int64_t i = blockIdx.x * (int64_t)kBlock + threadIdx.x; i < n_new; i += (int64_t)gridDim.x * kBlock) {
    const int64_t b0 = static_cast<int64_t>(taken_off[i]), b1 = static_cast<int64_t>(taken_off[i + 1]);
    const bool is_null = !taken_valid.bit(i);
    store_off[base + i + 1] = byte_base + b1 - o0;
    store_null[base + i] = is_null ? 1 : 0;
    uint32_t w[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    const int64_t len = b1 - b0;
    w[0] = is_null ? kRecNull : static_cast<uint32_t>(len > 0x7fffffff ? 0x7fffffff : len);
    const int head = len < kRecBytes ? static_cast<int>(len) : kRecBytes;
    for (int k = 0; k < head; ++k) w[1 + (k >> 2)] |= static_cast<uint32_t>(taken_bytes[b0 + k]) << (8 * (k & 3));
    store_rec[2 * (base + i)] = make_uint4(w[0], w[1], w[2], w[3]);
    store_rec[2 * (base + i) + 1] = make_uint4(w[4], w[5], w[6], w[7]);
  }
}

// every row against the store entry of its id.  Consume: counts the mismatches.  Lookup (out_validity != NULL):
// ids_valid says which rows found a hash; a row whose bytes differ is unknown, not an error.
template <typename OffT>
__global__ void __launch_bounds__(kBlock) verify_kernel(const OffT* __restrict__ offs, const uint8_t* __restrict__ bytes,
                                                        BitmapReader valid, int64_t n, const uint32_t* __restrict__ ids,
                                                        BitmapReader ids_valid, const int64_t* __restrict__ store_off,
                                                        const uint8_t* __restrict__ store_bytes,
                                                        const uint4* __restrict__ store_rec, uint32_t* out_validity,
                                                        int64_t* counter) {
  const int64_t nw = (n + 31) >> 5;
  int64_t local = 0;
  for (int64_t w = (blockIdx.x * (int64_t)kBlock + threadIdx.x) >> 5; w < nw; w += ((int64_t)gridDim.x * kBlock) >> 5) {
    const int64_t i = (w << 5) + lane_id();
    bool match = false, known = false;
    if (i < n) {
      known = out_validity ? ids_valid.bit(i) : true;
      if (known) {
        const uint32_t g = ids[i];
        const uint4 r0 = __ldg(store_rec + 2 * static_cast<int64_t>(g)), r1 = __ldg(store_rec + 2 * static_cast<int64_t>(g) + 1);
        const bool rnull = !valid.bit(i);
        if (rnull || r0.x == kRecNull) {
          match = rnull && r0.x == kRecNull;
        } else {
          const int64_t o0 = static_cast<int64_t>(offs[i]), len = static_cast<int64_t>(offs[i + 1]) - o0;
          match = static_cast<int64_t>(r0.x) == len || (r0.x == 0x7fffffffu && len >= 0x7fffffff);
          if (match) {
            const uint32_t rw[7] = {r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w};
            const int64_t head = len < kRecBytes ? len : kRecBytes;
            for (int64_t o = 0; o < head && match; o += 8) {
              const int nb = head - o >= 8 ? 8 : static_cast<int>(head - o);
              const int k = static_cast<int>(o >> 2);
              uint64_t want = rw[k] | (nb > 4 ? static_cast<uint64_t>(rw[k + 1]) << 32 : 0ull);
              if (nb < 8) want &= (1ull << (8 * nb)) - 1ull;
              match = load_bytes8(bytes + o0 + o, nb) == want;
            }
            if (match && len > kRecBytes) {  // the tail lives in the byte store
              const int64_t s0 = store_off[g];
              match = (store_off[g + 1] - s0 == len) && bytes_equal(bytes + o0 + kRecBytes, store_bytes + s0 + kRecBytes, len - kRecBytes);
            }
          }
        }
      }
    }
    if (out_validity) {
      const unsigned word = __ballot_sync(0xffffffffu, known && match);
      if (lane_id() == 0) {
        out_validity[w] = word;
        local += __popc(word);
      }
    } else {
      const unsigned word = __ballot_sync(0xffffffffu, i < n && !match);
      if (lane_id() == 0) local += __popc(word);
    }
  }
  const int64_t s = block_sum<kBlock>(local);
  if (threadIdx.x == 0 && s) atomicAdd(reinterpret_cast<unsigned long long*>(counter), (unsigned long long)s);
}

__global__ void __launch_bounds__(kBlock) count_not_iota_kernel(const uint32_t* __restrict__ ids, int64_t n, int64_t* counter) {
  int64_t local = 0;
  for (int64_t i = blockIdx.x * (int64_t)kBlock + threadIdx.x; i < n; i += (int64_t)gridDim.x * kBlock)
    local += ids[i] != static_cast<uint32_t>(i);
  const int64_t s = block_sum<kBlock>(local);
  if (threadIdx.x == 0 && s) atomicAdd(reinterpret_cast<unsigned long long*>(counter), (unsigned long long)s);
}

__global__ void __launch_bounds__(kBlock) pack_pair_kernel(const uint32_t* __restrict__ a, const uint32_t* __restrict__ b, int64_t n,
                                                           uint64_t* __restrict__ out) {
  for (int64_t i = blockIdx.x * (int64_t)kBlock + threadIdx.x; i < n; i += (int64_t)gridDim.x * kBlock)
    out[i] = (static_cast<uint64_t>(a[i]) << 32) | b[i];
}

__global__ void __launch_bounds__(kBlock) unpack_pair_kernel(const uint64_t* __restrict__ in, int64_t n, uint32_t* __restrict__ a,
                                                             uint32_t* __restrict__ b) {
  for (int64_t i = blockIdx.x * (int64_t)kBlock + threadIdx.x; i < n; i += (int64_t)gridDim.x * kBlock) {
    const uint64_t v = in[i];
    a[i] = static_cast<uint32_t>(v >> 32);
    b[i] = static_cast<uint32_t>(v);
  }
}

__global__ void __launch_bounds__(kBlock) null_bytes_to_bitmap_kernel(const uint8_t* __restrict__ nulls, int64_t n, uint32_t* out_validity) {
  const int64_t nw = (n + 31) >> 5;
  for (int64_t w = (blockIdx.x * (int64_t)kBlock + threadIdx.x) >> 5; w < nw; w += ((int64_t)gridDim.x * kBlock) >> 5) {
    const int64_t i = (w << 5) + lane_id();
    const unsigned word = __ballot_sync(0xffffffffu, i < n && nulls[i] == 0);
    if (lane_id() == 0) out_validity[w] = word;
  }
}

template <typename OffT>
__global__ void __launch_bounds__(kBlock) narrow_offsets_kernel(const int64_t* __restrict__ in, int64_t n, OffT* __restrict__ out) {
  for (int64_t i = blockIdx.x * (int64_t)kBlock + threadIdx.x; i < n; i += (int64_t)gridDim.x * kBlock) out[i] = static_cast<OffT>(in[i]);
}

inline int grid1(int64_t n) { return grid_for(n, kBlock * 4, kSMs * 8); }

B2Array u32_array(const void* data, int64_t n, const void* validity = nullptr, int64_t nulls = 0) {
  B2Array a{};
  a.type = B2_UINT32;
  a.data = data;
  a.length = n;
  a.validity = validity;
  a.null_count = nulls;
  return a;
}

B2Array u64_array(const void* data, int64_t n, const void* validity = nullptr, int64_t nulls = 0) {
  B2Array a = u32_array(data, n, validity, nulls);
  a.type = B2_UINT64;
  return a;
}

// ---- one utf8 / binary column -> dense ids -------------------------------------------------------------------------
struct StringPart {
  B2Context* ctx;
  int32_t type;
  B2Grouper* inner = nullptr;  // 64-bit grouper over the hashes (no nulls: a null value has a hash of its own)
  uint64_t seed = 0x243f6a8885a308d3ull;
  int hash_bits = 64;  // B2_GROUPER_HASH_BITS narrows the first attempts so tests reach the collision path
  // store of the distinct values in id order
  int64_t* off = nullptr;  // [cap_groups + 1]
  uint8_t* is_null = nullptr;
  uint4* rec = nullptr;  // [2 * cap_groups]: the 32-byte verification records
  uint8_t* bytes = nullptr;
  uint64_t cap_groups = 0, cap_bytes = 0;
  uint32_t n = 0;
  int64_t n_bytes = 0;
  bool has_null = false;

  bool large() const { return offset_width(type) == 8; }
  uint64_t mask() const { return hash_bits >= 64 ? ~0ull : ((1ull << hash_bits) - 1ull); }

  int init() {
    const int32_t kt = B2_UINT64;
    if (const char* e = getenv("B2_GROUPER_HASH_BITS")) {
      hash_bits = static_cast<int>(strtol(e, nullptr, 10));
      if (hash_bits < 1 || hash_bits > 64) hash_bits = 64;
    }
    B2_RETURN_NOT_OK(b2_grouper_create(ctx, &kt, 1, &inner));
    grouper_never_direct(inner);
    return B2_OK;
  }
  void destroy(cudaStream_t s) {
    if (inner) b2_grouper_destroy(inner);
    if (off) ctx->free(off, s);
    if (is_null) ctx->free(is_null, s);
    if (rec) ctx->free(rec, s);
    if (bytes) ctx->free(bytes, s);
  }
  int reset() {
    n = 0;
    n_bytes = 0;
    has_null = false;
    return b2_grouper_reset(inner);
  }

  int reserve(uint64_t groups, uint64_t nbytes, cudaStream_t s) {
    if (groups > cap_groups || !off) {
      uint64_t cap = 1024;
      while (cap < groups) cap <<= 1;
      void *o, *nl, *rc;
      B2_RETURN_NOT_OK(ctx->alloc((cap + 1) * 8, &o, s));
      B2_RETURN_NOT_OK(ctx->alloc(cap, &nl, s));
      B2_RETURN_NOT_OK(ctx->alloc(cap * 32, &rc, s));
      if (off) {
        B2_CUDA(cudaMemcpyAsync(o, off, ((size_t)n + 1) * 8, cudaMemcpyDeviceToDevice, s));
        B2_CUDA(cudaMemcpyAsync(nl, is_null, n, cudaMemcpyDeviceToDevice, s));
        B2_CUDA(cudaMemcpyAsync(rc, rec, (size_t)n * 32, cudaMemcpyDeviceToDevice, s));
        ctx->free(off, s);
        ctx->free(is_null, s);
        ctx->free(rec, s);
      } else {
        B2_CUDA(cudaMemsetAsync(o, 0, 8, s));
      }
      off = static_cast<int64_t*>(o);
      is_null = static_cast<uint8_t*>(nl);
      rec = static_cast<uint4*>(rc);
      cap_groups = cap;
    }
    if (nbytes > cap_bytes || !bytes) {
      uint64_t cap = 4096;
      while (cap < nbytes) cap <<= 1;
      void* b;
      B2_RETURN_NOT_OK(ctx->alloc(cap + 16, &b, s));
      if (bytes) {
        if (n_bytes) B2_CUDA(cudaMemcpyAsync(b, bytes, (size_t)n_bytes, cudaMemcpyDeviceToDevice, s));
        ctx->free(bytes, s);
      }
      bytes = static_cast<uint8_t*>(b);
      cap_bytes = cap;
    }
    return B2_OK;
  }

  template <typename OffT>
  int hash_batch(const B2Array* col, uint64_t* out, cudaStream_t s) const {
    const int64_t n_rows = col->length;
    hash_strings_kernel<OffT><<<grid1(n_rows), kBlock, 0, s>>>(
        static_cast<const OffT*>(col->data) + col->offset, static_cast<const uint8_t*>(col->data2),
        BitmapReader(col->null_count == 0 ? nullptr : col->validity, col->offset, n_rows), nullptr, n_rows, seed, mask(), out);
    B2_LAUNCHED();
    return B2_OK;
  }

  // new seed (and, under B2_GROUPER_HASH_BITS, a wider hash); the hash grouper is rebuilt from the store
  int reseed(cudaStream_t s) {
    for (int attempt = 0; attempt < 16; ++attempt) {
      seed = seed * 0x9e3779b97f4a7c15ull + 0x7f4a7c15ull;
      if (hash_bits < 64) hash_bits = hash_bits + 16 > 64 ? 64 : hash_bits + 16;
      B2_RETURN_NOT_OK(b2_grouper_reset(inner));
      if (n == 0) return B2_OK;
      Temp hashes(ctx, s);
      B2_RETURN_NOT_OK(hashes.alloc(sizeof(uint64_t) * (size_t)n));
      hash_strings_kernel<int64_t><<<grid1(n), kBlock, 0, s>>>(off, bytes, BitmapReader(), is_null, n, seed, mask(),
                                                                 hashes.as<uint64_t>());
      B2_LAUNCHED();
      B2Array h = u64_array(hashes.ptr, n);
      Owned ids(ctx, s);
      B2_RETURN_NOT_OK(b2_grouper_consume(inner, &h, &ids.a, s));
      ScalarSlot slot(ctx);
      B2_RETURN_NOT_OK(slot.zero(s));
      count_not_iota_kernel<<<grid1(n), kBlock, 0, s>>>(static_cast<const uint32_t*>(ids.a.data), n, slot.dev());
      B2_LAUNCHED();
      B2_RETURN_NOT_OK(slot.fetch(s));
      if (slot.host()[0] == 0) return B2_OK;  // the stored values are distinct, so ids 0..n-1 in order = no collision
    }
    return set_error(B2_UNKNOWN_ERROR, "grouper: could not find a collision-free 64-bit hash for the stored keys");
  }

  template <typename OffT>
  int run_typed(const B2Array* col, B2Array* out_ids, bool insert, cudaStream_t s) {
    const int64_t n_rows = col->length;
    const OffT* offs = static_cast<const OffT*>(col->data) + col->offset;
    const uint8_t* data = static_cast<const uint8_t*>(col->data2);
    const BitmapReader valid(col->null_count == 0 ? nullptr : col->validity, col->offset, n_rows);
    if (n_rows == 0) {
      Temp ids(ctx, s);
      B2_RETURN_NOT_OK(ids.alloc(4));
      fill_out(out_ids, B2_UINT32, 0, 0, nullptr, ids.release());
      return B2_OK;
    }
    Temp hashes(ctx, s);
    B2_RETURN_NOT_OK(hashes.alloc(sizeof(uint64_t) * (size_t)n_rows));
    if (!insert) {
      B2_RETURN_NOT_OK(hash_batch<OffT>(col, hashes.as<uint64_t>(), s));
      B2Array h = u64_array(hashes.ptr, n_rows);
      Owned ids(ctx, s);
      B2_RETURN_NOT_OK(b2_grouper_lookup(inner, &h, &ids.a, s));
      Temp bits(ctx, s);
      B2_RETURN_NOT_OK(bits.alloc(bitmap_alloc_bytes(n_rows)));
      B2_CUDA(cudaMemsetAsync(bits.ptr, 0, bitmap_alloc_bytes(n_rows), s));
      ScalarSlot slot(ctx);
      B2_RETURN_NOT_OK(slot.zero(s));
      B2_RETURN_NOT_OK(reserve(1, 1, s));  // an empty store still needs addressable arrays
      verify_kernel<OffT><<<grid1(n_rows), kBlock, 0, s>>>(offs, data, valid, n_rows, static_cast<const uint32_t*>(ids.a.data),
                                                           BitmapReader(ids.a.null_count == 0 ? nullptr : ids.a.validity, 0, n_rows),
                                                           off, bytes, rec, bits.as<uint32_t>(), slot.dev());
      B2_LAUNCHED();
      B2_RETURN_NOT_OK(slot.fetch(s));
      const int64_t nulls = n_rows - slot.host()[0];
      const void* id_data = ids.a.data;
      ids.a.data = nullptr;
      fill_out(out_ids, B2_UINT32, n_rows, nulls, nulls ? bits.release() : nullptr, id_data);
      return B2_OK;
    }
    for (int attempt = 0; attempt < 16; ++attempt) {
      B2_RETURN_NOT_OK(hash_batch<OffT>(col, hashes.as<uint64_t>(), s));
      B2Array h = u64_array(hashes.ptr, n_rows);
      Owned ids(ctx, s), first(ctx, s);
      // the 64-bit grouper already knows where this batch's new groups first occur (its first-occurrence flags): ask for the rows
      B2_RETURN_NOT_OK(grouper_consume_new_rows(inner, &h, &ids.a, &first.a, s));
      uint32_t total = 0;
      B2_RETURN_NOT_OK(b2_grouper_num_groups(inner, &total));
      const uint32_t n_new = total - n;
      const uint32_t* id_ptr = static_cast<const uint32_t*>(ids.a.data);
      int64_t new_bytes = 0;
      bool new_null = false;
      if (n_new) {
        if (first.a.length != (int64_t)n_new) return set_error(B2_UNKNOWN_ERROR, "grouper: first-occurrence rows out of step with the new groups");
        B2Array fr = u32_array(first.a.data, n_new);
        Owned taken(ctx, s);
        B2_RETURN_NOT_OK(b2_take(ctx, col, &fr, 0, &taken.a, s));
        B2_RETURN_NOT_OK(b2_binary_data_size(ctx, &taken.a, &new_bytes, s));
        new_null = taken.a.null_count > 0;
        B2_RETURN_NOT_OK(reserve((uint64_t)n + n_new, (uint64_t)(n_bytes + new_bytes), s));
        store_append_kernel<OffT><<<grid1(n_new), kBlock, 0, s>>>(
            static_cast<const OffT*>(taken.a.data) + taken.a.offset, static_cast<const uint8_t*>(taken.a.data2),
            BitmapReader(taken.a.null_count == 0 ? nullptr : taken.a.validity, taken.a.offset, n_new), n_new, n_bytes, off, is_null, rec, n);
        B2_LAUNCHED();
        if (new_bytes) {
          OffT first_off = 0;  // the taken array starts at offset 0 of its own data buffer
          (void)first_off;
          B2_CUDA(cudaMemcpyAsync(bytes + n_bytes, taken.a.data2, (size_t)new_bytes, cudaMemcpyDeviceToDevice, s));
        }
      } else {
        B2_RETURN_NOT_OK(reserve(1, 1, s));
      }
      ScalarSlot slot(ctx);
      B2_RETURN_NOT_OK(slot.zero(s));
      verify_kernel<OffT><<<grid1(n_rows), kBlock, 0, s>>>(offs, data, valid, n_rows, id_ptr, BitmapReader(), off, bytes, rec,
                                                           nullptr, slot.dev());
      B2_LAUNCHED();
      B2_RETURN_NOT_OK(slot.fetch(s));
      if (slot.host()[0] == 0) {
        n = total;
        n_bytes += new_bytes;
        has_null = has_null || new_null;
        ids.give(out_ids);
        return B2_OK;
      }
      // two different values share a hash: forget this batch (the store keeps its first n entries), re-seed
      B2_RETURN_NOT_OK(reseed(s));
    }
    return set_error(B2_UNKNOWN_ERROR, "grouper: could not find a collision-free 64-bit hash for this batch");
  }

  int run(const B2Array* col, B2Array* out_ids, bool insert, cudaStream_t s) {
    return large() ? run_typed<int64_t>(col, out_ids, insert, s) : run_typed<int32_t>(col, out_ids, insert, s);
  }

  // the distinct values in id order, as an array of the key's type (a copy: the store keeps growing)
  int uniques(B2Array* out, cudaStream_t s) {
    const int ow = offset_width(type);
    Temp o(ctx, s), b(ctx, s), v(ctx, s);
    B2_RETURN_NOT_OK(o.alloc(((size_t)n + 1) * ow));
    B2_RETURN_NOT_OK(b.alloc((size_t)n_bytes + 16));
    if (n == 0) {
      B2_CUDA(cudaMemsetAsync(o.ptr, 0, ow, s));
    } else if (ow == 8) {
      B2_CUDA(cudaMemcpyAsync(o.ptr, off, ((size_t)n + 1) * 8, cudaMemcpyDeviceToDevice, s));
    } else {
      if (n_bytes > 0x7fffffffll) return set_error(B2_CAPACITY_ERROR, "grouper: the distinct keys need more than 2^31 bytes; use large_utf8 / large_binary keys");
      narrow_offsets_kernel<int32_t><<<grid1((int64_t)n + 1), kBlock, 0, s>>>(off, (int64_t)n + 1, o.as<int32_t>());
      B2_LAUNCHED();
    }
    if (n_bytes) B2_CUDA(cudaMemcpyAsync(b.ptr, bytes, (size_t)n_bytes, cudaMemcpyDeviceToDevice, s));
    if (has_null) {
      B2_RETURN_NOT_OK(v.alloc(bitmap_alloc_bytes(n)));
      B2_CUDA(cudaMemsetAsync(v.ptr, 0, bitmap_alloc_bytes(n), s));
      null_bytes_to_bitmap_kernel<<<grid1(n), kBlock, 0, s>>>(is_null, n, v.as<uint32_t>());
      B2_LAUNCHED();
    }
    fill_out(out, type, n, has_null ? 1 : 0, has_null ? v.release() : nullptr, o.release(), b.release());
    return B2_OK;
  }
};

}  // namespace

// ---- the parts and their fold -------------------------------------------------------------------------------------
struct WideGrouper {
  B2Context* ctx;
  std::vector<int32_t> key_types;
  struct Part {
    int col0, n_cols;
    B2Grouper* narrow = nullptr;  // fixed-width run
    StringPart* str = nullptr;    // one utf8 / binary column
  };
  std::vector<Part> parts;
  std::vector<B2Grouper*> folds;  // folds[k-1]: (ids over parts 0..k-1, ids of part k) -> ids over parts 0..k
  uint32_t num_groups = 0;
};

static int part_run(WideGrouper* g, WideGrouper::Part& p, const B2Array* keys, B2Array* out_ids, bool insert, cudaStream_t s) {
  if (p.str) return p.str->run(&keys[p.col0], out_ids, insert, s);
  return insert ? b2_grouper_consume(p.narrow, keys + p.col0, out_ids, s) : b2_grouper_lookup(p.narrow, keys + p.col0, out_ids, s);
}

int wide_create(B2Context* ctx, const int32_t* key_types, int n_keys, WideGrouper** out) {
  for (int j = 0; j < n_keys; ++j)
    if (!type_is_binary_like(key_types[j]) && type_width(key_types[j]) == 0)
      return set_error(B2_NOT_IMPLEMENTED, "grouper: key type id %d is neither fixed-width numeric nor utf8 / binary", key_types[j]);
  WideGrouper* g = new WideGrouper();
  g->ctx = ctx;
  g->key_types.assign(key_types, key_types + n_keys);
  int st = B2_OK;
  for (int j = 0; j < n_keys && st == B2_OK;) {
    WideGrouper::Part p{};
    p.col0 = j;
    if (type_is_binary_like(key_types[j])) {
      p.n_cols = 1;
      p.str = new StringPart();
      p.str->ctx = ctx;
      p.str->type = key_types[j];
      st = p.str->init();
      ++j;
    } else {
      // the longest run of fixed-width columns whose packed encoding (+ one null flag per column when there are several) fits 64 bits
      int bits = 0, k = j;
      while (k < n_keys && !type_is_binary_like(key_types[k])) {
        const int w = 8 * type_width(key_types[k]);
        const int cols = k - j + 1;
        if (bits + w + (cols > 1 ? cols : 0) > 64) break;
        bits += w;
        ++k;
      }
      p.n_cols = k - j;
      st = b2_grouper_create(ctx, key_types + j, p.n_cols, &p.narrow);
      j = k;
    }
    g->parts.push_back(p);
  }
  for (size_t k = 1; k < g->parts.size() && st == B2_OK; ++k) {
    const int32_t kt = B2_UINT64;
    B2Grouper* f = nullptr;
    st = b2_grouper_create(ctx, &kt, 1, &f);
    if (st == B2_OK) g->folds.push_back(f);
  }
  if (st != B2_OK) {
    void wide_destroy(WideGrouper*);
    wide_destroy(g);
    return st;
  }
  *out = g;
  return B2_OK;
}

void wide_destroy(WideGrouper* g) {
  if (!g) return;
  for (auto& p : g->parts) {
    if (p.narrow) b2_grouper_destroy(p.narrow);
    if (p.str) {
      p.str->destroy(g->ctx->stream);
      delete p.str;
    }
  }
  for (B2Grouper* f : g->folds) b2_grouper_destroy(f);
  delete g;
}

int wide_reset(WideGrouper* g) {
  for (auto& p : g->parts) {
    if (p.narrow) B2_RETURN_NOT_OK(b2_grouper_reset(p.narrow));
    if (p.str) B2_RETURN_NOT_OK(p.str->reset());
  }
  for (B2Grouper* f : g->folds) B2_RETURN_NOT_OK(b2_grouper_reset(f));
  g->num_groups = 0;
  return B2_OK;
}

uint32_t wide_num_groups(const WideGrouper* g) { return g->num_groups; }

int wide_run(WideGrouper* g, const B2Array* keys, B2Array* out_ids, bool insert, cudaStream_t s) {
  B2Context* ctx = g->ctx;
  if (!keys) return set_error(B2_INVALID, "grouper: null keys");
  const int64_t n = keys[0].length;
  for (size_t j = 0; j < g->key_types.size(); ++j) {
    if (keys[j].type != g->key_types[j])
      return set_error(B2_INVALID, "expected batch value %d of type id %d but got %d", (int)j, g->key_types[j], keys[j].type);
    if (keys[j].length != n) return set_error(B2_INVALID, "grouper: key columns differ in length");
  }
  if (n > 0xfffffff0ll) return set_error(B2_NOT_IMPLEMENTED, "grouper: batches above 2^32 rows must be split");
  Owned cur(ctx, s);
  B2_RETURN_NOT_OK(part_run(g, g->parts[0], keys, &cur.a, insert, s));
  for (size_t k = 1; k < g->parts.size(); ++k) {
    Owned next(ctx, s);
    B2_RETURN_NOT_OK(part_run(g, g->parts[k], keys, &next.a, insert, s));
    Temp packed(ctx, s), bits(ctx, s);
    B2_RETURN_NOT_OK(packed.alloc(sizeof(uint64_t) * (size_t)n));
    int64_t nulls = 0;
    if (n) {
      pack_pair_kernel<<<grid1(n), kBlock, 0, s>>>(static_cast<const uint32_t*>(cur.a.data), static_cast<const uint32_t*>(next.a.data), n,
                                                   packed.as<uint64_t>());
      B2_LAUNCHED();
      if (cur.a.null_count || next.a.null_count) {  // Lookup only: a tuple with an unknown component is unknown
        B2_RETURN_NOT_OK(bits.alloc(bitmap_alloc_bytes(n)));
        B2_CUDA(cudaMemsetAsync(bits.ptr, 0, bitmap_alloc_bytes(n), s));
        ScalarSlot slot(ctx);
        B2_RETURN_NOT_OK(slot.zero(s));
        B2_RETURN_NOT_OK(launch_bitmap_and(cur.a.null_count ? cur.a.validity : nullptr, 0, next.a.null_count ? next.a.validity : nullptr, 0, n,
                                           bits.ptr, slot.dev(), s));
        B2_RETURN_NOT_OK(slot.fetch(s));
        nulls = n - slot.host()[0];
      }
    }
    cur.reset();
    next.reset();
    B2Array pk = u64_array(packed.ptr, n, nulls ? bits.ptr : nullptr, nulls);
    B2_RETURN_NOT_OK(insert ? b2_grouper_consume(g->folds[k - 1], &pk, &cur.a, s) : b2_grouper_lookup(g->folds[k - 1], &pk, &cur.a, s));
  }
  if (insert) {
    if (g->folds.empty()) g->num_groups = g->parts[0].str ? g->parts[0].str->n : 0;
    else B2_RETURN_NOT_OK(b2_grouper_num_groups(g->folds.back(), &g->num_groups));
    if (g->folds.empty() && g->parts[0].narrow) B2_RETURN_NOT_OK(b2_grouper_num_groups(g->parts[0].narrow, &g->num_groups));
  }
  cur.give(out_ids);
  return B2_OK;
}

// out[j] for every original key column, num_groups long, in group-id order
int wide_uniques(WideGrouper* g, B2Array* out_keys, cudaStream_t s) {
  B2Context* ctx = g->ctx;
  const size_t P = g->parts.size();
  const int64_t G = g->num_groups;
  // ids of every part for every final group: unfold the levels from the last one down
  std::vector<Temp*> part_ids(P, nullptr);
  struct Cleanup {
    std::vector<Temp*>& v;
    ~Cleanup() {
      for (Temp* t : v) delete t;
    }
  } cleanup{part_ids};
  if (P > 1) {
    Temp* cur = nullptr;  // ids into level k-1 for every final group
    for (size_t k = P - 1; k >= 1; --k) {
      Owned level(ctx, s);  // uniques of folds[k-1]: packed (ids over 0..k-1, ids of part k), one per group of level k
      B2_RETURN_NOT_OK(b2_grouper_uniques(g->folds[k - 1], &level.a, s));
      Owned sel(ctx, s);  // ... restricted / reordered to the final groups
      const B2Array* pairs = &level.a;
      if (cur) {
        B2Array idx = u32_array(cur->ptr, G);
        B2_RETURN_NOT_OK(b2_take(ctx, &level.a, &idx, 0, &sel.a, s));
        pairs = &sel.a;
      }
      Temp* lo = new Temp(ctx, s);
      Temp* hi = new Temp(ctx, s);
      part_ids[k] = lo;
      int st = lo->alloc(sizeof(uint32_t) * (size_t)(G ? G : 1));
      if (st == B2_OK) st = hi->alloc(sizeof(uint32_t) * (size_t)(G ? G : 1));
      if (st != B2_OK) {
        delete hi;
        delete cur;
        return st;
      }
      if (G) {
        unpack_pair_kernel<<<grid1(G), kBlock, 0, s>>>(static_cast<const uint64_t*>(pairs->data) + pairs->offset, G, hi->as<uint32_t>(),
                                                        lo->as<uint32_t>());
        g_launches.fetch_add(1, std::memory_order_relaxed);
      }
      delete cur;
      cur = hi;
      if (k == 1) part_ids[0] = cur;
    }
    B2_CUDA(cudaGetLastError());
  }
  for (size_t p = 0; p < P; ++p) {
    WideGrouper::Part& part = g->parts[p];
    std::vector<B2Array> cols(part.n_cols);
    struct Free {
      B2Context* ctx;
      cudaStream_t s;
      std::vector<B2Array>& v;
      ~Free() {
        for (B2Array& a : v) {
          if (a.validity) ctx->free(const_cast<void*>(a.validity), s);
          if (a.data) ctx->free(const_cast<void*>(a.data), s);
          if (a.data2) ctx->free(const_cast<void*>(a.data2), s);
        }
      }
    } free_cols{ctx, s, cols};
    if (part.str) B2_RETURN_NOT_OK(part.str->uniques(&cols[0], s));
    else B2_RETURN_NOT_OK(b2_grouper_uniques(part.narrow, cols.data(), s));
    for (int c = 0; c < part.n_cols; ++c) {
      if (P == 1) {
        out_keys[part.col0 + c] = cols[c];
        cols[c] = B2Array{};
      } else {
        B2Array idx = u32_array(part_ids[p]->ptr, G);
        B2_RETURN_NOT_OK(b2_take(ctx, &cols[c], &idx, 0, &out_keys[part.col0 + c], s));
      }
    }
  }
  return B2_OK;
}

}  // namespace b2

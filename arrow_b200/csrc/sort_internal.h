// sort_internal.h -- pieces of the radix sort (sort_indices.cu) shared with the utf8 / binary sort (sort_strings.cu).
#pragma once
#include "context.h"

namespace b2 {

// Stable LSD radix sort of (key, uint32 idx) pairs of n < 2^32 - 8192 rows; digits that are equal in every key are
// skipped.  The pairs start in (keys_a, idx_a); keys_b / idx_b are allocated when more than one pass runs.  With
// final_out set, the last pass writes only the indices, widened to uint64, there; otherwise *keys_out / *idx_out
// point at whichever buffers hold the sorted pairs.  K = uint32_t or uint64_t.
template <typename K>
int radix_sort_pairs(B2Context* ctx, int passes, K* keys_a, uint32_t* idx_a, Temp* keys_b, Temp* idx_b, uint32_t n,
                     uint64_t* final_out, K** keys_out, uint32_t** idx_out, cudaStream_t s);

// The sort of one numeric or string column into out[0, values.length) (sort_run minus its checks and allocation).
int sort_into(B2Context* ctx, const B2Array* values, int order, int null_placement, const uint32_t* payload, uint64_t* out,
              cudaStream_t s);

// A C-ABI output whose buffers go back to the pool unless released (owned = false).
struct PoolArray {
  B2Context* ctx;
  cudaStream_t s;
  B2Array a{};
  bool owned = false;
  PoolArray(B2Context* c, cudaStream_t st) : ctx(c), s(st) {}
  PoolArray(const PoolArray&) = delete;
  PoolArray& operator=(const PoolArray&) = delete;
  ~PoolArray() { reset(); }
  void reset() {
    if (!owned) return;
    if (a.validity) ctx->free(const_cast<void*>(a.validity), s);
    if (a.data) ctx->free(const_cast<void*>(a.data), s);
    if (a.data2) ctx->free(const_cast<void*>(a.data2), s);
    owned = false;
    a = B2Array{};
  }
};

// Which path sort_strings takes for this column: B2_SORT_STRINGS_PATH=dict|refine, else the sampled estimate.
int string_sort_path(B2Context* ctx, const B2Array* values, bool* dict, cudaStream_t s);

// sort_strings.cu: the stable sort of a utf8 / binary / large_utf8 / large_binary column (same contract as the
// numeric sort_typed: out = values.length uint64, row i carries payload[i] when payload is set).
int sort_strings(B2Context* ctx, const B2Array* values, int order, int null_placement, uint64_t* out, cudaStream_t s,
                 const uint32_t* payload);

// The round-0 keys of the string sort as a B2_UINT64 column with a copy of the string column's validity, re-based to bit 0:
// bytes [0, 7) big-endian in the high 56 bits, min(length, 8) in the low byte.  Comparing two keys agrees with
// comparing the strings whenever the keys differ.
int string_prefix_keys(B2Context* ctx, const B2Array* values, B2Array* out, cudaStream_t s);

}  // namespace b2

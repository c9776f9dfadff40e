// select_k.cu -- select_k_unstable over one numeric, utf8 or binary column: the indices of the first k rows of the sorted order.
//
// Replaces ArraySelector (kernels/vector_select_k.cc:157-232: null-like partition, then a k-element heap over the
// non-null values) -- k log k work per row on one CPU thread.  "Unstable" only frees the tie order; this implementation
// returns exactly sort_indices(values, order, null_placement)[0:k] (ties in row order), which is one of the permitted
// answers and makes the result deterministic.
//
// B200 design (k << n): a sorted 64Ki-row strided sample yields a threshold t whose rank is safely above k; ONE streaming
// compare pass (values <= t, or >= t for Descending: 8 B/row, HBM rate) gives the candidate mask, the candidates are
// compacted to their row numbers (GetTakeIndices), gathered and sorted -- a few thousand to a few million rows instead of
// n.  Every row that can be among the first k is a candidate (all rows <= t are taken, ties included), so the first k of
// the stably sorted candidates ARE the first k of the stable full sort.  If the sample misjudged (fewer than k candidates:
// skew, NaNs, nulls first) or k is a large fraction of n, the full radix sort runs and its prefix is returned.
#include <cstring>
#include <vector>

#include "common.cuh"
#include "context.h"
#include "sort_internal.h"

using namespace b2;

namespace {
struct Out {  // a C-ABI output whose buffers go back to the pool unless handed over
  B2Context* ctx;
  cudaStream_t s;
  B2Array a{};
  Out(B2Context* c, cudaStream_t st) : ctx(c), s(st) {}
  Out(const Out&) = delete;
  ~Out() {
    if (a.validity) ctx->free(const_cast<void*>(a.validity), s);
    if (a.data) ctx->free(const_cast<void*>(a.data), s);
    if (a.data2) ctx->free(const_cast<void*>(a.data2), s);
  }
  void give(B2Array* out) {
    *out = a;
    a = B2Array{};
  }
};

constexpr int64_t kSample = 1 << 16;

int full_sort_prefix(B2Context* ctx, const B2Array* values, int64_t k, int order, int null_placement, B2Array* out, void* stream) {
  B2_RETURN_NOT_OK(b2_sort_indices(ctx, values, order, null_placement, out, stream));
  if (k < out->length) out->length = k;  // a prefix view of the same buffer
  return B2_OK;
}

// utf8 / binary: the round-0 keys of the string sort (sort_strings.cu) order the rows wherever two keys differ, so the
// numeric selection over the key column gives a threshold key T (the last key it selected); every row that can be among
// the first k has a key at or before T, ties included.  Those candidates are sorted as strings.
int select_k_strings(B2Context* ctx, const B2Array* values, int64_t k, int order, int null_placement, B2Array* out,
                     void* stream) {
  const int64_t n = values->length;
  cudaStream_t s = ctx->pick(stream);
  const bool maybe_nulls = values->null_count != 0 && values->validity;
  if (n < (1 << 20) || k * 8 > n || (null_placement == 0 && maybe_nulls))
    return full_sort_prefix(ctx, values, k, order, null_placement, out, stream);
  Out keys(ctx, s), sel(ctx, s), pick(ctx, s);
  B2_RETURN_NOT_OK(string_prefix_keys(ctx, values, &keys.a, s));
  B2_RETURN_NOT_OK(b2_select_k(ctx, &keys.a, k, order, null_placement, &sel.a, stream));
  B2Array last = sel.a;
  last.offset += k - 1;
  last.length = 1;
  B2_RETURN_NOT_OK(b2_take(ctx, &keys.a, &last, 0, &pick.a, stream));
  if (pick.a.null_count != 0) return full_sort_prefix(ctx, values, k, order, null_placement, out, stream);  // < k valid rows
  uint64_t bits = 0;
  B2_CUDA(cudaMemcpyAsync(&bits, pick.a.data, sizeof(bits), cudaMemcpyDeviceToHost, s));
  B2_CUDA(cudaStreamSynchronize(s));

  B2Scalar t{bits, B2_UINT64, 1};
  B2Value l{&keys.a, nullptr}, r{nullptr, &t};
  Out mask(ctx, s), cand_rows(ctx, s);
  B2_RETURN_NOT_OK(b2_compare(ctx, order == 0 ? B2_LESS_EQUAL : B2_GREATER_EQUAL, &l, &r, &mask.a, stream));
  B2_RETURN_NOT_OK(b2_filter_indices(ctx, &mask.a, /*DROP=*/0, &cand_rows.a, stream));
  const int64_t m = cand_rows.a.length;
  if (m < k || m * 2 > n) return full_sort_prefix(ctx, values, k, order, null_placement, out, stream);

  Out cand(ctx, s), perm(ctx, s), picked(ctx, s), wide(ctx, s);
  B2_RETURN_NOT_OK(b2_take(ctx, values, &cand_rows.a, 0, &cand.a, stream));
  B2_RETURN_NOT_OK(b2_sort_indices(ctx, &cand.a, order, null_placement, &perm.a, stream));
  B2Array first_k = perm.a;
  first_k.length = k;
  B2_RETURN_NOT_OK(b2_take(ctx, &cand_rows.a, &first_k, 0, &picked.a, stream));
  B2CastOptions to_u64{B2_UINT64, 1, 1, 0};
  B2_RETURN_NOT_OK(b2_cast_numeric(ctx, &picked.a, &to_u64, &wide.a, stream));
  wide.give(out);
  return B2_OK;
}
}  // namespace

extern "C" int b2_select_k(B2Context* ctx, const B2Array* values, int64_t k, int order, int null_placement, B2Array* out,
                           void* stream) {
  if (!ctx || !values || !out) return set_error(B2_INVALID, "b2_select_k: null argument");
  if (k < 0) return set_error(B2_INVALID, "select_k_unstable requires a nonnegative `k`, got %lld", (long long)k);  // vector_select_k.cc:640
  if (order != 0 && order != 1) return set_error(B2_INVALID, "bad sort order %d", order);
  if (null_placement != 0 && null_placement != 1) return set_error(B2_INVALID, "bad null placement %d", null_placement);
  if (!type_is_numeric(values->type) && !type_is_binary_like(values->type))
    return set_error(B2_NOT_IMPLEMENTED, "select_k_unstable: unsupported type id %d", values->type);
  const int64_t n = values->length;
  if (k > n) k = n;
  cudaStream_t s = ctx->pick(stream);
  B2_CUDA(cudaSetDevice(ctx->device));
  if (k == 0) {
    fill_out(out, B2_UINT64, 0, 0, nullptr, nullptr);
    return B2_OK;
  }
  if (type_is_binary_like(values->type)) return select_k_strings(ctx, values, k, order, null_placement, out, stream);
  const bool is_float = values->type == B2_FLOAT || values->type == B2_DOUBLE;
  // the threshold path only ever selects non-null, non-NaN rows: with nulls (or possibly NaNs) FIRST they would be skipped
  const bool maybe_nulls = values->null_count != 0 && values->validity;
  if (n < (1 << 20) || k * 8 > n || (null_placement == 0 && (maybe_nulls || is_float)))
    return full_sort_prefix(ctx, values, k, order, null_placement, out, stream);

  // 1. strided sample, sorted (nulls and NaNs of the sample sort to the end)
  const int64_t stride = n / kSample;
  std::vector<uint32_t> rows(kSample);
  for (int64_t i = 0; i < kSample; ++i) rows[i] = static_cast<uint32_t>(i * stride + (stride >> 1));
  Temp sample_rows(ctx, s);
  B2_RETURN_NOT_OK(sample_rows.alloc(sizeof(uint32_t) * kSample));
  B2_CUDA(cudaMemcpyAsync(sample_rows.ptr, rows.data(), sizeof(uint32_t) * kSample, cudaMemcpyHostToDevice, s));
  B2_CUDA(cudaStreamSynchronize(s));  // `rows` is pageable and dies with this frame
  B2Array ridx{};
  ridx.type = B2_UINT32;
  ridx.data = sample_rows.ptr;
  ridx.length = kSample;
  Out sample(ctx, s), sample_perm(ctx, s), pick(ctx, s);
  B2_RETURN_NOT_OK(b2_take(ctx, values, &ridx, 0, &sample.a, stream));
  B2_RETURN_NOT_OK(b2_sort_indices(ctx, &sample.a, order, /*AtEnd=*/1, &sample_perm.a, stream));
  // rank of the threshold inside the sample: twice the expected rank of k plus a margin of ~6 standard deviations
  const double expect = static_cast<double>(k) / static_cast<double>(n) * kSample;
  int64_t rank = static_cast<int64_t>(expect * 2.0) + 96;
  if (rank >= kSample - 1) return full_sort_prefix(ctx, values, k, order, null_placement, out, stream);
  B2Array one = sample_perm.a;
  one.offset = rank;
  one.length = 1;
  B2_RETURN_NOT_OK(b2_take(ctx, &sample.a, &one, 0, &pick.a, stream));
  if (pick.a.null_count != 0) return full_sort_prefix(ctx, values, k, order, null_placement, out, stream);  // the sample ran out of values
  uint64_t bits = 0;
  const int w = type_width(values->type);
  B2_CUDA(cudaMemcpyAsync(&bits, pick.a.data, w, cudaMemcpyDeviceToHost, s));
  B2_CUDA(cudaStreamSynchronize(s));
  if (is_float) {
    bool nan;
    if (w == 4) {
      float f;
      uint32_t b32 = static_cast<uint32_t>(bits);
      memcpy(&f, &b32, 4);
      nan = f != f;
    } else {
      double d;
      memcpy(&d, &bits, 8);
      nan = d != d;
    }
    if (nan) return full_sort_prefix(ctx, values, k, order, null_placement, out, stream);
  }

  // 2. candidates = rows at or before the threshold (one streaming pass), as row numbers
  B2Scalar t{bits, values->type, 1};
  B2Value l{values, nullptr}, r{nullptr, &t};
  Out mask(ctx, s), cand_rows(ctx, s);
  B2_RETURN_NOT_OK(b2_compare(ctx, order == 0 ? B2_LESS_EQUAL : B2_GREATER_EQUAL, &l, &r, &mask.a, stream));
  B2_RETURN_NOT_OK(b2_filter_indices(ctx, &mask.a, /*DROP=*/0, &cand_rows.a, stream));
  const int64_t m = cand_rows.a.length;
  if (m < k || m * 2 > n) return full_sort_prefix(ctx, values, k, order, null_placement, out, stream);

  // 3. sort the candidates (row order in, stable), map the first k back to row numbers
  Out cand(ctx, s), perm(ctx, s), picked(ctx, s), wide(ctx, s);
  B2_RETURN_NOT_OK(b2_take(ctx, values, &cand_rows.a, 0, &cand.a, stream));
  B2_RETURN_NOT_OK(b2_sort_indices(ctx, &cand.a, order, null_placement, &perm.a, stream));
  B2Array first_k = perm.a;
  first_k.length = k;
  B2_RETURN_NOT_OK(b2_take(ctx, &cand_rows.a, &first_k, 0, &picked.a, stream));
  B2CastOptions to_u64{B2_UINT64, 1, 1, 0};
  B2_RETURN_NOT_OK(b2_cast_numeric(ctx, &picked.a, &to_u64, &wide.a, stream));
  wide.give(out);
  return B2_OK;
}

// sort_strings.cu -- stable argsort of one utf8 / binary / large_utf8 / large_binary column.
//
// Replaces, for base-binary keys:
//   ArraySortIndices over BinaryType / LargeBinaryType / StringType / LargeStringType
//                                               kernels/vector_array_sort.cc:588-594
//   ArrayCompareSorter (std::stable_sort, string_view comparator)   :144-178
//   PartitionNullsAndNans / NullLikePartition   kernels/vector_sort_internal.h:113-305
// Semantics kept: the order is unsigned byte-wise lexicographic, a proper prefix sorts first; the sort is STABLE;
// nulls are stably partitioned to the end (AtEnd) or the start (AtStart); Descending keeps ties in ascending row
// order; output = uint64 indices, never null.  Character data may be of any size (64-bit offsets).
//
// B200 design (no comparator, no per-row string copy): the strings are decided 7 bytes at a time.
//   key     : in round r, a row's 64-bit key holds bytes [d, d+7) of its string (d = 7r) big-endian in the high 56
//             bits, zero past the end, and min(len - d, 8) in the low byte.  Two keys compare as the 7-byte windows
//             do, and a proper prefix has the smaller low byte ("ab" < "ab\0", "abcdefg" < "abcdefgh").  Descending
//             uses ~key, as ordered_key does for numbers.
//   round 0 : the null partition (the Filter plan over the validity bitmap, as sort_typed), then one radix sort of
//             the keys of all valid rows, row numbers riding along.
//   runs    : rows with equal keys form a run.  A run is decided when it has one row or its low byte is < 8 (every
//             member ends inside the window, so all are equal and stability leaves them in row order).
//   later   : the rows of undecided runs are compacted (the Filter plan over a keep bitmap) with their output slots
//             and a run id, keyed by the next window, and sorted by (run id, key) -- a radix sort on the key, then a
//             stable one on the run id -- which leaves every run inside its own slot range.  Digits that are equal in
//             every key (the run id while few runs remain, the length byte) cost no pass.
// Row numbers travel through the rounds; a payload (b2_sort_payload, the multi-key permutation) is applied only
// when the result is written.  Rounds = 1 + (longest common prefix of two rows) / 7.
//
// Dictionary path (many duplicates): b2_vector_hash gives every valid row an index into the distinct values; the
// distinct values are sorted by the rounds above, each gets its rank, and one numeric radix sort of rank[index]
// (nulls kept null) orders the column.  Equal strings share a rank, so ties stay in row order.  The path is chosen
// from a strided 64Ki-row sample whose distinct values are counted on the device (see kDictDupShare).
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "selection.cuh"
#include "sort_internal.h"

namespace b2 {

namespace {

constexpr int64_t kSample = 1 << 16;
// Take the dictionary path when the column is estimated to hold at least this many rows per distinct value.  Measured
// on 50M words (B200, DESIGN.md section 3): dictionary / refinement 6.6 / 13.2 ms at 10 rows per value, 20.1 / 13.1 ms
// at 2.5; the refinement's time hardly depends on the cardinality.
constexpr double kDictRowsPerValue = 8.0;

__device__ __forceinline__ uint64_t bswap64(uint64_t v) {
  return (static_cast<uint64_t>(__byte_perm(static_cast<uint32_t>(v), 0, 0x0123)) << 32) |
         __byte_perm(static_cast<uint32_t>(v >> 32), 0, 0x0123);
}

// the round key of a row at depth d (see the header comment); offs is advanced by the array offset
template <typename OffT>
__device__ __forceinline__ uint64_t window_key(const OffT* __restrict__ offs, const uint8_t* __restrict__ chars, int64_t row,
                                               int64_t depth) {
  const int64_t b = static_cast<int64_t>(offs[row]);
  const int64_t rem = static_cast<int64_t>(offs[row + 1]) - b - depth;
  if (rem <= 0) return 0;
  const int nb = rem < 7 ? static_cast<int>(rem) : 7;
  return bswap64(load_bytes8(chars + b + depth, nb)) | static_cast<uint64_t>(rem < 8 ? rem : 8);
}

// null partition: valid rows -> order[] in row order, null rows -> their final slots
__global__ void __launch_bounds__(kBlock) str_partition_kernel(BitmapReader valid, const int64_t* __restrict__ tile_offsets,
                                                               int64_t n, const uint32_t* __restrict__ payload,
                                                               uint32_t* __restrict__ order, uint64_t* __restrict__ out_nulls) {
  __shared__ uint64_t s_sel[kTileWords];
  __shared__ uint32_t s_prefix[kTileWords];
  const int64_t tile = blockIdx.x, row0 = tile * kTileRows;
  if (threadIdx.x < 32) load_tile_prefix(valid, tile, s_sel, s_prefix);
  __syncthreads();
  const int64_t vbase = tile_offsets[tile], nbase = row0 - vbase;
  for (int r = threadIdx.x; r < kTileRows; r += kBlock) {
    const int64_t row = row0 + r;
    if (row >= n) break;
    const uint64_t w = s_sel[r >> 6];
    const unsigned before = s_prefix[r >> 6] + __popcll(w & ((1ull << (r & 63)) - 1ull));
    if ((w >> (r & 63)) & 1) order[vbase + before] = static_cast<uint32_t>(row);
    else out_nulls[nbase + (r - before)] = payload ? payload[row] : static_cast<uint64_t>(row);
  }
}

// keys of the active rows (act_slot NULL: every slot) at `depth`; rows[i] = their row numbers, idx[i] = i
template <typename OffT>
__global__ void __launch_bounds__(kBlock) str_extract_kernel(const OffT* __restrict__ offs, const uint8_t* __restrict__ chars,
                                                             const uint32_t* __restrict__ order,
                                                             const uint32_t* __restrict__ act_slot, int64_t m, int64_t depth,
                                                             uint64_t flip, uint32_t* __restrict__ rows,
                                                             uint64_t* __restrict__ keys, uint64_t* __restrict__ keys_copy,
                                                             uint32_t* __restrict__ idx) {
  for (int64_t i = blockIdx.x * (int64_t)kBlock + threadIdx.x; i < m; i += (int64_t)gridDim.x * kBlock) {
    const uint32_t row = order[act_slot ? act_slot[i] : i];
    const uint64_t k = window_key(offs, chars, row, depth) ^ flip;
    rows[i] = row;
    keys[i] = k;
    if (keys_copy) keys_copy[i] = k;
    idx[i] = static_cast<uint32_t>(i);
  }
}

template <typename T>
__global__ void __launch_bounds__(kBlock) gather_kernel(const T* __restrict__ src, const uint32_t* __restrict__ idx, int64_t m,
                                                        T* __restrict__ dst) {
  for (int64_t i = blockIdx.x * (int64_t)kBlock + threadIdx.x; i < m; i += (int64_t)gridDim.x * kBlock) dst[i] = src[idx[i]];
}

// the sorted active rows back into their slots
__global__ void __launch_bounds__(kBlock) str_writeback_kernel(const uint32_t* __restrict__ act_slot,
                                                               const uint32_t* __restrict__ rows,
                                                               const uint32_t* __restrict__ perm, int64_t m,
                                                               uint32_t* __restrict__ order) {
  for (int64_t i = blockIdx.x * (int64_t)kBlock + threadIdx.x; i < m; i += (int64_t)gridDim.x * kBlock)
    order[act_slot ? act_slot[i] : i] = rows[perm[i]];
}

// run heads and the rows of undecided runs, as bitmaps (32-bit words); ks / rs = keys / run ids in sorted order
__global__ void __launch_bounds__(kBlock) str_mark_kernel(const uint64_t* __restrict__ ks, const uint32_t* __restrict__ rs,
                                                          int64_t m, uint64_t flip, uint32_t* __restrict__ head_bits,
                                                          uint32_t* __restrict__ keep_bits) {
  const unsigned lane = lane_id();
  for (int64_t base = blockIdx.x * (int64_t)kBlock + (threadIdx.x & ~31u); base < m; base += (int64_t)gridDim.x * kBlock) {
    const int64_t j = base + lane;
    bool head = false, keep = false;
    if (j < m) {
      const uint64_t k = ks[j];
      const uint32_t r = rs ? rs[j] : 0;
      head = j == 0 || ks[j - 1] != k || (rs && rs[j - 1] != r);
      const bool tail = j + 1 == m || ks[j + 1] != k || (rs && rs[j + 1] != r);
      keep = !(head && tail) && ((k ^ flip) & 0xff) == 8;
    }
    const unsigned hb = __ballot_sync(0xffffffffu, head), kb = __ballot_sync(0xffffffffu, keep);
    if (lane == 0) {
      head_bits[base >> 5] = hb;
      keep_bits[base >> 5] = kb;
    }
  }
}

// compaction of the undecided rows: their slots and, as run id, the number of run heads before them
__global__ void __launch_bounds__(kBlock) str_compact_kernel(BitmapReader keep, BitmapReader head,
                                                             const int64_t* __restrict__ keep_offsets,
                                                             const int64_t* __restrict__ head_offsets,
                                                             const uint32_t* __restrict__ act_slot, int64_t m,
                                                             uint32_t* __restrict__ new_slot, uint32_t* __restrict__ new_run) {
  __shared__ uint64_t s_keep[kTileWords], s_head[kTileWords];
  __shared__ uint32_t p_keep[kTileWords], p_head[kTileWords];
  const int64_t tile = blockIdx.x, row0 = tile * kTileRows;
  if (threadIdx.x < 32) load_tile_prefix(keep, tile, s_keep, p_keep);
  else if (threadIdx.x < 64) load_tile_prefix(head, tile, s_head, p_head);
  __syncthreads();
  const int64_t kbase = keep_offsets[tile], hbase = head_offsets[tile];
  for (int r = threadIdx.x; r < kTileRows; r += kBlock) {
    const int64_t j = row0 + r;
    if (j >= m) break;
    const uint64_t w = s_keep[r >> 6];
    if (!((w >> (r & 63)) & 1)) continue;
    const int64_t dst = kbase + p_keep[r >> 6] + __popcll(w & ((1ull << (r & 63)) - 1ull));
    const uint64_t upto = (2ull << (r & 63)) - 1ull;  // bits 0..r&63 (all 64 when r&63 == 63)
    const int64_t heads = hbase + p_head[r >> 6] + __popcll(s_head[r >> 6] & upto);
    new_slot[dst] = act_slot ? act_slot[j] : static_cast<uint32_t>(j);
    new_run[dst] = static_cast<uint32_t>(heads - 1);
  }
}

__global__ void __launch_bounds__(kBlock) str_final_kernel(const uint32_t* __restrict__ order, const uint32_t* __restrict__ payload,
                                                           int64_t m, uint64_t* __restrict__ out) {
  for (int64_t i = blockIdx.x * (int64_t)kBlock + threadIdx.x; i < m; i += (int64_t)gridDim.x * kBlock)
    out[i] = payload ? payload[order[i]] : order[i];
}

__global__ void __launch_bounds__(kBlock) rank_scatter_kernel(const uint64_t* __restrict__ perm, int64_t m,
                                                              uint32_t* __restrict__ rank) {
  for (int64_t i = blockIdx.x * (int64_t)kBlock + threadIdx.x; i < m; i += (int64_t)gridDim.x * kBlock)
    rank[perm[i]] = static_cast<uint32_t>(i);
}

template <typename OffT>
__global__ void __launch_bounds__(kBlock) prefix_keys_kernel(const OffT* __restrict__ offs, const uint8_t* __restrict__ chars,
                                                             int64_t n, uint64_t* __restrict__ out) {
  for (int64_t i = blockIdx.x * (int64_t)kBlock + threadIdx.x; i < n; i += (int64_t)gridDim.x * kBlock)
    out[i] = window_key(offs, chars, i, 0);
}

inline int grid_of(int64_t m) { return grid_for(m, kBlock * 4, kSMs * 8); }

int partition_nulls(B2Context* ctx, const B2Array* values, bool at_start, const uint32_t* payload, uint64_t* out,
                    Temp* order, int64_t* nv, cudaStream_t s) {
  const int64_t n = values->length;
  FilterBitmaps fb;
  fb.mask_data = BitmapReader(values->null_count == 0 ? nullptr : values->validity, values->offset, n);
  fb.mask_valid = BitmapReader(nullptr, 0, n);
  fb.values_valid = BitmapReader(nullptr, 0, n);
  fb.emit_null = 0;
  Temp offsets(ctx, s);
  int64_t unused = 0;
  B2_RETURN_NOT_OK(filter_plan(ctx, fb, n, false, &offsets, nv, &unused, s));
  B2_RETURN_NOT_OK(order->alloc(sizeof(uint32_t) * (size_t)*nv));
  str_partition_kernel<<<(unsigned)tiles_for(n), kBlock, 0, s>>>(fb.mask_data, offsets.as<int64_t>(), n, payload,
                                                                 order->as<uint32_t>(), out + (at_start ? 0 : *nv));
  B2_LAUNCHED();
  return B2_OK;
}

// prefix refinement: order[0..nv) = valid row numbers in row order -> the same rows in string order
template <typename OffT>
int refine(B2Context* ctx, const B2Array* values, bool descending, uint32_t* order, int64_t nv, cudaStream_t s) {
  const OffT* offs = static_cast<const OffT*>(values->data) + values->offset;
  const uint8_t* chars = static_cast<const uint8_t*>(values->data2);
  const uint64_t flip = descending ? ~0ull : 0ull;
  Temp slots(ctx, s), runs(ctx, s);  // the undecided rows' slots and run ids; none in round 0 (one run: every slot)
  const uint32_t* act_slot = nullptr;
  const uint32_t* act_run = nullptr;
  int64_t m = nv;
  for (int64_t depth = 0; m > 0; depth += 7) {
    const size_t m4 = sizeof(uint32_t) * (size_t)m, m8 = sizeof(uint64_t) * (size_t)m;
    Temp rows(ctx, s), keys0(ctx, s), keysA(ctx, s), keysB(ctx, s), idxA(ctx, s), idxB(ctx, s);
    B2_RETURN_NOT_OK(rows.alloc(m4));
    B2_RETURN_NOT_OK(keysA.alloc(m8));
    B2_RETURN_NOT_OK(idxA.alloc(m4));
    if (act_run) B2_RETURN_NOT_OK(keys0.alloc(m8));
    str_extract_kernel<OffT><<<grid_of(m), kBlock, 0, s>>>(offs, chars, order, act_slot, m, depth, flip, rows.as<uint32_t>(),
                                                           keysA.as<uint64_t>(), keys0.as<uint64_t>(), idxA.as<uint32_t>());
    B2_LAUNCHED();
    uint64_t* ks;
    uint32_t* perm;
    B2_RETURN_NOT_OK(radix_sort_pairs<uint64_t>(ctx, 8, keysA.as<uint64_t>(), idxA.as<uint32_t>(), &keysB, &idxB,
                                                (uint32_t)m, nullptr, &ks, &perm, s));
    // stable by run id: every run keeps its slot range, sorted by key inside it
    Temp runsA(ctx, s), runsB(ctx, s), permB(ctx, s), ksorted(ctx, s);
    uint32_t* rs = nullptr;
    if (act_run) {
      B2_RETURN_NOT_OK(runsA.alloc(m4));
      gather_kernel<uint32_t><<<grid_of(m), kBlock, 0, s>>>(act_run, perm, m, runsA.as<uint32_t>());
      B2_LAUNCHED();
      B2_RETURN_NOT_OK(radix_sort_pairs<uint32_t>(ctx, 4, runsA.as<uint32_t>(), perm, &runsB, &permB, (uint32_t)m, nullptr,
                                                  &rs, &perm, s));
      B2_RETURN_NOT_OK(ksorted.alloc(m8));
      gather_kernel<uint64_t><<<grid_of(m), kBlock, 0, s>>>(keys0.as<uint64_t>(), perm, m, ksorted.as<uint64_t>());
      B2_LAUNCHED();
      ks = ksorted.as<uint64_t>();
    }
    str_writeback_kernel<<<grid_of(m), kBlock, 0, s>>>(act_slot, rows.as<uint32_t>(), perm, m, order);
    B2_LAUNCHED();

    // the undecided runs go to the next round
    Temp head(ctx, s), keep(ctx, s);
    B2_RETURN_NOT_OK(head.alloc(bitmap_alloc_bytes(m)));
    B2_RETURN_NOT_OK(keep.alloc(bitmap_alloc_bytes(m)));
    str_mark_kernel<<<grid_of(m), kBlock, 0, s>>>(ks, rs, m, flip, head.as<uint32_t>(), keep.as<uint32_t>());
    B2_LAUNCHED();
    FilterBitmaps fk, fh;
    fk.mask_data = BitmapReader(keep.ptr, 0, m);
    fh.mask_data = BitmapReader(head.ptr, 0, m);
    for (FilterBitmaps* f : {&fk, &fh}) {
      f->mask_valid = BitmapReader(nullptr, 0, m);
      f->values_valid = BitmapReader(nullptr, 0, m);
      f->emit_null = 0;
    }
    Temp keep_offs(ctx, s), head_offs(ctx, s);
    int64_t m2 = 0, n_heads = 0, unused = 0;
    B2_RETURN_NOT_OK(filter_plan(ctx, fk, m, false, &keep_offs, &m2, &unused, s));
    if (m2 == 0) break;
    B2_RETURN_NOT_OK(filter_plan(ctx, fh, m, false, &head_offs, &n_heads, &unused, s));
    Temp nslots(ctx, s), nruns(ctx, s);
    B2_RETURN_NOT_OK(nslots.alloc(sizeof(uint32_t) * (size_t)m2));
    B2_RETURN_NOT_OK(nruns.alloc(sizeof(uint32_t) * (size_t)m2));
    str_compact_kernel<<<(unsigned)tiles_for(m), kBlock, 0, s>>>(fk.mask_data, fh.mask_data, keep_offs.as<int64_t>(),
                                                                 head_offs.as<int64_t>(), act_slot, m, nslots.as<uint32_t>(),
                                                                 nruns.as<uint32_t>());
    B2_LAUNCHED();
    std::swap(slots.ptr, nslots.ptr);
    std::swap(runs.ptr, nruns.ptr);
    act_slot = slots.as<uint32_t>();
    act_run = runs.as<uint32_t>();
    m = m2;
  }
  return B2_OK;
}

int sort_refine(B2Context* ctx, const B2Array* values, int order, int null_placement, uint64_t* out, cudaStream_t s,
                const uint32_t* payload) {
  const bool at_start = null_placement == 0;
  Temp rows(ctx, s);
  int64_t nv = 0;
  B2_RETURN_NOT_OK(partition_nulls(ctx, values, at_start, payload, out, &rows, &nv, s));
  if (nv == 0) return B2_OK;
  if (offset_width(values->type) == 8)
    B2_RETURN_NOT_OK(refine<int64_t>(ctx, values, order == 1, rows.as<uint32_t>(), nv, s));
  else
    B2_RETURN_NOT_OK(refine<int32_t>(ctx, values, order == 1, rows.as<uint32_t>(), nv, s));
  str_final_kernel<<<grid_of(nv), kBlock, 0, s>>>(rows.as<uint32_t>(), payload, nv,
                                                  out + (at_start ? values->length - nv : 0));
  B2_LAUNCHED();
  return B2_OK;
}

int sort_dictionary(B2Context* ctx, const B2Array* values, int order, int null_placement, uint64_t* out, cudaStream_t s,
                    const uint32_t* payload) {
  // 1. indices (null where the row is null) and the distinct values
  PoolArray indices(ctx, s), dict(ctx, s);
  B2_RETURN_NOT_OK(b2_vector_hash(ctx, values, /*MASK=*/0, &indices.a, &dict.a, nullptr, s));
  indices.owned = dict.owned = true;
  const int64_t d = dict.a.length;
  // 2. the distinct values in the requested order; 3. rank[value] = its position
  Temp dperm(ctx, s), rank(ctx, s);
  B2_RETURN_NOT_OK(dperm.alloc(sizeof(uint64_t) * (size_t)d));
  B2_RETURN_NOT_OK(rank.alloc(sizeof(uint32_t) * (size_t)d));
  if (d > 0) {
    B2_RETURN_NOT_OK(sort_refine(ctx, &dict.a, order, /*AtEnd=*/1, dperm.as<uint64_t>(), s, nullptr));
    rank_scatter_kernel<<<grid_of(d), kBlock, 0, s>>>(dperm.as<uint64_t>(), d, rank.as<uint32_t>());
    B2_LAUNCHED();
  }
  // 4. rank of every row (nulls stay null); 5. one stable numeric sort, always ascending: ranks already carry the order
  B2Array rank_arr{};
  rank_arr.type = B2_UINT32;
  rank_arr.data = rank.ptr;
  rank_arr.length = d;
  PoolArray row_rank(ctx, s);
  B2_RETURN_NOT_OK(b2_take(ctx, &rank_arr, &indices.a, /*boundscheck=*/0, &row_rank.a, s));
  row_rank.owned = true;
  return sort_into(ctx, &row_rank.a, /*Ascending=*/0, null_placement, payload, out, s);
}

// Whether the dictionary path should sort this column.  A strided 64Ki-row sample is counted on the device
// (b2_vector_hash with counts; null rows are left out) and the column's distinct values are estimated from the sample's
// frequencies with the bias-corrected Chao1 estimator, D = d + f1 (f1 - 1) / (2 (f2 + 1)) (d distinct sample values,
// f1 / f2 of them seen once / twice), capped at the column's estimated valid rows.  A plain sample duplicate share
// would call a column of 500M rows over 1M words 97 % distinct: a sample this small rarely sees a word twice.
int choose_dictionary(B2Context* ctx, const B2Array* values, bool* dict, cudaStream_t s) {
  *dict = false;
  const int64_t n = values->length;
  if (n < 4 * kSample) return B2_OK;
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
  PoolArray sample(ctx, s), uniq(ctx, s), counts(ctx, s);
  B2_RETURN_NOT_OK(b2_take(ctx, values, &ridx, 0, &sample.a, s));
  sample.owned = true;
  B2_RETURN_NOT_OK(b2_vector_hash(ctx, &sample.a, /*MASK=*/0, nullptr, &uniq.a, &counts.a, s));
  uniq.owned = counts.owned = true;
  const int64_t d = counts.a.length;
  std::vector<int64_t> c(d);
  if (d > 0) B2_CUDA(cudaMemcpyAsync(c.data(), counts.a.data, sizeof(int64_t) * (size_t)d, cudaMemcpyDeviceToHost, s));
  B2_CUDA(cudaStreamSynchronize(s));
  int64_t valid = 0, f1 = 0, f2 = 0;
  for (int64_t x : c) {
    valid += x;
    f1 += x == 1;
    f2 += x == 2;
  }
  if (valid == 0) return B2_OK;
  const double column_valid = static_cast<double>(n) * static_cast<double>(valid) / static_cast<double>(kSample);
  double distinct = static_cast<double>(d) + static_cast<double>(f1) * static_cast<double>(f1 - 1) / (2.0 * static_cast<double>(f2 + 1));
  if (distinct > column_valid) distinct = column_valid;
  *dict = column_valid >= kDictRowsPerValue * distinct;
  return B2_OK;
}

}  // namespace

int sort_strings(B2Context* ctx, const B2Array* values, int order, int null_placement, uint64_t* out, cudaStream_t s,
                 const uint32_t* payload) {
  bool dict;
  B2_RETURN_NOT_OK(string_sort_path(ctx, values, &dict, s));
  return dict ? sort_dictionary(ctx, values, order, null_placement, out, s, payload)
              : sort_refine(ctx, values, order, null_placement, out, s, payload);
}

int string_sort_path(B2Context* ctx, const B2Array* values, bool* dict, cudaStream_t s) {
  // B2_SORT_STRINGS_PATH=dict|refine forces a path (tests cover both); otherwise the sample decides
  const char* force = std::getenv("B2_SORT_STRINGS_PATH");
  if (force && std::strcmp(force, "dict") == 0) {
    *dict = true;
    return B2_OK;
  }
  if (force && std::strcmp(force, "refine") == 0) {
    *dict = false;
    return B2_OK;
  }
  return choose_dictionary(ctx, values, dict, s);
}

int string_prefix_keys(B2Context* ctx, const B2Array* values, B2Array* out, cudaStream_t s) {
  const int64_t n = values->length;
  Temp data(ctx, s);
  B2_RETURN_NOT_OK(data.alloc(sizeof(uint64_t) * (size_t)n));
  void* validity = nullptr;
  int64_t null_count = 0;
  B2_RETURN_NOT_OK(make_validity(ctx, values, nullptr, n, &validity, &null_count, s));
  if (n > 0) {
    const uint8_t* chars = static_cast<const uint8_t*>(values->data2);
    if (offset_width(values->type) == 8)
      prefix_keys_kernel<int64_t><<<grid_of(n), kBlock, 0, s>>>(static_cast<const int64_t*>(values->data) + values->offset,
                                                                chars, n, data.as<uint64_t>());
    else
      prefix_keys_kernel<int32_t><<<grid_of(n), kBlock, 0, s>>>(static_cast<const int32_t*>(values->data) + values->offset,
                                                                chars, n, data.as<uint64_t>());
    B2_LAUNCHED();
  }
  fill_out(out, B2_UINT64, n, null_count, validity, data.release());
  return B2_OK;
}

}  // namespace b2

extern "C" int b2_sort_strings_path(B2Context* ctx, const B2Array* values, int32_t* out_path, void* stream) {
  if (!ctx || !values || !out_path) return b2::set_error(B2_INVALID, "b2_sort_strings_path: null argument");
  if (!b2::type_is_binary_like(values->type))
    return b2::set_error(B2_TYPE_ERROR, "b2_sort_strings_path: not a utf8 / binary column (type id %d)", values->type);
  cudaStream_t s = ctx->pick(stream);
  B2_CUDA(cudaSetDevice(ctx->device));
  bool dict = false;
  B2_RETURN_NOT_OK(b2::string_sort_path(ctx, values, &dict, s));
  *out_path = dict ? 1 : 0;
  return B2_OK;
}

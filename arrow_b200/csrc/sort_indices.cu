// sort_indices.cu -- stable argsort of one numeric column: device-wide LSD radix sort.
//
// Replaces:
//   ArraySortIndices::Exec                      kernels/vector_array_sort.cc:524-540
//   ArrayCompareSorter (std::stable_sort with an indirect comparator)   :144-178
//   ArrayCountSorter / ArrayCountOrCompareSorter  :277-446
//   PartitionNullsAndNans / NullLikePartition   kernels/vector_sort_internal.h:113-305
// Semantics kept: output = uint64 indices, never null; the sort is STABLE; nulls are
// stably partitioned to the end (AtEnd) or the start (AtStart); for floats NaNs sit
// between the values and the nulls (values,NaNs,nulls | nulls,NaNs,values); comparator is
// `<` on values, so -0.0 == +0.0 keep index order; Descending keeps ties in ascending
// index order.
//
// B200 design:
//   prepare  : null partition with the Filter machinery (selection = validity bitmap):
//              valid rows emit (ordered-key, row) compacted, null rows go straight to
//              their final slots.  ordered-key: sign-flip for ints, IEEE total-order
//              flip with -0.0 canonicalised for floats, NaN -> all-ones (AtEnd) or 0
//              (AtStart), bitwise NOT for Descending (ties stay in index order).
//   histogram: one read of the keys builds all digit histograms in shared memory.
//   onesweep : per 8-bit digit ONE kernel -- 4096-key tiles (256 threads x 16 keys, 3 CTAs
//              per SM) are claimed through an atomic ticket and ranked stably into
//              per-warp digit counters (lanes with equal digits find each other with one
//              ballot per digit bit -- registers only; MATCH.ANY costs 1.83 cycles/lane on
//              this part); the tile's 256 digit counts are published, keys and indices are
//              staged in shared memory in digit order, and only then the exclusive prefix
//              over earlier tiles is fetched with a 4-deep prefetching decoupled look-back
//              (no global scan pass), so global writes are contiguous runs.  Passes whose
//              digit is constant are skipped; indices stay uint32 until the last executed
//              pass, which writes the uint64 result directly.
// Traffic per executed pass: read (K+4) + write (K+4) bytes per row (K = key bytes).
// Algorithmic bytes (SURVEY section 8d): 16.125 B/row for int64 + validity.
#include <cmath>
#include <type_traits>

#include "selection.cuh"
#include "sort_internal.h"

namespace b2 {

constexpr int kRadixBits = 8;
constexpr int kRadix = 1 << kRadixBits;
constexpr int kSortThreads = 256;
constexpr int kSortWarps = kSortThreads / 32;
constexpr int kSortItems = 16;
constexpr int kSortTile = kSortThreads * kSortItems;  // 4096 keys per tile (2048 measured 16 % slower); 256 x 16 = 3 CTAs/SM beat 512 x 8 by 4 %
constexpr uint32_t kFlagAgg = 1u << 30, kFlagIncl = 2u << 30, kValMask = (1u << 30) - 1u;

// ---- ordered keys ----------------------------------------------------------------------
template <typename T>
struct KeyOf {
  using type = typename std::conditional<sizeof(T) == 8, uint64_t, uint32_t>::type;
};

template <typename T>
__device__ __forceinline__ typename KeyOf<T>::type ordered_key(T v, bool descending, bool nan_first) {
  using K = typename KeyOf<T>::type;
  K k;
  if constexpr (std::is_floating_point<T>::value) {
    using B = typename std::conditional<sizeof(T) == 8, uint64_t, uint32_t>::type;
    if (v != v) return nan_first ? K(0) : ~K(0);
    if (v == T(0)) v = T(0);  // -0.0 -> +0.0: equal under `<`, must tie
    B b;
    memcpy(&b, &v, sizeof(T));
    const B sign = B(1) << (sizeof(T) * 8 - 1);
    k = (b & sign) ? ~b : (b | sign);
    if (descending) k = ~k;
    return k;
  } else if constexpr (std::is_signed<T>::value) {
    using UT = typename std::make_unsigned<T>::type;
    k = static_cast<K>(static_cast<UT>(static_cast<UT>(v) ^ (UT(1) << (sizeof(T) * 8 - 1))));
  } else {
    k = static_cast<K>(v);
  }
  if (descending) {
    k = ~k;
    if constexpr (sizeof(T) < sizeof(K)) k &= (K(1) << (sizeof(T) * 8)) - 1;  // keep unused digits constant
  }
  return k;
}

// ---- prepare: null partition + key transform ---------------------------------------------
template <typename T>
struct PrepareArgs {
  const T* values;  // advanced by offset
  BitmapReader valid;
  const int64_t* tile_offsets;  // exclusive prefix of valid counts per 4096-row tile
  typename KeyOf<T>::type* keys;
  uint32_t* idx;
  uint64_t* out_nulls;  // final slots of the null rows (already offset to the null region)
  const uint32_t* payload;  // NULL: row numbers; else the value that travels with row i instead of i (b2_sort_payload)
  int64_t n;
  bool descending, nan_first;
};

template <typename T>
__global__ void __launch_bounds__(kBlock) sort_prepare_kernel(PrepareArgs<T> a) {
  __shared__ uint64_t s_sel[kTileWords];
  __shared__ uint32_t s_prefix[kTileWords];
  const int64_t tile = blockIdx.x;
  const int64_t row0 = tile * kTileRows;
  if (threadIdx.x < 32) load_tile_prefix(a.valid, tile, s_sel, s_prefix);
  __syncthreads();
  const int64_t vbase = a.tile_offsets[tile];
  const int64_t nbase = row0 - vbase;  // nulls before this tile
  // rows are visited lane-contiguously: row = pass*256 + tid, so a warp's valid rows have
  // consecutive ranks and every store instruction writes a contiguous span
#pragma unroll 4
  for (int p = 0; p < kTileRows / kBlock; ++p) {
    const int r = p * kBlock + threadIdx.x;
    const int64_t row = row0 + r;
    if (row >= a.n) break;
    const uint64_t selw = s_sel[r >> 6];
    const unsigned before = s_prefix[r >> 6] + __popcll(selw & ((1ull << (r & 63)) - 1ull));
    if ((selw >> (r & 63)) & 1) {
      T v = __ldcs(a.values + row);
      a.keys[vbase + before] = ordered_key<T>(v, a.descending, a.nan_first);
      a.idx[vbase + before] = a.payload ? a.payload[row] : static_cast<uint32_t>(row);
    } else {
      a.out_nulls[nbase + (r - before)] = a.payload ? static_cast<uint64_t>(a.payload[row]) : static_cast<uint64_t>(row);
    }
  }
}

// ---- histogram of every digit ------------------------------------------------------------
template <typename K>
__global__ void __launch_bounds__(kSortThreads) radix_hist_kernel(const K* __restrict__ keys, uint32_t n,
                                                                  int passes,
                                                                  unsigned long long* __restrict__ hist) {
  __shared__ uint32_t s_hist[8 * kRadix];
  for (int i = threadIdx.x; i < passes * kRadix; i += kSortThreads) s_hist[i] = 0;
  __syncthreads();
  for (uint64_t i = blockIdx.x * kSortThreads + threadIdx.x; i < n; i += (uint64_t)gridDim.x * kSortThreads) {  // 64-bit: n may be close to 2^32
    K k = __ldcs(keys + i);
#pragma unroll
    for (int p = 0; p < (int)sizeof(K); ++p)
      if (p < passes) atomicAdd(&s_hist[p * kRadix + ((k >> (p * kRadixBits)) & (kRadix - 1))], 1u);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < passes * kRadix; i += kSortThreads)
    if (s_hist[i]) atomicAdd(&hist[i], (unsigned long long)s_hist[i]);
}

// exclusive scan of each pass's 256 bins; trivial[p] = 1 when one bin holds every key
__global__ void __launch_bounds__(kRadix) radix_scan_kernel(const unsigned long long* hist, uint32_t n,
                                                            uint32_t* digit_base, int64_t* trivial) {
  __shared__ uint32_t s[kRadix];
  const int p = blockIdx.x, d = threadIdx.x;
  uint32_t c = static_cast<uint32_t>(hist[p * kRadix + d]);
  s[d] = c;
  __syncthreads();
  if (d == 0) {
    uint32_t run = 0;
    bool triv = false;
    for (int i = 0; i < kRadix; ++i) {
      uint32_t v = s[i];
      if (v == n) triv = true;
      s[i] = run;
      run += v;
    }
    trivial[p] = triv ? 1 : 0;
  }
  __syncthreads();
  digit_base[p * kRadix + d] = s[d];
}

// ---- one radix pass ---------------------------------------------------------------------
template <typename K>
struct OnesweepArgs {
  const K* keys_in;
  const uint32_t* idx_in;
  K* keys_out;
  uint32_t* idx_out;
  uint64_t* final_out;  // LAST pass: uint64 indices
  uint32_t n;
  int shift;
  const uint32_t* digit_base;  // [256] exclusive bin offsets of this pass
  void* lookback;              // [n_tiles][256] cells (uint32, or uint64 for >= 2^30 rows), zeroed
  uint32_t* ticket;            // zeroed
};

template <typename K>
constexpr size_t onesweep_smem() {
  return kSortTile * sizeof(K) + kSortTile * sizeof(uint32_t) + kSortWarps * kRadix * sizeof(uint32_t) +
         kRadix * sizeof(uint32_t);
}

// WIDE: 64-bit look-back cells -- an inclusive prefix no longer fits 30 bits once the column has 2^30 rows
template <typename K, bool LAST, bool WIDE>
__global__ void __launch_bounds__(kSortThreads, 3) onesweep_kernel(OnesweepArgs<K> a) {
  extern __shared__ __align__(16) uint8_t smem[];
  K* s_keys = reinterpret_cast<K*>(smem);
  uint32_t* s_idx = reinterpret_cast<uint32_t*>(s_keys + kSortTile);
  uint32_t* s_cnt = s_idx + kSortTile;              // [warps][256] counts, then tile-local offsets
  uint32_t* s_gbase = s_cnt + kSortWarps * kRadix;  // [256] global base - local bin offset
  __shared__ uint32_t s_tile;
  __shared__ uint32_t s_warp_tot[kRadix / 32];

  const unsigned tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) s_tile = atomicAdd(a.ticket, 1u);
  for (int i = tid; i < kSortWarps * kRadix; i += kSortThreads) s_cnt[i] = 0;
  __syncthreads();
  const uint32_t tile = s_tile;
  const uint32_t base = tile * kSortTile;
  const uint32_t tile_n = (a.n - base) < (uint32_t)kSortTile ? (a.n - base) : (uint32_t)kSortTile;

  // warp-striped loads of keys AND indices up front: item j of lane l is element
  // warp*(32*ITEMS) + j*32 + l of the tile; 2*ITEMS independent requests per lane in flight
  K key[kSortItems];
  uint32_t idxv[kSortItems];
#pragma unroll
  for (int j = 0; j < kSortItems; ++j) {
    const uint32_t i = warp * (32 * kSortItems) + j * 32 + lane;
    key[j] = i < tile_n ? __ldcs(a.keys_in + base + i) : ~K(0);
  }
#pragma unroll
  for (int j = 0; j < kSortItems; ++j) {
    const uint32_t i = warp * (32 * kSortItems) + j * 32 + lane;
    idxv[j] = (i < tile_n && a.idx_in) ? __ldcs(a.idx_in + base + i) : base + i;
  }
  // rank within the warp's segment, in element order (=> stable).  Lanes holding the same digit
  // find each other with 8 ballots (one per digit bit) -- registers only; the kernel is bound by
  // shared-memory wavefronts (ncu: 51 % short-scoreboard + MIO stalls, 58 % of the wavefronts
  // bank conflicts of random digits), and MATCH.ANY costs 1.83 cycles/lane on this part
  // (profiles/smem_probe_r01.txt).  Only the lowest lane of a group touches the warp's counter.
  uint32_t* wc = s_cnt + warp * kRadix;
  uint16_t rank[kSortItems];
  const unsigned lt = lanemask_lt();
#pragma unroll
  for (int j = 0; j < kSortItems; ++j) {
    const unsigned digit = static_cast<unsigned>(key[j] >> a.shift) & (kRadix - 1);
    unsigned peers = 0xffffffffu;
#pragma unroll
    for (int b = 0; b < kRadixBits; ++b) {
      const bool bit = (digit >> b) & 1u;
      const unsigned bal = __ballot_sync(0xffffffffu, bit);
      peers &= bit ? bal : ~bal;
    }
    const int leader = __ffs(peers) - 1;
    unsigned prev = 0;
    if ((int)lane == leader) {
      prev = wc[digit];
      wc[digit] = prev + __popc(peers);
    }
    prev = __shfl_sync(0xffffffffu, prev, leader);
    rank[j] = static_cast<uint16_t>(prev + __popc(peers & lt));
    __syncwarp();  // the next item's leader may be another lane reading the counter just written
  }
  __syncthreads();

  // threads 0..255 each own one digit: exclusive scan over warps, tile count, look-back
  uint32_t run = 0, count = 0, incl = 0;
  if (tid < kRadix) {
#pragma unroll
    for (int w = 0; w < kSortWarps; ++w) {
      uint32_t c = s_cnt[w * kRadix + tid];
      s_cnt[w * kRadix + tid] = run;
      run += c;
    }
    count = run;
    if (tid == kRadix - 1) count -= (kSortTile - tile_n);  // padding keys are all-ones
    if (WIDE) {
      volatile unsigned long long* lb = static_cast<volatile unsigned long long*>(a.lookback);
      if (tile == 0) lb[tid] = (2ull << 62) | count;
      else lb[(size_t)tile * kRadix + tid] = (1ull << 62) | count;
    } else {
      volatile uint32_t* lb = static_cast<volatile uint32_t*>(a.lookback);
      if (tile == 0) lb[tid] = kFlagIncl | count;
      else lb[(size_t)tile * kRadix + tid] = kFlagAgg | count;
    }
    // block exclusive scan of `run` over the 256 digits (padding only occupies the tail of bin 255)
    incl = run;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      uint32_t v = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += v;
    }
    if (lane == 31) s_warp_tot[warp] = incl;
  }
  __syncthreads();
  uint32_t bin_off = 0;
  if (tid < kRadix) {
    uint32_t woff = 0;
#pragma unroll
    for (int w = 0; w < kRadix / 32; ++w)
      if (w < (int)warp) woff += s_warp_tot[w];
    bin_off = woff + incl - run;
    // fold the digit's tile-local start into the per-warp offsets: one lookup per key when staging
#pragma unroll
    for (int w = 0; w < kSortWarps; ++w) s_cnt[w * kRadix + tid] += bin_off;
  }
  __syncthreads();

  // stage keys and indices in digit order first: it needs only tile-local offsets, and it gives
  // the predecessors time to publish before the look-back below has to wait for them
#pragma unroll
  for (int j = 0; j < kSortItems; ++j) {
    const unsigned digit = static_cast<unsigned>(key[j] >> a.shift) & (kRadix - 1);
    const uint32_t pos = wc[digit] + rank[j];
    s_keys[pos] = key[j];
    s_idx[pos] = idxv[j];
  }
  if (tid < kRadix) {
    uint32_t excl = 0;
    if (tile > 0) {
      if (WIDE) {
        volatile unsigned long long* lb = static_cast<volatile unsigned long long*>(a.lookback);
        const unsigned long long e = lookback_exclusive64(lb + tid, tile, kRadix);
        lb[(size_t)tile * kRadix + tid] = (2ull << 62) | (e + count);
        excl = static_cast<uint32_t>(e);  // < 2^32: positions stay 32-bit
      } else {
        volatile uint32_t* lb = static_cast<volatile uint32_t*>(a.lookback);
        excl = lookback_exclusive(lb + tid, tile, kRadix);
        lb[(size_t)tile * kRadix + tid] = kFlagIncl | (excl + count);
      }
    }
    s_gbase[tid] = a.digit_base[tid] + excl - bin_off;
  }
  __syncthreads();
  // contiguous runs out
#pragma unroll
  for (int j = 0; j < kSortItems; ++j) {
    const uint32_t p = j * kSortThreads + tid;
    if (p < tile_n) {
      const K k = s_keys[p];
      const unsigned digit = static_cast<unsigned>(k >> a.shift) & (kRadix - 1);
      const uint32_t dst = s_gbase[digit] + p;
      if (LAST) {
        a.final_out[dst] = static_cast<uint64_t>(s_idx[p]);
      } else {
        a.keys_out[dst] = k;
        a.idx_out[dst] = s_idx[p];
      }
    }
  }
}

__global__ void __launch_bounds__(kBlock) widen_idx_kernel(const uint32_t* in, uint64_t* out, int64_t n) {
  for (int64_t i = blockIdx.x * (int64_t)kBlock + threadIdx.x; i < n; i += (int64_t)gridDim.x * kBlock)
    out[i] = in[i];
}

template <typename T>
static int sort_typed(B2Context* ctx, const B2Array* values, int order, int null_placement, uint64_t* out,
                      cudaStream_t s, const uint32_t* payload = nullptr) {
  using K = typename KeyOf<T>::type;
  const int64_t n = values->length;
  const bool descending = order == 1, at_start = null_placement == 0;

  // 1. null partition plan (selection = validity bitmap)
  FilterBitmaps fb;
  fb.mask_data = BitmapReader(values->null_count == 0 ? nullptr : values->validity, values->offset, n);
  fb.mask_valid = BitmapReader(nullptr, 0, n);
  fb.values_valid = BitmapReader(nullptr, 0, n);
  fb.emit_null = 0;
  Temp offsets(ctx, s);
  int64_t nv = 0, unused = 0;
  B2_RETURN_NOT_OK(filter_plan(ctx, fb, n, false, &offsets, &nv, &unused, s));
  const int64_t nn = n - nv;

  Temp keysA(ctx, s), keysB(ctx, s), idxA(ctx, s), idxB(ctx, s);
  B2_RETURN_NOT_OK(keysA.alloc(sizeof(K) * (size_t)nv));
  B2_RETURN_NOT_OK(idxA.alloc(sizeof(uint32_t) * (size_t)nv));
  uint64_t* out_values = out + (at_start ? nn : 0);
  uint64_t* out_nulls = out + (at_start ? 0 : nv);
  {
    PrepareArgs<T> pa;
    pa.values = static_cast<const T*>(values->data) + values->offset;
    pa.valid = fb.mask_data;
    pa.tile_offsets = offsets.as<int64_t>();
    pa.keys = keysA.as<K>();
    pa.idx = idxA.as<uint32_t>();
    pa.out_nulls = out_nulls;
    pa.payload = payload;
    pa.n = n;
    pa.descending = descending;
    pa.nan_first = at_start;
    sort_prepare_kernel<T><<<(unsigned)tiles_for(n), kBlock, 0, s>>>(pa);
    B2_LAUNCHED();
  }
  if (nv == 0) return B2_OK;

  // 2. the radix passes; the last one writes the uint64 result
  K* unused_keys;
  uint32_t* unused_idx;
  return radix_sort_pairs<K>(ctx, sizeof(T), keysA.as<K>(), idxA.as<uint32_t>(), &keysB, &idxB, (uint32_t)nv, out_values,
                             &unused_keys, &unused_idx, s);
}

template <typename K>
int radix_sort_pairs(B2Context* ctx, int passes, K* keys_a, uint32_t* idx_a, Temp* keys_b, Temp* idx_b, uint32_t n,
                     uint64_t* final_out, K** keys_out, uint32_t** idx_out, cudaStream_t s) {
  *keys_out = keys_a;
  *idx_out = idx_a;
  if (n == 0) return B2_OK;
  // histograms of all digits
  Temp hist(ctx, s), dbase(ctx, s);
  B2_RETURN_NOT_OK(hist.alloc(sizeof(unsigned long long) * 8 * kRadix));
  B2_RETURN_NOT_OK(dbase.alloc(sizeof(uint32_t) * 8 * kRadix));
  B2_CUDA(cudaMemsetAsync(hist.ptr, 0, sizeof(unsigned long long) * 8 * kRadix, s));
  ScalarSlot slot(ctx);
  B2_RETURN_NOT_OK(slot.zero(s));
  {
    int grid = grid_for(n, kSortThreads * 16, kSMs * 8);
    radix_hist_kernel<K><<<grid, kSortThreads, 0, s>>>(keys_a, n, passes, hist.as<unsigned long long>());
    B2_LAUNCHED();
    radix_scan_kernel<<<passes, kRadix, 0, s>>>(hist.as<unsigned long long>(), n, dbase.as<uint32_t>(), slot.dev());
    B2_LAUNCHED();
  }
  B2_RETURN_NOT_OK(slot.fetch(s));
  int todo[8], n_todo = 0;
  for (int p = 0; p < passes; ++p)
    if (!slot.host()[p]) todo[n_todo++] = p;

  if (n_todo == 0) {
    if (final_out) {
      widen_idx_kernel<<<grid_for(n, kBlock * 4, kSMs * 8), kBlock, 0, s>>>(idx_a, final_out, n);
      B2_LAUNCHED();
    }
    return B2_OK;
  }
  if (n_todo > 1 || !final_out) {
    if (!keys_b->ptr) B2_RETURN_NOT_OK(keys_b->alloc(sizeof(K) * (size_t)n));
    if (!idx_b->ptr) B2_RETURN_NOT_OK(idx_b->alloc(sizeof(uint32_t) * (size_t)n));
  }
  const uint32_t n_tiles = (uint32_t)((n + kSortTile - 1) / kSortTile);
  Temp lookback(ctx, s);
  const bool wide = n >= (1u << 30);
  const size_t cell = wide ? sizeof(unsigned long long) : sizeof(uint32_t);
  const size_t lb_bytes = (size_t)n_tiles * kRadix * cell + 256;
  B2_RETURN_NOT_OK(lookback.alloc(lb_bytes));
  uint32_t* ticket = reinterpret_cast<uint32_t*>(lookback.as<char>() + (size_t)n_tiles * kRadix * cell);
  // the attribute is per DEVICE (a process may sort on several): set it on every call, it is cheap
  constexpr size_t smem = onesweep_smem<K>();
  B2_CUDA(cudaFuncSetAttribute(onesweep_kernel<K, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  B2_CUDA(cudaFuncSetAttribute(onesweep_kernel<K, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  B2_CUDA(cudaFuncSetAttribute(onesweep_kernel<K, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  B2_CUDA(cudaFuncSetAttribute(onesweep_kernel<K, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  K* kin = keys_a;
  K* kout = keys_b->as<K>();
  uint32_t* iin = idx_a;
  uint32_t* iout = idx_b->as<uint32_t>();
  for (int t = 0; t < n_todo; ++t) {
    const int p = todo[t];
    const bool last = final_out && t == n_todo - 1;
    B2_CUDA(cudaMemsetAsync(lookback.ptr, 0, lb_bytes, s));
    OnesweepArgs<K> a;
    a.keys_in = kin;
    a.idx_in = iin;
    a.keys_out = kout;
    a.idx_out = iout;
    a.final_out = final_out;
    a.n = n;
    a.shift = p * kRadixBits;
    a.digit_base = dbase.as<uint32_t>() + p * kRadix;
    a.lookback = lookback.ptr;
    a.ticket = ticket;
    if (wide) {
      if (last) onesweep_kernel<K, true, true><<<n_tiles, kSortThreads, smem, s>>>(a);
      else onesweep_kernel<K, false, true><<<n_tiles, kSortThreads, smem, s>>>(a);
    } else {
      if (last) onesweep_kernel<K, true, false><<<n_tiles, kSortThreads, smem, s>>>(a);
      else onesweep_kernel<K, false, false><<<n_tiles, kSortThreads, smem, s>>>(a);
    }
    B2_LAUNCHED();
    K* tk = kin; kin = kout; kout = tk;
    uint32_t* ti = iin; iin = iout; iout = ti;
  }
  *keys_out = kin;
  *idx_out = iin;
  return B2_OK;
}

template int radix_sort_pairs<uint32_t>(B2Context*, int, uint32_t*, uint32_t*, Temp*, Temp*, uint32_t, uint64_t*,
                                        uint32_t**, uint32_t**, cudaStream_t);
template int radix_sort_pairs<uint64_t>(B2Context*, int, uint64_t*, uint32_t*, Temp*, Temp*, uint32_t, uint64_t*,
                                        uint64_t**, uint32_t**, cudaStream_t);

}  // namespace b2

using namespace b2;

static int sort_run(B2Context* ctx, const B2Array* values, int order, int null_placement, const uint32_t* payload, B2Array* out, void* stream);

extern "C" int b2_sort_indices(B2Context* ctx, const B2Array* values, int order, int null_placement,
                               B2Array* out, void* stream) {
  return sort_run(ctx, values, order, null_placement, nullptr, out, stream);
}

extern "C" int b2_sort_payload(B2Context* ctx, const B2Array* values, const B2Array* payload, int order, int null_placement,
                               B2Array* out, void* stream) {
  if (!payload) return set_error(B2_INVALID, "b2_sort_payload: null argument");
  if (payload->type != B2_UINT32 || payload->null_count > 0 || !values || payload->length != values->length)
    return set_error(B2_INVALID, "b2_sort_payload: payload must be a uint32 array without nulls of the values' length");
  return sort_run(ctx, values, order, null_placement, static_cast<const uint32_t*>(payload->data) + payload->offset, out, stream);
}

static int sort_run(B2Context* ctx, const B2Array* values, int order, int null_placement, const uint32_t* payload, B2Array* out, void* stream) {
  if (!ctx || !values || !out) return set_error(B2_INVALID, "b2_sort_indices: null argument");
  if (order != 0 && order != 1) return set_error(B2_INVALID, "bad sort order %d", order);
  if (null_placement != 0 && null_placement != 1) return set_error(B2_INVALID, "bad null placement %d", null_placement);
  if (values->length < 0 || values->offset < 0) return set_error(B2_INVALID, "negative length/offset");
  if (!type_is_numeric(values->type) && !type_is_binary_like(values->type))
    return set_error(B2_NOT_IMPLEMENTED, "sort_indices: unsupported type id %d", values->type);
  const int64_t n = values->length;
  if (n >= (1ll << 32) - 8192)  // row numbers travel as uint32 between the passes
    return set_error(B2_NOT_IMPLEMENTED, "sort_indices: arrays of 2^32 rows or more must be sorted as chunks");
  cudaStream_t s = ctx->pick(stream);
  B2_CUDA(cudaSetDevice(ctx->device));
  Temp data(ctx, s);
  B2_RETURN_NOT_OK(data.alloc(sizeof(uint64_t) * (size_t)n));
  B2_RETURN_NOT_OK(sort_into(ctx, values, order, null_placement, payload, data.as<uint64_t>(), s));
  fill_out(out, B2_UINT64, n, 0, nullptr, data.release());
  return B2_OK;
}

int b2::sort_into(B2Context* ctx, const B2Array* values, int order, int null_placement, const uint32_t* payload, uint64_t* o,
                  cudaStream_t s) {
  if (values->length == 0) return B2_OK;
  int st;
  switch (values->type) {
    case B2_INT8: st = sort_typed<int8_t>(ctx, values, order, null_placement, o, s, payload); break;
    case B2_UINT8: st = sort_typed<uint8_t>(ctx, values, order, null_placement, o, s, payload); break;
    case B2_INT16: st = sort_typed<int16_t>(ctx, values, order, null_placement, o, s, payload); break;
    case B2_UINT16: st = sort_typed<uint16_t>(ctx, values, order, null_placement, o, s, payload); break;
    case B2_INT32: st = sort_typed<int32_t>(ctx, values, order, null_placement, o, s, payload); break;
    case B2_UINT32: st = sort_typed<uint32_t>(ctx, values, order, null_placement, o, s, payload); break;
    case B2_INT64: st = sort_typed<int64_t>(ctx, values, order, null_placement, o, s, payload); break;
    case B2_UINT64: st = sort_typed<uint64_t>(ctx, values, order, null_placement, o, s, payload); break;
    case B2_FLOAT: st = sort_typed<float>(ctx, values, order, null_placement, o, s, payload); break;
    case B2_STRING: case B2_BINARY: case B2_LARGE_STRING: case B2_LARGE_BINARY:
      st = sort_strings(ctx, values, order, null_placement, o, s, payload);
      break;
    default: st = sort_typed<double>(ctx, values, order, null_placement, o, s, payload); break;
  }
  return st;
}

// Multi-key sort (SortIndices over a record batch / table, kernels/vector_sort.cc:386-600 MultipleKeyRecordBatchSorter
// and :850-1027): rows ordered by keys[0], ties by keys[1], ...; per key its own order, one null placement; nulls (then
// NaNs) of a key compare equal among themselves and fall through to the next key; stable.
//
// B200 design: least-significant key first, every round a STABLE single-key radix sort whose payload is the
// permutation so far -- round k gathers key k through the current permutation (b2_take) and sorts it with the
// permutation riding along the radix passes (sort_run's payload), so no comparator and no per-row key tuple exist.
extern "C" int b2_sort_indices_multi(B2Context* ctx, const B2Array* keys, int n_keys, const int32_t* orders, int null_placement,
                                     B2Array* out, void* stream) {
  if (!ctx || !keys || !orders || !out) return set_error(B2_INVALID, "b2_sort_indices_multi: null argument");
  if (n_keys < 1) return set_error(B2_INVALID, "Must specify one or more sort keys");
  for (int k = 1; k < n_keys; ++k)
    if (keys[k].length != keys[0].length) return set_error(B2_INVALID, "sort keys differ in length");
  cudaStream_t s = ctx->pick(stream);
  PoolArray perm(ctx, s);
  B2_RETURN_NOT_OK(sort_run(ctx, &keys[n_keys - 1], orders[n_keys - 1], null_placement, nullptr, &perm.a, stream));
  perm.owned = true;
  for (int k = n_keys - 2; k >= 0; --k) {
    PoolArray perm32(ctx, s), gathered(ctx, s), next(ctx, s);
    B2CastOptions narrow{B2_UINT32, 1, 1, 0};  // row numbers < 2^32 (sort_run's limit)
    B2_RETURN_NOT_OK(b2_cast_numeric(ctx, &perm.a, &narrow, &perm32.a, stream));
    perm32.owned = true;
    perm.reset();
    B2_RETURN_NOT_OK(b2_take(ctx, &keys[k], &perm32.a, /*boundscheck=*/0, &gathered.a, stream));
    gathered.owned = true;
    B2_RETURN_NOT_OK(sort_run(ctx, &gathered.a, orders[k], null_placement,
                              static_cast<const uint32_t*>(perm32.a.data) + perm32.a.offset, &next.a, stream));
    perm.a = next.a;
    perm.owned = true;
  }
  *out = perm.a;
  perm.owned = false;
  return B2_OK;
}

// selection.cuh -- pieces shared by Filter, GetTakeIndices, var-binary selection and the
// null partition of SortIndices: the selection-word builder and the count + scan passes
// that turn a (mask data, mask validity) bitmap pair into per-tile output offsets.
// See selection_filter.cu for the design notes and reference citations.
#pragma once
#include "bitmap.h"
#include "common.cuh"
#include "context.h"

namespace b2 {

constexpr int kTileRows = 4096;  // rows per compaction tile = 64 bitmap words
constexpr int kTileWords = kTileRows / 64;

struct FilterBitmaps {
  BitmapReader mask_data, mask_valid, values_valid;
  int emit_null;
  // selection word: DROP = data & valid ; EMIT_NULL = data | ~valid
  __device__ __forceinline__ uint64_t sel(int64_t w) const {
    uint64_t d = mask_data.word(w);
    if (!mask_valid.present()) return d;
    uint64_t v = mask_valid.word(w);
    if (!emit_null) return d & v;
    // ~v must not leak past nbits: build the in-range mask from an all-ones reader
    int64_t rem = mask_data.nbits - (w << 6);
    uint64_t in_range = rem >= 64 ? ~0ull : (rem <= 0 ? 0ull : ((1ull << rem) - 1ull));
    return (d | ~v) & in_range;
  }
  // validity of the selected rows before compaction
  __device__ __forceinline__ uint64_t out_valid(int64_t w) const {
    return values_valid.word(w) & mask_valid.word(w);
  }
};

// warp 0 of a compaction tile: the tile's 64 selection words and, per word, the selected rows before it in the tile
// (the rank of row r is s_prefix[r >> 6] + popcount of the bits below r in s_sel[r >> 6])
__device__ __forceinline__ void load_tile_prefix(const BitmapReader& sel, int64_t tile, uint64_t* s_sel, uint32_t* s_prefix) {
  const unsigned lane = lane_id();
  const int64_t w0 = tile * kTileWords + 2 * lane;
  const uint64_t s0 = sel.word(w0), s1 = sel.word(w0 + 1);
  const int c0 = __popcll(s0), c1 = __popcll(s1);
  int incl = c0 + c1;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    int v = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += v;
  }
  const int excl = incl - c0 - c1;
  s_sel[2 * lane] = s0;
  s_sel[2 * lane + 1] = s1;
  s_prefix[2 * lane] = excl;
  s_prefix[2 * lane + 1] = excl + c0;
}

inline int64_t tiles_for(int64_t n) { return (n + kTileRows - 1) / kTileRows; }

// passes 1+2: per-tile exclusive output offsets (int64[n_tiles+1], device), the output
// length and -- when want_valid -- the number of selected rows whose output is valid.
// chunk_rel (optional): uint16 survivors before each 512-row chunk, relative to its tile.
int filter_plan(B2Context* ctx, const FilterBitmaps& fb, int64_t n, bool want_valid, Temp* offsets,
                int64_t* out_length, int64_t* out_valid, cudaStream_t s, Temp* chunk_rel = nullptr);

FilterBitmaps make_filter_bitmaps(const B2Array* values, const B2Array* mask, int null_selection);

}  // namespace b2

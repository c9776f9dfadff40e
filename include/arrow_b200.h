/*
 * arrow_b200.h -- C-ABI of the B200-native execution layer for arrow::compute's
 * ExecBatch hot path (Filter/Take, Cast, arithmetic/compare, SortIndices,
 * Grouper + hash aggregates).
 *
 * This is the drop-in boundary: every entry point below replaces one reference
 * kernel entry (an ArrayKernelExec, a Grouper method or a HashAggregateKernel
 * callback) and takes exactly the information the reference passes through an
 * ArraySpan (cpp/src/arrow/array/data.h:525-690): validity bitmap, data buffer(s),
 * length, offset, null_count, type id -- but with DEVICE addresses.  No torch, no
 * arrow C++ type appears in a signature; the C++ host plugin (arrow_b200/cpp) and
 * the Python ctypes mirror (arrow_b200/_cabi.py) both bind these symbols.
 *
 * Conventions
 *  - every function returns a B2Status (0 = OK); b2_last_error() gives the message
 *    for the calling thread.  Status codes map 1:1 to arrow::StatusCode
 *    (cpp/src/arrow/status.h:86-110) so the trampolines can rebuild the same Status.
 *  - all pointers inside B2Array are device pointers valid on ctx's device.
 *  - validity bitmaps and boolean data are LSB-first bit-packed
 *    (cpp/src/arrow/util/bit_util.h), addressed with `offset` in bits.
 *  - outputs are allocated through the context's allocator (built-in pool, or the
 *    callbacks the host installs with b2_context_set_allocator so memory stays in
 *    the host-side MemoryManager pool); ownership passes to the caller, who
 *    releases with b2_free().
 *  - calls are stream-ordered on `stream` (a cudaStream_t passed as void*; NULL =
 *    the context's own non-blocking stream).  Calls that return a length or a null
 *    count synchronise that stream once before returning (the one unavoidable
 *    read-back, SURVEY.md section 3.5).
 */
#ifndef ARROW_B200_H
#define ARROW_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B2_API __attribute__((visibility("default")))

/* ---- status codes: values follow arrow::StatusCode (status.h:86-110) ---- */
typedef enum B2Status {
  B2_OK = 0,
  B2_OUT_OF_MEMORY = 1,
  B2_KEY_ERROR = 2,
  B2_TYPE_ERROR = 3,
  B2_INVALID = 4,
  B2_IO_ERROR = 5,
  B2_CAPACITY_ERROR = 6,
  B2_INDEX_ERROR = 7,
  B2_CANCELLED = 8,
  B2_UNKNOWN_ERROR = 9,
  B2_NOT_IMPLEMENTED = 10,
  B2_CUDA_ERROR = 100
} B2Status;

/* ---- type ids: values follow arrow::Type::type (type_fwd.h:328-460) ---- */
typedef enum B2Type {
  B2_NA = 0,
  B2_BOOL = 1,
  B2_UINT8 = 2,
  B2_INT8 = 3,
  B2_UINT16 = 4,
  B2_INT16 = 5,
  B2_UINT32 = 6,
  B2_INT32 = 7,
  B2_UINT64 = 8,
  B2_INT64 = 9,
  B2_HALF_FLOAT = 10,
  B2_FLOAT = 11,
  B2_DOUBLE = 12,
  B2_STRING = 13,
  B2_BINARY = 14,
  B2_FIXED_SIZE_BINARY = 15,
  B2_LARGE_STRING = 34,
  B2_LARGE_BINARY = 35
} B2Type;

/* One ArraySpan with device addresses (array/data.h:525-690).
 *   fixed width : data  = values                       (data2 unused)
 *   bool        : data  = bit-packed values
 *   (large_)utf8/binary : data = int32/int64 offsets (length+1 entries, indexed
 *                 from `offset`), data2 = character bytes
 * byte_width is only read for B2_FIXED_SIZE_BINARY. */
typedef struct B2Array {
  const void* validity; /* NULL = no nulls */
  const void* data;
  const void* data2;
  int64_t length;
  int64_t offset;
  int64_t null_count; /* -1 = unknown (kUnknownNullCount) */
  int32_t type;       /* B2Type */
  int32_t byte_width;
} B2Array;

/* A Scalar operand (scalar.h): value bits in `bits` (little-endian, low bytes),
 * is_valid = 0 for a null scalar. */
typedef struct B2Scalar {
  uint64_t bits;
  int32_t type;
  int32_t is_valid;
} B2Scalar;

/* Binary-kernel operand: an array or a scalar (exec.h:275-330 ExecValue). */
typedef struct B2Value {
  const B2Array* array;   /* non-NULL => array operand */
  const B2Scalar* scalar; /* used when array == NULL */
} B2Value;

typedef struct B2Context B2Context;

/* ---------------------------------------------------------------------------
 * Context, device pool, streams.
 * Replaces: arrow::cuda::CudaContext / CudaMemoryManager allocation path
 * (cpp/src/arrow/gpu/cuda_context.cc:110-121 = one cuMemAlloc per buffer) with a
 * size-binned caching pool.
 * ------------------------------------------------------------------------- */
typedef void* (*B2AllocFn)(size_t nbytes, void* stream, void* user);
typedef void (*B2FreeFn)(void* ptr, size_t nbytes, void* stream, void* user);

B2_API int b2_context_create(int device, B2Context** out);
B2_API void b2_context_destroy(B2Context* ctx);
B2_API int b2_context_device(const B2Context* ctx);
B2_API void* b2_context_stream(const B2Context* ctx);
B2_API int b2_context_set_allocator(B2Context* ctx, B2AllocFn alloc, B2FreeFn free_fn,
                                    void* user);
B2_API int b2_alloc(B2Context* ctx, size_t nbytes, void** out);
B2_API int b2_free(B2Context* ctx, void* ptr);
B2_API int b2_pool_stats(const B2Context* ctx, int64_t* bytes_in_use,
                         int64_t* bytes_reserved, int64_t* max_in_use);
B2_API int b2_pool_trim(B2Context* ctx);
B2_API int b2_sync(B2Context* ctx, void* stream);
B2_API int b2_memcpy_h2d(B2Context* ctx, void* dst, const void* src, size_t n, void* stream);
B2_API int b2_memcpy_d2h(B2Context* ctx, void* dst, const void* src, size_t n, void* stream);
B2_API int b2_memset(B2Context* ctx, void* dst, int byte, size_t n, void* stream);
/* Events (cudaEvent_t as void*): the synchronisation object of the C Device Data Interface --
 * ArrowDeviceArray.sync_event is a cudaEvent_t* for ARROW_DEVICE_CUDA (c/abi.h:140-157); the producer
 * records it after the last kernel that writes the buffers, the consumer makes its stream wait on it
 * (arrow::Device::SyncEvent / Stream::WaitEvent, device.h:86-165). */
B2_API int b2_event_create(B2Context* ctx, void** out_event);
B2_API int b2_event_destroy(void* event);
B2_API int b2_event_record(B2Context* ctx, void* event, void* stream);
B2_API int b2_event_synchronize(void* event);
B2_API int b2_stream_wait_event(B2Context* ctx, void* stream, void* event);
/* pinned host staging (CudaHostBuffer, cuda_memory.h:113) */
B2_API int b2_host_alloc(size_t nbytes, void** out);
B2_API int b2_host_free(void* ptr);

B2_API const char* b2_last_error(void);
B2_API const char* b2_version(void);
/* number of kernels this library has launched in this process (bench.py's
 * gpu_launches claim) */
B2_API int64_t b2_launch_count(void);

/* ---------------------------------------------------------------------------
 * Bitmap utilities.  Replaces internal::CopyBitmap / BitmapAnd / CountSetBits
 * (cpp/src/arrow/util/bitmap_ops.cc) as used by NullPropagator
 * (cpp/src/arrow/compute/exec.cc:527-686).
 * ------------------------------------------------------------------------- */
/* number of set bits in bits[offset, offset+length) */
B2_API int b2_bitmap_count(B2Context* ctx, const void* bits, int64_t offset, int64_t length,
                           int64_t* out_count, void* stream);
/* dst[dst_offset..] = src[src_offset..]; dst must be a fresh buffer, padding zeroed */
B2_API int b2_bitmap_copy(B2Context* ctx, const void* src, int64_t src_offset, int64_t length,
                          void* dst, void* stream);
/* dst = a & b (either may be NULL = all ones); returns popcount if out_count != NULL */
B2_API int b2_bitmap_and(B2Context* ctx, const void* a, int64_t a_offset, const void* b,
                         int64_t b_offset, int64_t length, void* dst, int64_t* out_count,
                         void* stream);

/* ---------------------------------------------------------------------------
 * Cast.  Replaces CastNumberToNumberUnsafe + the safety checks
 * (kernels/scalar_cast_internal.cc:41-53,155; kernels/scalar_cast_numeric.cc:45-279).
 * out is allocated by the callee (data + validity copy at offset 0).
 * ------------------------------------------------------------------------- */
typedef struct B2CastOptions { /* compute/cast.h CastOptions */
  int32_t to_type;
  int32_t allow_int_overflow;
  int32_t allow_float_truncate;
  int32_t reserved;
} B2CastOptions;
B2_API int b2_cast_numeric(B2Context* ctx, const B2Array* in, const B2CastOptions* options,
                           B2Array* out, void* stream);

/* ---------------------------------------------------------------------------
 * Arithmetic.  Replaces ScalarBinary<..>::{ArrayArray,ArrayScalar,ScalarArray}
 * with the Add/Subtract/Multiply(+Checked)/Divide op functors
 * (kernels/codegen_internal.h:813-976, kernels/base_arithmetic_internal.h:44-330).
 * Both operands must already have the same (dispatched) type, as after
 * ArithmeticFunction::DispatchBest (kernels/scalar_arithmetic.cc:734-781).
 * ------------------------------------------------------------------------- */
typedef enum B2ArithOp {
  B2_ADD = 0,
  B2_SUBTRACT = 1,
  B2_MULTIPLY = 2,
  B2_DIVIDE = 3,
  B2_ADD_CHECKED = 16,
  B2_SUBTRACT_CHECKED = 17,
  B2_MULTIPLY_CHECKED = 18,
  B2_DIVIDE_CHECKED = 19
} B2ArithOp;
B2_API int b2_binary_arith(B2Context* ctx, int op, const B2Value* left, const B2Value* right,
                           B2Array* out, void* stream);

/* ---------------------------------------------------------------------------
 * Compare -> bit-packed boolean.  Replaces CompareKernel::Exec
 * (kernels/scalar_compare.cc:164-303).  less/less_equal are the flipped
 * greater/greater_equal exactly as MakeFlippedCompare does (:910).
 * ------------------------------------------------------------------------- */
typedef enum B2CompareOp {
  B2_EQUAL = 0,
  B2_NOT_EQUAL = 1,
  B2_GREATER = 2,
  B2_GREATER_EQUAL = 3,
  B2_LESS = 4,
  B2_LESS_EQUAL = 5
} B2CompareOp;
B2_API int b2_compare(B2Context* ctx, int op, const B2Value* left, const B2Value* right,
                      B2Array* out, void* stream);

/* ---------------------------------------------------------------------------
 * Boolean logic and validity predicates (what a filter Expression is made of; SURVEY.md 8f rank 3).
 * Replaces AndOp / OrOp / XorOp / AndNotOp / InvertOp and the Kleene variants
 * (kernels/scalar_boolean.cc:30-270) and IsValidExec / IsNullExec / TrueUnlessNullExec / is_nan
 * (kernels/scalar_validity.cc:35-311; NullOptions{nan_is_null} compute/api_scalar.h).
 * Operands are B2_BOOL arrays (or one B2_BOOL scalar); `right` is NULL for B2_BOOL_INVERT.
 * ------------------------------------------------------------------------- */
typedef enum B2BooleanOp {
  B2_BOOL_AND = 0,
  B2_BOOL_OR = 1,
  B2_BOOL_XOR = 2,
  B2_BOOL_AND_NOT = 3,
  B2_BOOL_AND_KLEENE = 4,
  B2_BOOL_OR_KLEENE = 5,
  B2_BOOL_AND_NOT_KLEENE = 6,
  B2_BOOL_INVERT = 7
} B2BooleanOp;
B2_API int b2_boolean(B2Context* ctx, int op, const B2Value* left, const B2Value* right, B2Array* out,
                      void* stream);
typedef enum B2ValidityOp {
  B2_IS_VALID = 0,
  B2_IS_NULL = 1,          /* nan_is_null != 0: NaN values of float arrays count as null too */
  B2_TRUE_UNLESS_NULL = 2,
  B2_IS_NAN = 3            /* float32 / float64 only; null in -> null out */
} B2ValidityOp;
B2_API int b2_validity(B2Context* ctx, int op, const B2Array* in, int nan_is_null, B2Array* out,
                       void* stream);

/* if_else(cond, left, right).  Replaces IfElseFunctor<Type>::Call and the AAA/ASA/AAS/ASS shapes
 * (kernels/scalar_if_else.cc:62-520): out = cond ? left : right; out is null where cond is null or the chosen side
 * is.  cond: boolean array or scalar; left / right: arrays or scalars of ONE fixed-width numeric or boolean type (the
 * caller applies DispatchBest's casts); at least one of the three is an array, arrays agree in length
 * (else B2_INVALID "Array arguments must all be the same length"). */
B2_API int b2_if_else(B2Context* ctx, const B2Value* cond, const B2Value* left, const B2Value* right,
                      B2Array* out, void* stream);

/* ---------------------------------------------------------------------------
 * Filter.  Replaces PrimitiveFilterExec / BinaryFilterExec /
 * DictionaryFilterExec (kernels/vector_selection_filter_internal.cc:445-510,
 * 806-856,871-881) and GetFilterOutputSize (:62-114).
 * null_selection: 0 = DROP, 1 = EMIT_NULL (compute/api_vector.h:37-51).
 * mask is a B2_BOOL array.
 * ------------------------------------------------------------------------- */
B2_API int b2_filter_output_size(B2Context* ctx, const B2Array* mask, int null_selection,
                                 int64_t* out_length, void* stream);
B2_API int b2_filter(B2Context* ctx, const B2Array* values, const B2Array* mask,
                     int null_selection, B2Array* out, void* stream);
/* mask -> selection indices (GetTakeIndices, vector_selection_take_internal.cc:62-305);
 * out type is B2_UINT32 if mask length <= UINT32_MAX else error as the reference. */
B2_API int b2_filter_indices(B2Context* ctx, const B2Array* mask, int null_selection,
                             B2Array* out, void* stream);

/* ---------------------------------------------------------------------------
 * Take.  Replaces FixedWidthTakeExec / Gather / VarBinaryTakeExec / DictionaryTake
 * (kernels/vector_selection_take_internal.cc:336-497, kernels/gather_internal.h:84-251)
 * and CheckIndexBounds (util/int_util.cc:452-560).
 * ------------------------------------------------------------------------- */
B2_API int b2_take(B2Context* ctx, const B2Array* values, const B2Array* indices,
                   int boundscheck, B2Array* out, void* stream);

/* Fused Take -> Cast -> arithmetic: out[i] = op(cast<to_type>(values[indices[i]]), other[i]) in one pass, i.e. the
 * Expression add(cast(take(values, indices), T), other) that ExecuteScalarExpression (compute/expression.cc:722-797) runs
 * as three kernels with two materialised intermediates.  Results are identical to b2_take + b2_cast_numeric(unsafe) +
 * b2_binary_arith: same validity (indices AND values-at-index AND other), same IndexError, one IEEE operation per slot.
 * values: float64 / float32 / int64 / int32; indices: 32- or 64-bit integers; to_type: B2_FLOAT or B2_DOUBLE;
 * op: B2_ADD / B2_SUBTRACT / B2_MULTIPLY; other: array (or valid scalar) of to_type. */
B2_API int b2_take_cast_arith(B2Context* ctx, const B2Array* values, const B2Array* indices, int32_t to_type, int op,
                              const B2Value* other, B2Array* out, void* stream);

/* Bytes of character data a (large_)utf8/binary array spans: offsets[offset+length] -
 * offsets[offset] (one D2H read).  Lets the host size the data buffer of an output the
 * way BufferSpan::size does (array/data.h:525-532). */
B2_API int b2_binary_data_size(B2Context* ctx, const B2Array* array, int64_t* out_bytes, void* stream);

/* ---------------------------------------------------------------------------
 * SortIndices.  Replaces ArraySortIndices::Exec + ArrayCompareSorter /
 * ArrayCountSorter (kernels/vector_array_sort.cc:144-446,524-540) and
 * PartitionNullsAndNans (kernels/vector_sort_internal.h:113-305).
 * order: 0 = Ascending, 1 = Descending; null_placement: 0 = AtStart, 1 = AtEnd
 * (compute/ordering.h:30-44).  out: B2_UINT64, length = values.length, no nulls.
 * values: a numeric column, or a B2_STRING / B2_BINARY / B2_LARGE_STRING / B2_LARGE_BINARY column ordered
 * unsigned byte-wise with a proper prefix first (ArrayCompareSorter over base-binary types,
 * kernels/vector_array_sort.cc:144-178,588-594; csrc/sort_strings.cu).  Fewer than 2^32 - 8192 rows;
 * character data of any size.  fixed_size_binary, string_view, dictionary and nested values are
 * B2_NOT_IMPLEMENTED.
 * ------------------------------------------------------------------------- */
B2_API int b2_sort_indices(B2Context* ctx, const B2Array* values, int order,
                           int null_placement, B2Array* out, void* stream);
/* The same stable sort (same value types), but row i carries payload[i] (B2_UINT32, no nulls) instead of its row number i:
 * out[k] = payload of the k-th row in sorted order (B2_UINT64).  The owner GPU of the distributed SortIndices sorts the
 * received (key, global row) pairs with it, so the row numbers ride along the radix passes instead of being gathered
 * afterwards (b2_sort_indices + b2_take = a second, random-access-bound pass). */
B2_API int b2_sort_payload(B2Context* ctx, const B2Array* values, const B2Array* payload, int order,
                           int null_placement, B2Array* out, void* stream);
/* Multi-key SortIndices (record batch / table sort, kernels/vector_sort.cc:386-600,850-1027): rows ordered by keys[0],
 * ties by keys[1], ...; orders[k] = 0 ascending / 1 descending per key; one null placement (0 = AtStart, 1 = AtEnd); stable.  Every key column
 * is numeric or utf8 / binary (as b2_sort_indices; MultipleKeyRecordBatchSorter over base-binary columns,
 * kernels/vector_sort.cc:386-600) and of the same length (< 2^32 - 8192 rows).  out: B2_UINT64 row indices. */
B2_API int b2_sort_indices_multi(B2Context* ctx, const B2Array* keys, int n_keys, const int32_t* orders,
                                 int null_placement, B2Array* out, void* stream);

/* The path b2_sort_indices / b2_sort_payload take for this utf8 / binary column: *out_path = 0 prefix refinement,
 * 1 dictionary (csrc/sort_strings.cu).  The environment variable B2_SORT_STRINGS_PATH=dict|refine forces a path;
 * otherwise a strided sample estimates the column's rows per distinct value.  Benchmarks label their measurements with
 * it and tests pin the selection. */
B2_API int b2_sort_strings_path(B2Context* ctx, const B2Array* values, int32_t* out_path, void* stream);

/* select_k_unstable over one numeric or utf8 / binary column (ArraySelector, kernels/vector_select_k.cc:157-232, and
 * its base-binary instantiations): out = the B2_UINT64 indices of the first min(k, length) rows in sort order =
 * b2_sort_indices(...)[0:k] (ties in row order).  For k << n the column is read once: a sampled threshold, one compare
 * pass, a sort of the few candidates (csrc/select_k.cu); strings are thresholded on their first 7 bytes. */
B2_API int b2_select_k(B2Context* ctx, const B2Array* values, int64_t k, int order, int null_placement,
                       B2Array* out, void* stream);

/* ---------------------------------------------------------------------------
 * Hash join: the matching row pairs of an equi-join.  Replaces the build / probe / match core of HashJoinNode
 * (acero/hash_join_node.cc, acero/swiss_join.cc; JoinType acero/options.h:365-374, JoinKeyCmp::EQ :384-392: a null key
 * matches nothing).  left_keys / right_keys: n_keys columns each, pairwise of equal type (anything the Grouper takes).
 *   INNER       out_left[k], out_right[k] (B2_UINT32, no nulls) = the k-th matching pair
 *   LEFT_OUTER  as INNER plus one pair per unmatched left row whose out_right slot is null
 *   FULL_OUTER  as LEFT_OUTER, followed by one pair per unmatched right row whose out_left slot is null
 *   LEFT_SEMI / LEFT_ANTI   out_left = the left rows with / without a match (out_right may be NULL)
 * Pairs come in left-row order, the matches of one left row in right-row order (the reference's order is unspecified).
 * The caller gathers the payload columns with b2_take, as HashJoinNode's materialize step does.
 * ------------------------------------------------------------------------- */
typedef enum B2JoinType {
  B2_JOIN_INNER = 0,
  B2_JOIN_LEFT_OUTER = 1,
  B2_JOIN_LEFT_SEMI = 2,
  B2_JOIN_LEFT_ANTI = 3,
  B2_JOIN_FULL_OUTER = 4
} B2JoinType;
B2_API int b2_hash_join(B2Context* ctx, const B2Array* left_keys, const B2Array* right_keys, int n_keys, int join_type,
                        B2Array* out_left, B2Array* out_right, void* stream);

/* ---------------------------------------------------------------------------
 * Grouper.  Replaces Grouper::{Make,Consume,Lookup,GetUniques,num_groups,Reset}
 * (compute/row/grouper.h:104-196; GrouperFastImpl row/grouper.cc:555-963, GrouperImpl :300-553)
 * for 1..8 key columns, each fixed-width numeric (1/2/4/8 bytes) or utf8 / binary / large_utf8 /
 * large_binary.  Keys that pack into 64 bits use one table (csrc/grouper.cu); wider keys and string
 * keys are reduced part by part to 32-bit ids and folded (csrc/grouper_wide.cu; strings through a
 * 64-bit hash whose every row is verified against the stored key bytes).
 * Group ids are dense uint32 assigned in first-occurrence row order.
 * ------------------------------------------------------------------------- */
typedef struct B2Grouper B2Grouper;
B2_API int b2_grouper_create(B2Context* ctx, const int32_t* key_types, int n_keys,
                             B2Grouper** out);
B2_API void b2_grouper_destroy(B2Grouper* g);
/* keys: n_keys arrays of equal length; out_ids: B2_UINT32 array, no nulls */
B2_API int b2_grouper_consume(B2Grouper* g, const B2Array* keys, B2Array* out_ids,
                              void* stream);
/* as consume but never inserts; unknown keys give null ids */
B2_API int b2_grouper_lookup(B2Grouper* g, const B2Array* keys, B2Array* out_ids,
                             void* stream);
B2_API int b2_grouper_num_groups(const B2Grouper* g, uint32_t* out);
/* out_keys: n_keys arrays, each num_groups long, in group-id order */
B2_API int b2_grouper_uniques(B2Grouper* g, B2Array* out_keys, void* stream);
B2_API int b2_grouper_reset(B2Grouper* g);

/* ---------------------------------------------------------------------------
 * Ungrouped sum / mean / min_max / count of one numeric column: everything the
 * reference's scalar-aggregate states keep, in one pass.  Replaces SumImpl / MeanImpl
 * (compute/kernels/aggregate_basic.inc.cc:49-107,227-290), MinMaxState / MinMaxImpl
 * (:657-701,776-860) and CountImpl (compute/kernels/aggregate_basic.cc:98-130); the
 * caller applies ScalarAggregateOptions{skip_nulls, min_count} (compute/api_aggregate.h:48-50)
 * the way their Finalize does.
 * ------------------------------------------------------------------------- */
typedef struct B2ReduceResult {
  int64_t count;      /* valid (non-null) rows */
  int64_t null_count; /* length - count */
  uint64_t sum_bits;  /* sum over valid rows in acc_type: int64 (wrapping) / uint64 / double bits */
  uint64_t min_bits;  /* min over valid rows widened to int64 / uint64 / double bits; the type's
                         anti-extremum (NaN for floats) when count == 0 or every value is NaN */
  uint64_t max_bits;
  uint64_t dsum_bits; /* the sum as a double for MeanImpl's sum / count (:263-283): floats = sum_bits,
                         integers = the exact 128-bit sum rounded once (never the int64 wrap-around) */
  int32_t acc_type;   /* B2_INT64, B2_UINT64 or B2_DOUBLE (FindAccumulatorType) */
  int32_t value_type;
} B2ReduceResult;
B2_API int b2_reduce(B2Context* ctx, const B2Array* values, B2ReduceResult* out, void* stream);

/* ---------------------------------------------------------------------------
 * unique / value_counts / dictionary_encode over one fixed-width numeric or utf8 / binary column.
 * Replaces UniqueAction / ValueCountsAction / DictEncodeAction + RegularHashKernel
 * (compute/kernels/vector_hash.cc:65-235,236-470; registration :782-830;
 * DictionaryEncodeOptions compute/api_vector.h:66-82).
 *   out_dictionary : the distinct values in first-occurrence order (required)
 *   out_indices    : int32 index of every row into the dictionary, or NULL if not wanted
 *   out_counts     : int64 occurrences of every dictionary entry, or NULL if not wanted
 *   null_encoding  : 0 = MASK  (null rows -> null index; no null in the dictionary)
 *                    1 = ENCODE (null is a dictionary entry; what unique / value_counts use)
 * unique = (ENCODE, NULL, &d, NULL); value_counts = (ENCODE, NULL, &d, &c);
 * dictionary_encode = (mode, &i, &d, NULL).
 * ------------------------------------------------------------------------- */
B2_API int b2_vector_hash(B2Context* ctx, const B2Array* values, int null_encoding,
                          B2Array* out_indices, B2Array* out_dictionary, B2Array* out_counts,
                          void* stream);

/* ---------------------------------------------------------------------------
 * Hash aggregates.  Replaces the HashAggregateKernel contract
 * {init,resize,consume,merge,finalize} (compute/kernel.h:720-769) for
 * GroupedSumImpl / GroupedCountImpl / GroupedCountAllImpl / GroupedMeanImpl /
 * GroupedMinMaxImpl (kernels/hash_aggregate_numeric.cc:44-295,330-,
 * kernels/hash_aggregate.cc:61-272).
 * ------------------------------------------------------------------------- */
typedef enum B2HashAggKind {
  B2_HASH_SUM = 0,
  B2_HASH_COUNT = 1,
  B2_HASH_COUNT_ALL = 2,
  B2_HASH_MEAN = 3,
  B2_HASH_MIN = 4,
  B2_HASH_MAX = 5,
  B2_HASH_PRODUCT = 6, /* GroupedProductImpl, hash_aggregate_numeric.cc:311-335 (integers wrap mod 2^64) */
  B2_HASH_ANY = 7,     /* GroupedAnyImpl / GroupedAllImpl over a B2_BOOL column, hash_aggregate.cc:1232-1397 */
  B2_HASH_ALL = 8,
  B2_HASH_COUNT_DISTINCT = 9 /* GroupedCountDistinctImpl, hash_aggregate.cc:1400-1478: distinct (value, group) pairs
                                through a Grouper, counted per group under CountOptions::mode; numeric and utf8 / binary values */
} B2HashAggKind;
typedef struct B2HashAggOptions {
  int32_t skip_nulls;  /* ScalarAggregateOptions (api_aggregate.h:48-50), default 1 */
  uint32_t min_count;  /* default 1 */
  int32_t count_mode;  /* CountOptions: 0 ONLY_VALID, 1 ONLY_NULL, 2 ALL (api_aggregate.h:64-78) */
  int32_t reserved;
} B2HashAggOptions;
typedef struct B2HashAgg B2HashAgg;
B2_API int b2_hashagg_create(B2Context* ctx, int kind, int32_t value_type,
                             const B2HashAggOptions* options, B2HashAgg** out);
B2_API void b2_hashagg_destroy(B2HashAgg* a);
B2_API int b2_hashagg_resize(B2HashAgg* a, int64_t num_groups, void* stream);
/* values may be NULL for count_all; ids: B2_UINT32 array of the same length */
B2_API int b2_hashagg_consume(B2HashAgg* a, const B2Array* values, const B2Array* ids,
                              void* stream);
/* state[mapping[i]] (+)= other.state[i]; mapping: B2_UINT32, length = other groups */
B2_API int b2_hashagg_merge(B2HashAgg* a, B2HashAgg* other, const B2Array* group_id_mapping,
                            void* stream);
B2_API int b2_hashagg_finalize(B2HashAgg* a, B2Array* out, void* stream);
B2_API int32_t b2_hashagg_out_type(const B2HashAgg* a);

/* Fused group-by for the Acero aggregate node (acero/groupby_aggregate_node.cc:210-253
 * Consume = grouper->Consume + kernel->consume per aggregate): one pass over
 * (key, value) rows updating an on-device table, no uint32 id column materialised.
 * Semantically identical to b2_grouper_consume followed by b2_hashagg_consume of a
 * sum and a count(ONLY_VALID) aggregator over the same value column. */
/* expected_groups: cardinality hint (like reserving a builder).  0 = unknown: the table grows batch by
 * batch and large batches are processed in 64M-row chunks.  > 0: the table is sized for it and a batch is
 * processed in one chunk (fastest: rows of a key meet in shared memory); if the true number of groups
 * exceeds the hint by more than the table slack + 64M inside one batch, consume fails with
 * B2_CAPACITY_ERROR (nothing is silently dropped). */
typedef struct B2GroupBySumCount B2GroupBySumCount;
B2_API int b2_groupby_sumcount_create(B2Context* ctx, int32_t key_type, int32_t value_type,
                                      int64_t expected_groups, B2GroupBySumCount** out);
B2_API void b2_groupby_sumcount_destroy(B2GroupBySumCount* g);
B2_API int b2_groupby_sumcount_consume(B2GroupBySumCount* g, const B2Array* keys,
                                       const B2Array* values, void* stream);
/* Adds partial states into the table: keys / sums (the accumulator type b2_groupby_sumcount_finalize returns) /
 * counts (int64) of ANOTHER group-by over the same key and value types -- a peer GPU's groups after the exchange, or
 * another thread's.  The fused twin of HashAggregateKernel::merge (compute/kernel.h:720-725) as GroupByNode::Merge uses
 * it (acero/groupby_aggregate_node.cc:255-298).  A partial with count 0 only asserts the group exists. */
B2_API int b2_groupby_sumcount_merge(B2GroupBySumCount* g, const B2Array* keys, const B2Array* sums,
                                     const B2Array* counts, void* stream);
/* how many consume() chunks ran on each internal path (diagnostics for tests / bench):
 *   dense   : direct-addressed packed state in L2, one reduction per row (dense key range, narrow verified value window)
 *   compact : 8-byte tuples + bulk-async partition passes (key range + value window fit 63 bits)
 *   general : 17-byte tuples, any key / value
 *   atomic  : small batches, one global-table update per row */
B2_API int b2_groupby_sumcount_path_counts(const B2GroupBySumCount* g, int64_t* dense, int64_t* compact,
                                           int64_t* general, int64_t* atomic);
/* out_keys / out_sums / out_counts: num_groups long, group order unspecified */
B2_API int b2_groupby_sumcount_finalize(B2GroupBySumCount* g, B2Array* out_keys,
                                        B2Array* out_sums, B2Array* out_counts, void* stream);

/* ---------------------------------------------------------------------------
 * Multi-GPU exchange helpers (no reference counterpart: the reference is single-process;
 * its per-thread analogue is GroupByNode::Merge, acero/groupby_aggregate_node.cc:255-298).
 * out_ids: B2_UINT32, one destination id per row.
 *   hash : id = hash64(key) % n_parts, null keys -> 0          (hash-aggregate shuffle)
 *   range: id = #splitters <= value in SortIndices' total order; nulls -> n_splitters + 1
 *          (SortIndices shuffle; order as in b2_sort_indices)
 * ------------------------------------------------------------------------- */
B2_API int b2_hash_partition(B2Context* ctx, const B2Array* keys, int n_parts, B2Array* out_ids,
                             void* stream);
B2_API int b2_range_partition(B2Context* ctx, const B2Array* values, const B2Array* splitters,
                              int order, B2Array* out_ids, void* stream);
/* Sender side of the distributed SortIndices in one call: a STABLE split of (value, row number) pairs by range id
 * (bin b = #splitters <= value in SortIndices' order, b = 0 .. n_splitters; rows with a null value form the last bin).
 *   out_values : values regrouped bin by bin (row order kept inside a bin), no validity
 *   out_rows   : B2_UINT32 row_base + original row, regrouped the same way (the payload of b2_sort_payload at the owner)
 *   out_counts : HOST array of n_splitters + 2 int64 = rows per bin
 * count -> scan -> scatter: two streaming passes instead of ids + sort_indices(ids) + two takes + an offset add. */
B2_API int b2_range_split(B2Context* ctx, const B2Array* values, const B2Array* splitters, int order,
                          uint64_t row_base, B2Array* out_values, B2Array* out_rows, int64_t* out_counts,
                          void* stream);
/* out_counts[b] (HOST array of n_bins int64) = rows whose id == b: the send counts of the exchange.
 * ids: B2_UINT32 without nulls, every id < n_bins (else B2_INDEX_ERROR); n_bins <= 8192. */
B2_API int b2_bincount(B2Context* ctx, const B2Array* ids, int n_bins, int64_t* out_counts, void* stream);

/* The exchange itself: one process per GPU, NCCL over NVLink / NVSwitch (resolved with dlopen at the
 * first call; libarrow_b200.so does not link NCCL).  Rank 0 creates the 128-byte id, the host
 * application distributes it (MPI, a torch.distributed store, a file) and every rank calls
 * b2_comm_init with the same id.  All calls are stream-ordered on `stream` like every other entry.
 *   all_gather    : recv[r * bytes_per_rank ..] = rank r's `send` (the P x P count matrix)
 *   all_reduce_i64: element-wise sum / max / min of `count` int64 values
 *   all_to_all_v  : rank p receives send[send_offsets[p] .. + send_bytes[p]) of every rank q at
 *                   recv[recv_offsets[q] ..]; the P-1 sends and receives are one NCCL group
 *                   (host arrays of `world` entries, in bytes; recv_bytes must match the peers' send_bytes) */
#define B2_COMM_ID_BYTES 128
typedef struct B2Comm B2Comm;
typedef enum B2CommOp { B2_COMM_SUM = 0, B2_COMM_MAX = 1, B2_COMM_MIN = 2 } B2CommOp;
B2_API int b2_comm_unique_id(uint8_t* out_id /* [B2_COMM_ID_BYTES] */);
B2_API int b2_comm_init(B2Context* ctx, int rank, int world, const uint8_t* id, B2Comm** out);
B2_API void b2_comm_destroy(B2Comm* comm);
B2_API int b2_comm_rank(const B2Comm* comm);
B2_API int b2_comm_world(const B2Comm* comm);
B2_API int b2_comm_nccl_version(int* out);
/* all_to_all_v calls between group_start and group_end (one per column) are issued as ONE NCCL launch */
B2_API int b2_comm_group_start(B2Comm* comm);
B2_API int b2_comm_group_end(B2Comm* comm);
B2_API int b2_comm_all_gather(B2Comm* comm, const void* send, void* recv, int64_t bytes_per_rank, void* stream);
B2_API int b2_comm_all_reduce_i64(B2Comm* comm, const void* send, void* recv, int64_t count, int op, void* stream);
B2_API int b2_comm_all_to_all_v(B2Comm* comm, const void* send, const int64_t* send_offsets,
                                const int64_t* send_bytes, void* recv, const int64_t* recv_offsets,
                                const int64_t* recv_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* ARROW_B200_H */

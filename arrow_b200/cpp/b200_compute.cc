// b200_compute.cc -- kernel trampolines and function registration (see b200_compute.h).
//
// Every trampoline has the reference's kernel entry signature
//   Status exec(KernelContext*, const ExecSpan&, ExecResult*)          compute/kernel.h:556
// and registers with null_handling = COMPUTED_NO_PREALLOCATE and
// mem_allocation = NO_PREALLOCATE, because the stock executor cannot see device bitmaps
// (ArraySpan::SetBuffer stores Buffer::data() == nullptr for device buffers,
// array/data.h:578-582, and SetSlice then resets null_count, :680-690): validity is
// computed on device and null_count is always set explicitly.  Device addresses are read
// through BufferSpan::owner -> Buffer::address().
#include "b200_compute.h"

#include <cmath>
#include <cstring>

#include <arrow/compute/cast.h>
#include <arrow/compute/registry.h>
#include <arrow/util/checked_cast.h>

#include <map>
#include <mutex>

namespace arrow_b200 {

namespace cp = arrow::compute;
using arrow::ArrayData;
using arrow::ArraySpan;
using arrow::DataType;
using arrow::Datum;
using arrow::Result;
using arrow::Status;
using arrow::Type;
using arrow::TypeHolder;
using arrow::internal::checked_cast;

// ------------------------------------------------------------------------------------------
// type mapping and (de)marshalling
// ------------------------------------------------------------------------------------------
static Result<int> B2TypeId(const DataType& t) {
  switch (t.id()) {
    case Type::BOOL: return B2_BOOL;
    case Type::UINT8: return B2_UINT8;
    case Type::INT8: return B2_INT8;
    case Type::UINT16: return B2_UINT16;
    case Type::INT16: return B2_INT16;
    case Type::UINT32: return B2_UINT32;
    case Type::INT32: case Type::DATE32: case Type::TIME32: return B2_INT32;
    case Type::UINT64: return B2_UINT64;
    case Type::INT64: case Type::DATE64: case Type::TIME64: case Type::TIMESTAMP: case Type::DURATION: return B2_INT64;
    case Type::FLOAT: return B2_FLOAT;
    case Type::DOUBLE: return B2_DOUBLE;
    case Type::STRING: return B2_STRING;
    case Type::BINARY: return B2_BINARY;
    case Type::LARGE_STRING: return B2_LARGE_STRING;
    case Type::LARGE_BINARY: return B2_LARGE_BINARY;
    case Type::FIXED_SIZE_BINARY: return B2_FIXED_SIZE_BINARY;
    case Type::DICTIONARY: return B2TypeId(*checked_cast<const arrow::DictionaryType&>(t).index_type());
    default: return Status::NotImplemented("arrow_b200: type ", t.ToString(), " is not supported on device");
  }
}

static const void* Addr(const arrow::BufferSpan& b) {
  return b.owner && *b.owner ? reinterpret_cast<const void*>((*b.owner)->address()) : nullptr;
}
static const void* Addr(const std::shared_ptr<arrow::Buffer>& b) {
  return b ? reinterpret_cast<const void*>(b->address()) : nullptr;
}

Status SpanToB2(const ArraySpan& span, B2Array* out) {
  ARROW_ASSIGN_OR_RAISE(int tid, B2TypeId(*span.type));
  out->validity = Addr(span.buffers[0]);
  out->data = Addr(span.buffers[1]);
  out->data2 = Addr(span.buffers[2]);
  out->length = span.length;
  out->offset = span.offset;
  // never trust span.null_count for device data (SetSlice resets it): unknown unless no bitmap
  out->null_count = out->validity ? -1 : 0;
  out->type = tid;
  out->byte_width = span.type->id() == Type::FIXED_SIZE_BINARY ? span.type->byte_width() : 0;
  return Status::OK();
}

Status DataToB2(const ArrayData& data, B2Array* out) {
  ARROW_ASSIGN_OR_RAISE(int tid, B2TypeId(*data.type));
  out->validity = data.buffers.size() > 0 ? Addr(data.buffers[0]) : nullptr;
  out->data = data.buffers.size() > 1 ? Addr(data.buffers[1]) : nullptr;
  out->data2 = data.buffers.size() > 2 ? Addr(data.buffers[2]) : nullptr;
  out->length = data.length;
  out->offset = data.offset;
  out->null_count = out->validity ? data.null_count.load() : 0;
  out->type = tid;
  out->byte_width = data.type->id() == Type::FIXED_SIZE_BINARY ? data.type->byte_width() : 0;
  return Status::OK();
}

static int64_t DataBytes(const B2Array& o) {
  switch (o.type) {
    case B2_BOOL: return (o.length + 7) / 8;
    case B2_STRING: case B2_BINARY: return 4 * (o.length + 1);
    case B2_LARGE_STRING: case B2_LARGE_BINARY: return 8 * (o.length + 1);
    case B2_FIXED_SIZE_BINARY: return o.length * o.byte_width;
    case B2_UINT8: case B2_INT8: return o.length;
    case B2_UINT16: case B2_INT16: return 2 * o.length;
    case B2_UINT32: case B2_INT32: case B2_FLOAT: return 4 * o.length;
    default: return 8 * o.length;
  }
}

std::shared_ptr<ArrayData> AdoptOutput(Runtime* rt, const B2Array& o, std::shared_ptr<DataType> type,
                                       std::shared_ptr<ArrayData> dictionary) {
  auto out = std::make_shared<ArrayData>(std::move(type), o.length, o.null_count, o.offset);
  out->buffers.push_back(rt->mm()->Adopt(o.validity, (o.length + 7) / 8));
  out->buffers.push_back(rt->mm()->Adopt(o.data, DataBytes(o)));
  const bool binary = o.type == B2_STRING || o.type == B2_BINARY || o.type == B2_LARGE_STRING || o.type == B2_LARGE_BINARY;
  if (binary) {
    int64_t nbytes = 0;
    b2_binary_data_size(rt->context(), &o, &nbytes, nullptr);  // outputs start at offset 0: size = last offset
    out->buffers.push_back(rt->mm()->Adopt(o.data2, nbytes));
  }
  out->dictionary = std::move(dictionary);
  return out;
}

static void MoveInto(std::shared_ptr<ArrayData> produced, cp::ExecResult* out) {
  // keep the ArrayData object the executor handed us (it already carries the output type)
  ArrayData* dst = out->array_data().get();
  dst->length = produced->length;
  dst->null_count = produced->null_count.load();
  dst->offset = produced->offset;
  dst->buffers = std::move(produced->buffers);
  dst->child_data = std::move(produced->child_data);
  dst->dictionary = std::move(produced->dictionary);
}

static bool AnyOnDevice(const std::vector<Datum>& args) {
  for (const auto& a : args) {
    if (a.is_array() && IsOnDevice(*a.array())) return true;
    if (a.is_chunked_array())
      for (const auto& c : a.chunked_array()->chunks())
        if (IsOnDevice(*c->data())) return true;
    if (a.kind() == Datum::RECORD_BATCH)
      for (const auto& c : a.record_batch()->column_data())
        if (IsOnDevice(*c)) return true;
    if (a.kind() == Datum::TABLE)
      for (const auto& col : a.table()->columns())
        for (const auto& c : col->chunks())
          if (IsOnDevice(*c->data())) return true;
  }
  return false;
}

// ------------------------------------------------------------------------------------------
// runtime singleton
// ------------------------------------------------------------------------------------------
Result<Runtime*> Runtime::Get(int device) {
  static std::mutex mu;
  static std::map<int, std::unique_ptr<Runtime>> instances;
  std::lock_guard<std::mutex> lk(mu);
  auto it = instances.find(device);
  if (it != instances.end()) return it->second.get();
  auto rt = std::unique_ptr<Runtime>(new Runtime());
  ARROW_ASSIGN_OR_RAISE(rt->device_, B200Device::Make(device));
  rt->mm_ = rt->device_->default_memory_manager();
  rt->registry_ = cp::FunctionRegistry::Make(cp::GetFunctionRegistry());
  ARROW_RETURN_NOT_OK(RegisterFunctions(rt->registry_.get(), rt.get()));
  Runtime* raw = rt.get();
  instances[device] = std::move(rt);
  return raw;
}

// per-kernel immutable data: which runtime, which op
struct KernelData : public cp::KernelState {
  KernelData(Runtime* r, int o) : rt(r), op(o) {}
  Runtime* rt;
  int op;
};
static const KernelData& DataOf(cp::KernelContext* ctx) { return checked_cast<const KernelData&>(*ctx->kernel()->data); }

template <typename Options>
struct OptionsState : public cp::KernelState {
  explicit OptionsState(Options o) : options(std::move(o)) {}
  Options options;
  static Result<std::unique_ptr<cp::KernelState>> Init(cp::KernelContext*, const cp::KernelInitArgs& args) {
    if (auto o = static_cast<const Options*>(args.options)) return std::make_unique<OptionsState>(*o);
    return std::make_unique<OptionsState>(Options::Defaults());
  }
  static const Options& Get(cp::KernelContext* ctx) { return checked_cast<const OptionsState&>(*ctx->state()).options; }
};

// ------------------------------------------------------------------------------------------
// a function that forwards host arguments to the parent registry's stock function
// ------------------------------------------------------------------------------------------
template <typename Base>
class Forwarding : public Base {
 public:
  using Base::Base;
  Result<Datum> Execute(const std::vector<Datum>& args, const cp::FunctionOptions* options,
                        cp::ExecContext* ctx) const override {
    if (!AnyOnDevice(args)) {
      ARROW_ASSIGN_OR_RAISE(auto parent, cp::GetFunctionRegistry()->GetFunction(this->name()));
      cp::ExecContext host_ctx(ctx ? ctx->memory_pool() : arrow::default_memory_pool(), ctx ? ctx->executor() : nullptr,
                               cp::GetFunctionRegistry());
      return parent->Execute(args, options, &host_ctx);
    }
    return Base::Execute(args, options, ctx);
  }
};

static const cp::FunctionDoc kDoc{"B200 device kernel", "Runs on the GPU through libarrow_b200 (see include/arrow_b200.h).", {}};
static cp::FunctionDoc DocFor(std::vector<std::string> arg_names, const char* options_class = "", bool required = false) {
  cp::FunctionDoc d = kDoc;
  d.arg_names = std::move(arg_names);
  d.options_class = options_class;
  d.options_required = required;
  return d;
}

static const std::vector<std::shared_ptr<DataType>>& NumericTypes() {
  static std::vector<std::shared_ptr<DataType>> t = {arrow::int8(),  arrow::uint8(),  arrow::int16(),   arrow::uint16(),
                                                     arrow::int32(), arrow::uint32(), arrow::int64(),   arrow::uint64(),
                                                     arrow::float32(), arrow::float64()};
  return t;
}

// CommonNumeric (compute/kernels/codegen_internal.cc:166-218)
static std::shared_ptr<DataType> CommonNumeric(const std::vector<TypeHolder>& types) {
  for (const auto& t : types)
    if (!arrow::is_floating(t.id()) && !arrow::is_integer(t.id())) return nullptr;
  for (const auto& t : types)
    if (t.id() == Type::HALF_FLOAT) return nullptr;
  for (const auto& t : types)
    if (t.id() == Type::DOUBLE) return arrow::float64();
  for (const auto& t : types)
    if (t.id() == Type::FLOAT) return arrow::float32();
  int max_s = 0, max_u = 0;
  for (const auto& t : types) {
    int& m = arrow::is_signed_integer(t.id()) ? max_s : max_u;
    m = std::max(arrow::bit_width(t.id()), m);
  }
  if (max_s == 0) {
    if (max_u >= 64) return arrow::uint64();
    if (max_u == 32) return arrow::uint32();
    if (max_u == 16) return arrow::uint16();
    return arrow::uint8();
  }
  if (max_s <= max_u) {
    int v = max_u + 1, p = 1;
    while (p < v) p <<= 1;
    max_s = p;
  }
  if (max_s >= 64) return arrow::int64();
  if (max_s == 32) return arrow::int32();
  if (max_s == 16) return arrow::int16();
  return arrow::int8();
}

// ------------------------------------------------------------------------------------------
// arithmetic + compare (ScalarBinary applicators, codegen_internal.h:813-976)
// ------------------------------------------------------------------------------------------
struct BinaryOperand {
  B2Array array;
  B2Scalar scalar;
  B2Value value;
};

static Status MakeOperand(const cp::ExecValue& v, BinaryOperand* o) {
  if (v.is_array()) {
    ARROW_RETURN_NOT_OK(SpanToB2(v.array, &o->array));
    o->value.array = &o->array;
    o->value.scalar = nullptr;
  } else {
    ARROW_ASSIGN_OR_RAISE(int tid, B2TypeId(*v.scalar->type));
    o->scalar.type = tid;
    o->scalar.is_valid = v.scalar->is_valid;
    o->scalar.bits = 0;
    if (v.scalar->is_valid) {
      auto view = checked_cast<const arrow::internal::PrimitiveScalarBase&>(*v.scalar).view();
      memcpy(&o->scalar.bits, view.data(), std::min<size_t>(8, view.size()));
    }
    o->value.array = nullptr;
    o->value.scalar = &o->scalar;
  }
  return Status::OK();
}

static Status ArithExec(cp::KernelContext* ctx, const cp::ExecSpan& batch, cp::ExecResult* out) {
  const KernelData& kd = DataOf(ctx);
  BinaryOperand l, r;
  ARROW_RETURN_NOT_OK(MakeOperand(batch[0], &l));
  ARROW_RETURN_NOT_OK(MakeOperand(batch[1], &r));
  B2Array o;
  B200_RETURN_NOT_OK(b2_binary_arith(kd.rt->context(), kd.op, &l.value, &r.value, &o, nullptr));
  MoveInto(AdoptOutput(kd.rt, o, out->type()->GetSharedPtr()), out);
  return Status::OK();
}

static Status CompareExec(cp::KernelContext* ctx, const cp::ExecSpan& batch, cp::ExecResult* out) {
  const KernelData& kd = DataOf(ctx);
  BinaryOperand l, r;
  ARROW_RETURN_NOT_OK(MakeOperand(batch[0], &l));
  ARROW_RETURN_NOT_OK(MakeOperand(batch[1], &r));
  B2Array o;
  B200_RETURN_NOT_OK(b2_compare(kd.rt->context(), kd.op, &l.value, &r.value, &o, nullptr));
  MoveInto(AdoptOutput(kd.rt, o, arrow::boolean()), out);
  return Status::OK();
}

// ArithmeticFunction / CompareFunction dispatch: exact, else promote to CommonNumeric
// (kernels/scalar_arithmetic.cc:734-781, kernels/scalar_compare.cc:340-366)
class NumericBinaryFunction : public Forwarding<cp::ScalarFunction> {
 public:
  using Forwarding<cp::ScalarFunction>::Forwarding;
  Result<const cp::Kernel*> DispatchBest(std::vector<TypeHolder>* values) const override {
    auto exact = DispatchExact(*values);
    if (exact.ok()) return exact;
    if (auto common = CommonNumeric(*values)) {
      for (auto& v : *values) v = common;
      return DispatchExact(*values);
    }
    return exact;
  }
};

static Status AddBinaryFunction(cp::FunctionRegistry* reg, Runtime* rt, const std::string& name, int op, bool compare) {
  auto fn = std::make_shared<NumericBinaryFunction>(name, cp::Arity::Binary(), DocFor({"x", "y"}));
  for (const auto& ty : NumericTypes()) {
    cp::ScalarKernel k({cp::InputType(ty), cp::InputType(ty)}, compare ? cp::OutputType(arrow::boolean()) : cp::OutputType(ty),
                       compare ? CompareExec : ArithExec);
    k.null_handling = cp::NullHandling::COMPUTED_NO_PREALLOCATE;
    k.mem_allocation = cp::MemAllocation::NO_PREALLOCATE;
    k.can_write_into_slices = false;
    k.data = std::make_shared<KernelData>(rt, op);
    ARROW_RETURN_NOT_OK(fn->AddKernel(std::move(k)));
  }
  return reg->AddFunction(std::move(fn), /*allow_overwrite=*/true);
}

// ------------------------------------------------------------------------------------------
// boolean logic, validity predicates, if_else (kernels/scalar_boolean.cc, scalar_validity.cc, scalar_if_else.cc):
// the kernels an Expression (filter predicate, projection) is made of besides arithmetic and compare
// ------------------------------------------------------------------------------------------
static Status BooleanExec(cp::KernelContext* ctx, const cp::ExecSpan& batch, cp::ExecResult* out) {
  const KernelData& kd = DataOf(ctx);
  BinaryOperand l, r;
  ARROW_RETURN_NOT_OK(MakeOperand(batch[0], &l));
  if (batch.num_values() > 1) ARROW_RETURN_NOT_OK(MakeOperand(batch[1], &r));
  B2Array o;
  B200_RETURN_NOT_OK(b2_boolean(kd.rt->context(), kd.op, &l.value, batch.num_values() > 1 ? &r.value : nullptr, &o, nullptr));
  MoveInto(AdoptOutput(kd.rt, o, arrow::boolean()), out);
  return Status::OK();
}

static Status ValidityExec(cp::KernelContext* ctx, const cp::ExecSpan& batch, cp::ExecResult* out) {
  const KernelData& kd = DataOf(ctx);
  if (!batch[0].is_array()) return Status::NotImplemented("arrow_b200: validity predicates need an array argument");
  B2Array in, o;
  ARROW_RETURN_NOT_OK(SpanToB2(batch[0].array, &in));
  const int nan_is_null = (kd.op == B2_IS_NULL && ctx->state()) ? OptionsState<cp::NullOptions>::Get(ctx).nan_is_null : 0;
  B200_RETURN_NOT_OK(b2_validity(kd.rt->context(), kd.op, &in, nan_is_null, &o, nullptr));
  MoveInto(AdoptOutput(kd.rt, o, arrow::boolean()), out);
  return Status::OK();
}

static Status IfElseExec(cp::KernelContext* ctx, const cp::ExecSpan& batch, cp::ExecResult* out) {
  const KernelData& kd = DataOf(ctx);
  BinaryOperand c, l, r;
  ARROW_RETURN_NOT_OK(MakeOperand(batch[0], &c));
  ARROW_RETURN_NOT_OK(MakeOperand(batch[1], &l));
  ARROW_RETURN_NOT_OK(MakeOperand(batch[2], &r));
  B2Array o;
  B200_RETURN_NOT_OK(b2_if_else(kd.rt->context(), &c.value, &l.value, &r.value, &o, nullptr));
  MoveInto(AdoptOutput(kd.rt, o, out->type()->GetSharedPtr()), out);
  return Status::OK();
}

// IfElseFunction::DispatchBest (kernels/scalar_if_else.cc:1227-1266): left / right are cast to their common numeric type
class IfElseFunction : public Forwarding<cp::ScalarFunction> {
 public:
  using Forwarding<cp::ScalarFunction>::Forwarding;
  Result<const cp::Kernel*> DispatchBest(std::vector<TypeHolder>* values) const override {
    auto exact = DispatchExact(*values);
    if (exact.ok() || values->size() != 3) return exact;
    if (auto common = CommonNumeric({(*values)[1], (*values)[2]})) {
      (*values)[1] = (*values)[2] = common;
      return DispatchExact(*values);
    }
    return exact;
  }
};

static cp::ScalarKernel DeviceScalarKernel(Runtime* rt, std::vector<cp::InputType> in, cp::OutputType out, cp::ArrayKernelExec exec,
                                           int op, cp::KernelInit init = nullptr) {
  cp::ScalarKernel k(std::move(in), std::move(out), exec, init);
  k.null_handling = cp::NullHandling::COMPUTED_NO_PREALLOCATE;
  k.mem_allocation = cp::MemAllocation::NO_PREALLOCATE;
  k.can_write_into_slices = false;
  k.data = std::make_shared<KernelData>(rt, op);
  return k;
}

static Status AddLogicFunctions(cp::FunctionRegistry* reg, Runtime* rt) {
  const std::pair<const char*, int> binary[] = {{"and", B2_BOOL_AND}, {"or", B2_BOOL_OR}, {"xor", B2_BOOL_XOR},
                                                {"and_not", B2_BOOL_AND_NOT}, {"and_kleene", B2_BOOL_AND_KLEENE},
                                                {"or_kleene", B2_BOOL_OR_KLEENE}, {"and_not_kleene", B2_BOOL_AND_NOT_KLEENE}};
  const auto b = cp::InputType(arrow::boolean());
  for (const auto& f : binary) {
    auto fn = std::make_shared<Forwarding<cp::ScalarFunction>>(f.first, cp::Arity::Binary(), DocFor({"x", "y"}));
    ARROW_RETURN_NOT_OK(fn->AddKernel(DeviceScalarKernel(rt, {b, b}, cp::OutputType(arrow::boolean()), BooleanExec, f.second)));
    ARROW_RETURN_NOT_OK(reg->AddFunction(std::move(fn), true));
  }
  {
    auto fn = std::make_shared<Forwarding<cp::ScalarFunction>>("invert", cp::Arity::Unary(), DocFor({"values"}));
    ARROW_RETURN_NOT_OK(fn->AddKernel(DeviceScalarKernel(rt, {b}, cp::OutputType(arrow::boolean()), BooleanExec, B2_BOOL_INVERT)));
    ARROW_RETURN_NOT_OK(reg->AddFunction(std::move(fn), true));
  }
  static const cp::NullOptions kNullDefaults = cp::NullOptions::Defaults();
  const std::pair<const char*, int> unary[] = {{"is_valid", B2_IS_VALID}, {"is_null", B2_IS_NULL},
                                               {"true_unless_null", B2_TRUE_UNLESS_NULL}, {"is_nan", B2_IS_NAN}};
  for (const auto& f : unary) {
    const bool with_options = f.second == B2_IS_NULL;
    auto fn = with_options ? std::make_shared<Forwarding<cp::ScalarFunction>>(f.first, cp::Arity::Unary(), DocFor({"values"}, "NullOptions"),
                                                                              &kNullDefaults)
                           : std::make_shared<Forwarding<cp::ScalarFunction>>(f.first, cp::Arity::Unary(), DocFor({"values"}));
    auto types = NumericTypes();
    if (f.second != B2_IS_NAN) types.push_back(arrow::boolean());
    for (const auto& ty : types) {
      if (f.second == B2_IS_NAN && !arrow::is_floating(ty->id())) continue;
      ARROW_RETURN_NOT_OK(fn->AddKernel(DeviceScalarKernel(rt, {cp::InputType(ty)}, cp::OutputType(arrow::boolean()), ValidityExec, f.second,
                                                           with_options ? OptionsState<cp::NullOptions>::Init : nullptr)));
    }
    ARROW_RETURN_NOT_OK(reg->AddFunction(std::move(fn), true));
  }
  auto fn = std::make_shared<IfElseFunction>("if_else", cp::Arity::Ternary(), DocFor({"cond", "left", "right"}));
  auto types = NumericTypes();
  types.push_back(arrow::boolean());
  for (const auto& ty : types)
    ARROW_RETURN_NOT_OK(fn->AddKernel(DeviceScalarKernel(rt, {b, cp::InputType(ty), cp::InputType(ty)}, cp::OutputType(ty), IfElseExec, 0)));
  return reg->AddFunction(std::move(fn), true);
}

// ------------------------------------------------------------------------------------------
// cast: a MetaFunction like the reference's CastMetaFunction (compute/cast.cc:78-127)
// ------------------------------------------------------------------------------------------
class CastFunction : public cp::MetaFunction {
 public:
  explicit CastFunction(Runtime* rt) : cp::MetaFunction("cast", cp::Arity::Unary(), DocFor({"input"}, "CastOptions", true)), rt_(rt) {}
  Result<Datum> ExecuteImpl(const std::vector<Datum>& args, const cp::FunctionOptions* options,
                            cp::ExecContext* ctx) const override {
    if (!AnyOnDevice(args)) {
      ARROW_ASSIGN_OR_RAISE(auto parent, cp::GetFunctionRegistry()->GetFunction("cast"));
      return parent->Execute(args, options, ctx);
    }
    auto opts = static_cast<const cp::CastOptions*>(options);
    if (!opts || !opts->to_type.type) return Status::Invalid("Cast requires that options.to_type has been set");
    if (!args[0].is_array()) return Status::NotImplemented("arrow_b200 cast: only Array inputs (chunks are cast one by one by the caller)");
    const ArrayData& in = *args[0].array();
    if (in.type->Equals(*opts->to_type.type)) return args[0];
    // Temporal / dictionary / other logical types share integer storage with the numeric types but not
    // their cast semantics (unit rescaling, kernels/scalar_cast_temporal.cc): never relabel raw storage.
    auto genuinely_numeric = [](const DataType& t) {
      return (arrow::is_integer(t.id()) || t.id() == Type::FLOAT || t.id() == Type::DOUBLE);
    };
    if (!genuinely_numeric(*in.type) || !genuinely_numeric(*opts->to_type.type))
      return Status::NotImplemented("Unsupported cast from ", in.type->ToString(), " to ", opts->to_type.type->ToString(),
                                    " using function cast_", opts->to_type.type->name());
    B2Array bin, bout;
    ARROW_RETURN_NOT_OK(DataToB2(in, &bin));
    ARROW_ASSIGN_OR_RAISE(int to, B2TypeId(*opts->to_type.type));
    B2CastOptions co{to, opts->allow_int_overflow, opts->allow_float_truncate, 0};
    int st = b2_cast_numeric(rt_->context(), &bin, &co, &bout, nullptr);
    if (st == B2_NOT_IMPLEMENTED)
      return Status::NotImplemented("Unsupported cast from ", in.type->ToString(), " to ", opts->to_type.type->ToString(),
                                    " using function cast_", opts->to_type.type->name());
    B200_RETURN_NOT_OK(st);
    return Datum(AdoptOutput(rt_, bout, opts->to_type.GetSharedPtr()));
  }

 private:
  Runtime* rt_;
};

// sort_indices on a record batch / single-chunk table of device columns: the multi-key sort (kernels/vector_sort.cc:850-1027
// SortIndicesMetaFunction -> :386-600 MultipleKeyRecordBatchSorter).  Arrays and chunked arrays keep the stock meta
// function, which reaches array_sort_indices above through this registry.
class SortIndicesFunction : public cp::MetaFunction {
 public:
  explicit SortIndicesFunction(Runtime* rt)
      : cp::MetaFunction("sort_indices", cp::Arity::Unary(), DocFor({"input"}, "SortOptions"), &kDefaults), rt_(rt) {}
  Result<Datum> ExecuteImpl(const std::vector<Datum>& args, const cp::FunctionOptions* options, cp::ExecContext* ctx) const override {
    const bool tabular = args[0].kind() == Datum::RECORD_BATCH || args[0].kind() == Datum::TABLE;
    if (!tabular || !AnyOnDevice(args)) {
      ARROW_ASSIGN_OR_RAISE(auto parent, cp::GetFunctionRegistry()->GetFunction("sort_indices"));
      return parent->Execute(args, options, ctx);
    }
    const auto& so = options ? *static_cast<const cp::SortOptions*>(options) : kDefaults;
    if (so.sort_keys.empty()) return Status::Invalid("Must specify one or more sort keys");
    std::shared_ptr<arrow::Schema> schema = args[0].schema();
    std::vector<B2Array> keys(so.sort_keys.size());
    std::vector<int32_t> orders(so.sort_keys.size());
    for (size_t k = 0; k < so.sort_keys.size(); ++k) {
      ARROW_ASSIGN_OR_RAISE(auto match, so.sort_keys[k].target.FindOne(*schema));
      if (match.indices().size() != 1) return Status::NotImplemented("arrow_b200 sort_indices: nested sort keys");
      const int col = match.indices()[0];
      std::shared_ptr<ArrayData> data;
      if (args[0].kind() == Datum::RECORD_BATCH) {
        data = args[0].record_batch()->column_data(col);
      } else {
        const auto& chunked = args[0].table()->column(col);
        if (chunked->num_chunks() != 1) return Status::NotImplemented("arrow_b200 sort_indices: device tables must hold one chunk per column");
        data = chunked->chunk(0)->data();
      }
      const Type::type id = data->type->id();
      if (!arrow::is_integer(id) && !arrow::is_floating(id) && !arrow::is_base_binary_like(id))
        return Status::NotImplemented("arrow_b200 sort_indices: sort key of type ", data->type->ToString());
      ARROW_RETURN_NOT_OK(DataToB2(*data, &keys[k]));
      orders[k] = so.sort_keys[k].order == cp::SortOrder::Descending ? 1 : 0;
    }
    B2Array o;
    B200_RETURN_NOT_OK(b2_sort_indices_multi(rt_->context(), keys.data(), static_cast<int>(keys.size()), orders.data(),
                                             so.null_placement == cp::NullPlacement::AtEnd ? 1 : 0, &o, nullptr));
    return Datum(AdoptOutput(rt_, o, arrow::uint64()));
  }

 private:
  static const cp::SortOptions kDefaults;
  Runtime* rt_;
};
const cp::SortOptions SortIndicesFunction::kDefaults = cp::SortOptions::Defaults();

// select_k_unstable on a device array (SelectKUnstableMetaFunction, kernels/vector_select_k.cc:615-690): b2_select_k --
// a sampled threshold, one compare pass, a sort of the few candidates; anything else goes to the stock function
class SelectKFunction : public cp::MetaFunction {
 public:
  explicit SelectKFunction(Runtime* rt)
      : cp::MetaFunction("select_k_unstable", cp::Arity::Unary(), DocFor({"input"}, "SelectKOptions"), &kDefaults), rt_(rt) {}
  Result<Datum> ExecuteImpl(const std::vector<Datum>& args, const cp::FunctionOptions* options, cp::ExecContext* ctx) const override {
    if (!args[0].is_array() || !AnyOnDevice(args)) {
      ARROW_ASSIGN_OR_RAISE(auto parent, cp::GetFunctionRegistry()->GetFunction("select_k_unstable"));
      return parent->Execute(args, options, ctx);
    }
    const auto& so = options ? *static_cast<const cp::SelectKOptions*>(options) : kDefaults;
    if (so.k < 0) return Status::Invalid("select_k_unstable requires a nonnegative `k`, got ", so.k);
    if (so.sort_keys.size() != 1) return Status::Invalid("select_k_unstable on an array takes exactly one sort key");
    const auto& type = *args[0].type();
    if (!arrow::is_integer(type.id()) && !arrow::is_floating(type.id()) && !arrow::is_base_binary_like(type.id()))
      return Status::NotImplemented("arrow_b200 select_k_unstable: values of type ", type.ToString());
    B2Array v, o;
    ARROW_RETURN_NOT_OK(DataToB2(*args[0].array(), &v));
    B200_RETURN_NOT_OK(b2_select_k(rt_->context(), &v, so.k, so.sort_keys[0].order == cp::SortOrder::Descending ? 1 : 0, /*AtEnd=*/1, &o, nullptr));
    return Datum(AdoptOutput(rt_, o, arrow::uint64()));
  }

 private:
  static const cp::SelectKOptions kDefaults;
  Runtime* rt_;
};
const cp::SelectKOptions SelectKFunction::kDefaults = cp::SelectKOptions::Defaults();

// ------------------------------------------------------------------------------------------
// selection + sort vector kernels
// ------------------------------------------------------------------------------------------
static Result<TypeHolder> FirstType(cp::KernelContext*, const std::vector<TypeHolder>& types) { return types.front(); }

static std::shared_ptr<ArrayData> DictionaryOf(const ArraySpan& span) {
  return span.type->id() == Type::DICTIONARY ? span.dictionary().ToArrayData() : nullptr;
}

static Status FilterExec(cp::KernelContext* ctx, const cp::ExecSpan& batch, cp::ExecResult* out) {
  const KernelData& kd = DataOf(ctx);
  const auto& opts = OptionsState<cp::FilterOptions>::Get(ctx);
  // the stock VectorExecutor raises this for mismatched array arguments (exec.cc CheckAllArrayOrScalar/InferBatchLength)
  if (batch[0].array.length != batch[1].array.length)
    return Status::Invalid("Arguments for execution of vector kernel function 'array_filter' must all be the same length");
  B2Array v, m, o;
  ARROW_RETURN_NOT_OK(SpanToB2(batch[0].array, &v));
  ARROW_RETURN_NOT_OK(SpanToB2(batch[1].array, &m));
  B200_RETURN_NOT_OK(b2_filter(kd.rt->context(), &v, &m, opts.null_selection_behavior == cp::FilterOptions::EMIT_NULL ? 1 : 0, &o, nullptr));
  MoveInto(AdoptOutput(kd.rt, o, batch[0].type()->GetSharedPtr(), DictionaryOf(batch[0].array)), out);
  return Status::OK();
}

static Status TakeExec(cp::KernelContext* ctx, const cp::ExecSpan& batch, cp::ExecResult* out) {
  const KernelData& kd = DataOf(ctx);
  const auto& opts = OptionsState<cp::TakeOptions>::Get(ctx);
  B2Array v, i, o;
  ARROW_RETURN_NOT_OK(SpanToB2(batch[0].array, &v));
  ARROW_RETURN_NOT_OK(SpanToB2(batch[1].array, &i));
  B200_RETURN_NOT_OK(b2_take(kd.rt->context(), &v, &i, opts.boundscheck, &o, nullptr));
  MoveInto(AdoptOutput(kd.rt, o, batch[0].type()->GetSharedPtr(), DictionaryOf(batch[0].array)), out);
  return Status::OK();
}

static Status SortExec(cp::KernelContext* ctx, const cp::ExecSpan& batch, cp::ExecResult* out) {
  const KernelData& kd = DataOf(ctx);
  const auto& opts = OptionsState<cp::ArraySortOptions>::Get(ctx);
  B2Array v, o;
  ARROW_RETURN_NOT_OK(SpanToB2(batch[0].array, &v));
  B200_RETURN_NOT_OK(b2_sort_indices(kd.rt->context(), &v, opts.order == cp::SortOrder::Descending ? 1 : 0,
                                     opts.null_placement == cp::NullPlacement::AtEnd ? 1 : 0, &o, nullptr));
  MoveInto(AdoptOutput(kd.rt, o, arrow::uint64()), out);
  return Status::OK();
}

static cp::VectorKernel MakeVectorKernel(Runtime* rt, std::vector<cp::InputType> in, cp::OutputType out, cp::ArrayKernelExec exec,
                                         cp::KernelInit init) {
  cp::VectorKernel k(std::move(in), std::move(out), exec, std::move(init));
  k.null_handling = cp::NullHandling::COMPUTED_NO_PREALLOCATE;
  k.mem_allocation = cp::MemAllocation::NO_PREALLOCATE;
  k.can_write_into_slices = false;
  k.can_execute_chunkwise = false;  // as array_take / array_sort_indices in the reference
  k.output_chunked = false;
  k.data = std::make_shared<KernelData>(rt, 0);
  return k;
}

static Status AddSelectionFunctions(cp::FunctionRegistry* reg, Runtime* rt) {
  static const cp::FilterOptions kFilterDefaults = cp::FilterOptions::Defaults();
  static const cp::TakeOptions kTakeDefaults = cp::TakeOptions::Defaults();
  static const cp::ArraySortOptions kSortDefaults = cp::ArraySortOptions::Defaults();
  auto filter = std::make_shared<Forwarding<cp::VectorFunction>>("array_filter", cp::Arity::Binary(),
                                                                 DocFor({"array", "selection_filter"}, "FilterOptions"), &kFilterDefaults);
  ARROW_RETURN_NOT_OK(filter->AddKernel(MakeVectorKernel(rt, {cp::InputType::Any(), cp::InputType(arrow::boolean())},
                                                         cp::OutputType(FirstType), FilterExec, OptionsState<cp::FilterOptions>::Init)));
  ARROW_RETURN_NOT_OK(reg->AddFunction(std::move(filter), true));

  auto take = std::make_shared<Forwarding<cp::VectorFunction>>("array_take", cp::Arity::Binary(),
                                                               DocFor({"array", "indices"}, "TakeOptions"), &kTakeDefaults);
  for (const auto& it : arrow::IntTypes()) {
    ARROW_RETURN_NOT_OK(take->AddKernel(MakeVectorKernel(rt, {cp::InputType::Any(), cp::InputType(it)}, cp::OutputType(FirstType),
                                                         TakeExec, OptionsState<cp::TakeOptions>::Init)));
  }
  ARROW_RETURN_NOT_OK(reg->AddFunction(std::move(take), true));

  auto sort = std::make_shared<Forwarding<cp::VectorFunction>>("array_sort_indices", cp::Arity::Unary(),
                                                               DocFor({"array"}, "ArraySortOptions"), &kSortDefaults);
  std::vector<std::shared_ptr<arrow::DataType>> sort_types = NumericTypes();
  for (const auto& ty : arrow::BaseBinaryTypes()) sort_types.push_back(ty);  // utf8, large_utf8, binary, large_binary
  for (const auto& ty : sort_types) {
    ARROW_RETURN_NOT_OK(sort->AddKernel(MakeVectorKernel(rt, {cp::InputType(ty)}, cp::OutputType(arrow::uint64()), SortExec,
                                                         OptionsState<cp::ArraySortOptions>::Init)));
  }
  return reg->AddFunction(std::move(sort), true);
}

// ------------------------------------------------------------------------------------------
// unique / value_counts / dictionary_encode (compute/kernels/vector_hash.cc:782-830)
// ------------------------------------------------------------------------------------------
static Status UniqueExec(cp::KernelContext* ctx, const cp::ExecSpan& batch, cp::ExecResult* out) {
  const KernelData& kd = DataOf(ctx);
  B2Array v, d;
  ARROW_RETURN_NOT_OK(SpanToB2(batch[0].array, &v));
  B200_RETURN_NOT_OK(b2_vector_hash(kd.rt->context(), &v, /*ENCODE*/ 1, nullptr, &d, nullptr, nullptr));
  MoveInto(AdoptOutput(kd.rt, d, batch[0].type()->GetSharedPtr()), out);
  return Status::OK();
}

static Status ValueCountsExec(cp::KernelContext* ctx, const cp::ExecSpan& batch, cp::ExecResult* out) {
  const KernelData& kd = DataOf(ctx);
  B2Array v, d, c;
  ARROW_RETURN_NOT_OK(SpanToB2(batch[0].array, &v));
  B200_RETURN_NOT_OK(b2_vector_hash(kd.rt->context(), &v, /*ENCODE*/ 1, nullptr, &d, &c, nullptr));
  // struct<values, counts> with no top-level validity (vector_hash.cc:634)
  auto produced = std::make_shared<ArrayData>(out->type()->GetSharedPtr(), d.length, 0);
  produced->buffers.push_back(nullptr);
  produced->child_data.push_back(AdoptOutput(kd.rt, d, batch[0].type()->GetSharedPtr()));
  produced->child_data.push_back(AdoptOutput(kd.rt, c, arrow::int64()));
  MoveInto(std::move(produced), out);
  return Status::OK();
}

static Status DictEncodeExec(cp::KernelContext* ctx, const cp::ExecSpan& batch, cp::ExecResult* out) {
  const KernelData& kd = DataOf(ctx);
  const auto& opts = OptionsState<cp::DictionaryEncodeOptions>::Get(ctx);
  B2Array v, i, d;
  ARROW_RETURN_NOT_OK(SpanToB2(batch[0].array, &v));
  const int mode = opts.null_encoding_behavior == cp::DictionaryEncodeOptions::ENCODE ? 1 : 0;
  B200_RETURN_NOT_OK(b2_vector_hash(kd.rt->context(), &v, mode, &i, &d, nullptr, nullptr));
  MoveInto(AdoptOutput(kd.rt, i, out->type()->GetSharedPtr(), AdoptOutput(kd.rt, d, batch[0].type()->GetSharedPtr())), out);
  return Status::OK();
}

static Result<TypeHolder> ValueCountsType(cp::KernelContext*, const std::vector<TypeHolder>& types) {
  return TypeHolder(arrow::struct_({arrow::field("values", types[0].GetSharedPtr()), arrow::field("counts", arrow::int64())}));
}
static Result<TypeHolder> DictEncodeType(cp::KernelContext*, const std::vector<TypeHolder>& types) {
  return TypeHolder(arrow::dictionary(arrow::int32(), types[0].GetSharedPtr()));
}

static Status AddHashFunctions(cp::FunctionRegistry* reg, Runtime* rt) {
  static const cp::DictionaryEncodeOptions kDictDefaults = cp::DictionaryEncodeOptions::Defaults();
  auto unique = std::make_shared<Forwarding<cp::VectorFunction>>("unique", cp::Arity::Unary(), DocFor({"array"}, ""), nullptr);
  auto counts = std::make_shared<Forwarding<cp::VectorFunction>>("value_counts", cp::Arity::Unary(), DocFor({"array"}, ""), nullptr);
  auto encode = std::make_shared<Forwarding<cp::VectorFunction>>("dictionary_encode", cp::Arity::Unary(),
                                                                 DocFor({"array"}, "DictionaryEncodeOptions"), &kDictDefaults);
  // numeric columns and (r2) utf8 / binary ones: the string grouper of csrc/grouper_wide.cu (vector_hash.cc:782-830 registers both)
  std::vector<std::shared_ptr<DataType>> hashable = NumericTypes();
  for (const auto& ty : {arrow::utf8(), arrow::large_utf8(), arrow::binary(), arrow::large_binary()}) hashable.push_back(ty);
  for (const auto& ty : hashable) {
    ARROW_RETURN_NOT_OK(unique->AddKernel(MakeVectorKernel(rt, {cp::InputType(ty)}, cp::OutputType(FirstType), UniqueExec, nullptr)));
    ARROW_RETURN_NOT_OK(counts->AddKernel(MakeVectorKernel(rt, {cp::InputType(ty)}, cp::OutputType(ValueCountsType), ValueCountsExec, nullptr)));
    ARROW_RETURN_NOT_OK(encode->AddKernel(MakeVectorKernel(rt, {cp::InputType(ty)}, cp::OutputType(DictEncodeType), DictEncodeExec,
                                                           OptionsState<cp::DictionaryEncodeOptions>::Init)));
  }
  ARROW_RETURN_NOT_OK(reg->AddFunction(std::move(unique), true));
  ARROW_RETURN_NOT_OK(reg->AddFunction(std::move(counts), true));
  return reg->AddFunction(std::move(encode), true);
}

// ------------------------------------------------------------------------------------------
// ungrouped sum / mean / min_max / count: the ScalarAggregateKernel contract
// {init, consume, merge, finalize} (compute/kernel.h:640-700) over b2_reduce
// ------------------------------------------------------------------------------------------
enum ScalarAggKind { kAggSum, kAggMean, kAggMinMax, kAggCount };

struct ScalarAggState : public cp::KernelState {
  int kind = kAggSum;
  Runtime* rt = nullptr;  // consume runs under a KernelContext without a kernel (exec.cc:1175-1177), so keep it here
  cp::ScalarAggregateOptions options = cp::ScalarAggregateOptions::Defaults();
  cp::CountOptions count_options = cp::CountOptions::Defaults();
  std::shared_ptr<DataType> in_type;
  int acc_type = B2_INT64;
  int64_t length = 0, count = 0, nulls = 0;
  uint64_t sum_bits = 0;  // int64 / uint64 sums wrap the same way in two's complement
  double fsum = 0, dsum = 0;
  uint64_t min_bits = 0, max_bits = 0;
  bool has_minmax = false;

  static double AsDouble(uint64_t b) {
    double d;
    std::memcpy(&d, &b, 8);
    return d;
  }
  void MergeMinMax(uint64_t lo, uint64_t hi) {
    if (!has_minmax) {
      min_bits = lo;
      max_bits = hi;
      has_minmax = true;
      return;
    }
    if (acc_type == B2_DOUBLE) {  // std::fmin / std::fmax: NaN is the identity (aggregate_basic.inc.cc:680-701)
      double a = std::fmin(AsDouble(min_bits), AsDouble(lo)), b = std::fmax(AsDouble(max_bits), AsDouble(hi));
      std::memcpy(&min_bits, &a, 8);
      std::memcpy(&max_bits, &b, 8);
    } else if (acc_type == B2_INT64) {
      min_bits = static_cast<uint64_t>(std::min(static_cast<int64_t>(min_bits), static_cast<int64_t>(lo)));
      max_bits = static_cast<uint64_t>(std::max(static_cast<int64_t>(max_bits), static_cast<int64_t>(hi)));
    } else {
      min_bits = std::min(min_bits, lo);
      max_bits = std::max(max_bits, hi);
    }
  }
};

template <int KIND>
static Result<std::unique_ptr<cp::KernelState>> ScalarAggInit(cp::KernelContext*, const cp::KernelInitArgs& args) {
  auto st = std::make_unique<ScalarAggState>();
  st->kind = KIND;
  st->rt = checked_cast<const KernelData&>(*args.kernel->data).rt;
  st->in_type = args.inputs[0].GetSharedPtr();
  if (KIND == kAggCount) {
    if (auto o = static_cast<const cp::CountOptions*>(args.options)) st->count_options = *o;
  } else if (auto o = static_cast<const cp::ScalarAggregateOptions*>(args.options)) {
    st->options = *o;
  }
  return st;
}

static Status ScalarAggConsume(cp::KernelContext* ctx, const cp::ExecSpan& batch) {
  auto* st = checked_cast<ScalarAggState*>(ctx->state());
  if (!batch[0].is_array()) return Status::NotImplemented("device aggregates over a scalar argument");
  B2Array v;
  ARROW_RETURN_NOT_OK(SpanToB2(batch[0].array, &v));
  st->length += v.length;
  if (st->kind == kAggCount) {
    int64_t valid = v.length;
    if (v.validity && v.null_count != 0) B200_RETURN_NOT_OK(b2_bitmap_count(st->rt->context(), v.validity, v.offset, v.length, &valid, nullptr));
    st->count += valid;
    st->nulls += v.length - valid;
    return Status::OK();
  }
  B2ReduceResult r;
  B200_RETURN_NOT_OK(b2_reduce(st->rt->context(), &v, &r, nullptr));
  st->acc_type = r.acc_type;
  st->count += r.count;
  st->nulls += r.null_count;
  st->sum_bits += r.sum_bits;
  st->fsum += ScalarAggState::AsDouble(r.sum_bits);
  st->dsum += ScalarAggState::AsDouble(r.dsum_bits);
  if (r.count > 0) st->MergeMinMax(r.min_bits, r.max_bits);
  return Status::OK();
}

static Status ScalarAggMerge(cp::KernelContext*, cp::KernelState&& src, cp::KernelState* dst) {
  auto& o = checked_cast<ScalarAggState&>(src);
  auto* st = checked_cast<ScalarAggState*>(dst);
  st->acc_type = o.length ? o.acc_type : st->acc_type;
  st->length += o.length;
  st->count += o.count;
  st->nulls += o.nulls;
  st->sum_bits += o.sum_bits;
  st->fsum += o.fsum;
  st->dsum += o.dsum;
  if (o.has_minmax) st->MergeMinMax(o.min_bits, o.max_bits);
  return Status::OK();
}

static Status ScalarAggFinalize(cp::KernelContext* ctx, Datum* out) {
  auto* st = checked_cast<ScalarAggState*>(ctx->state());
  const auto& o = st->options;
  const bool floating = arrow::is_floating(st->in_type->id());
  const bool is_signed = arrow::is_signed_integer(st->in_type->id());
  switch (st->kind) {
    case kAggCount: {
      const auto mode = st->count_options.mode;
      const int64_t v = mode == cp::CountOptions::ONLY_VALID ? st->count : (mode == cp::CountOptions::ONLY_NULL ? st->nulls : st->length);
      *out = Datum(std::make_shared<arrow::Int64Scalar>(v));
      return Status::OK();
    }
    case kAggSum: {
      const bool null = (!o.skip_nulls && st->nulls > 0) || st->count < static_cast<int64_t>(o.min_count);
      if (floating) *out = Datum(null ? std::make_shared<arrow::DoubleScalar>() : std::make_shared<arrow::DoubleScalar>(st->fsum));
      else if (is_signed) *out = Datum(null ? std::make_shared<arrow::Int64Scalar>() : std::make_shared<arrow::Int64Scalar>(static_cast<int64_t>(st->sum_bits)));
      else *out = Datum(null ? std::make_shared<arrow::UInt64Scalar>() : std::make_shared<arrow::UInt64Scalar>(st->sum_bits));
      return Status::OK();
    }
    case kAggMean: {
      const bool null = (!o.skip_nulls && st->nulls > 0) || st->count < static_cast<int64_t>(o.min_count);
      *out = Datum(null ? std::make_shared<arrow::DoubleScalar>() : std::make_shared<arrow::DoubleScalar>(st->dsum / static_cast<double>(st->count)));
      return Status::OK();
    }
    default: {
      auto type = arrow::struct_({arrow::field("min", st->in_type), arrow::field("max", st->in_type)});
      const int64_t min_count = std::max<int64_t>(1, o.min_count);  // aggregate_basic.inc.cc:783
      std::shared_ptr<arrow::Scalar> lo = arrow::MakeNullScalar(st->in_type), hi = lo;
      if (!((st->nulls > 0 && !o.skip_nulls) || st->count < min_count)) {
        std::shared_ptr<arrow::Scalar> wlo, whi;
        if (floating) {
          wlo = std::make_shared<arrow::DoubleScalar>(ScalarAggState::AsDouble(st->min_bits));
          whi = std::make_shared<arrow::DoubleScalar>(ScalarAggState::AsDouble(st->max_bits));
        } else if (is_signed) {
          wlo = std::make_shared<arrow::Int64Scalar>(static_cast<int64_t>(st->min_bits));
          whi = std::make_shared<arrow::Int64Scalar>(static_cast<int64_t>(st->max_bits));
        } else {
          wlo = std::make_shared<arrow::UInt64Scalar>(st->min_bits);
          whi = std::make_shared<arrow::UInt64Scalar>(st->max_bits);
        }
        ARROW_ASSIGN_OR_RAISE(lo, wlo->CastTo(st->in_type));
        ARROW_ASSIGN_OR_RAISE(hi, whi->CastTo(st->in_type));
      }
      *out = Datum(std::make_shared<arrow::StructScalar>(arrow::ScalarVector{lo, hi}, type));
      return Status::OK();
    }
  }
}

static Result<TypeHolder> SumType(cp::KernelContext*, const std::vector<TypeHolder>& types) {
  const auto id = types[0].id();
  if (arrow::is_floating(id)) return TypeHolder(arrow::float64());
  return TypeHolder(arrow::is_signed_integer(id) ? arrow::int64() : arrow::uint64());
}
static Result<TypeHolder> MinMaxType(cp::KernelContext*, const std::vector<TypeHolder>& types) {
  return TypeHolder(arrow::struct_({arrow::field("min", types[0].GetSharedPtr()), arrow::field("max", types[0].GetSharedPtr())}));
}

static Status AddScalarAggregates(cp::FunctionRegistry* reg, Runtime* rt) {
  static const cp::ScalarAggregateOptions kAggDefaults = cp::ScalarAggregateOptions::Defaults();
  static const cp::CountOptions kCountDefaults = cp::CountOptions::Defaults();
  auto add = [&](const char* name, cp::KernelInit init, cp::OutputType out, const cp::FunctionOptions* defaults, const char* options_class,
                 bool any_type) -> Status {
    auto fn = std::make_shared<Forwarding<cp::ScalarAggregateFunction>>(name, cp::Arity::Unary(), DocFor({"array"}, options_class), defaults);
    auto add_kernel = [&](cp::InputType in) {
      cp::ScalarAggregateKernel k(cp::KernelSignature::Make({std::move(in)}, out), init, ScalarAggConsume, ScalarAggMerge, ScalarAggFinalize,
                                  /*ordered=*/false);
      k.data = std::make_shared<KernelData>(rt, 0);
      return fn->AddKernel(std::move(k));
    };
    if (any_type) ARROW_RETURN_NOT_OK(add_kernel(cp::InputType::Any()));
    else
      for (const auto& ty : NumericTypes()) ARROW_RETURN_NOT_OK(add_kernel(cp::InputType(ty)));
    return reg->AddFunction(std::move(fn), true);
  };
  ARROW_RETURN_NOT_OK(add("sum", ScalarAggInit<kAggSum>, cp::OutputType(SumType), &kAggDefaults, "ScalarAggregateOptions", false));
  ARROW_RETURN_NOT_OK(add("mean", ScalarAggInit<kAggMean>, cp::OutputType(arrow::float64()), &kAggDefaults, "ScalarAggregateOptions", false));
  ARROW_RETURN_NOT_OK(add("min_max", ScalarAggInit<kAggMinMax>, cp::OutputType(MinMaxType), &kAggDefaults, "ScalarAggregateOptions", false));
  return add("count", ScalarAggInit<kAggCount>, cp::OutputType(arrow::int64()), &kCountDefaults, "CountOptions", true);
}

// ------------------------------------------------------------------------------------------
// hash aggregates: the HashAggregateKernel contract (compute/kernel.h:720-769)
// ------------------------------------------------------------------------------------------
struct HashAggState : public cp::KernelState {
  ~HashAggState() override {
    if (agg) b2_hashagg_destroy(agg);
  }
  Runtime* rt = nullptr;
  B2HashAgg* agg = nullptr;
  std::shared_ptr<DataType> out_type;
};

struct HashAggKernelData : public cp::KernelState {
  HashAggKernelData(Runtime* r, int k) : rt(r), kind(k) {}
  Runtime* rt;
  int kind;
};

static std::shared_ptr<DataType> HashAggOutType(int kind, const DataType& in) {
  switch (kind) {
    case B2_HASH_COUNT: case B2_HASH_COUNT_ALL: case B2_HASH_COUNT_DISTINCT: return arrow::int64();
    case B2_HASH_MEAN: return arrow::float64();
    case B2_HASH_ANY: case B2_HASH_ALL: return arrow::boolean();
    case B2_HASH_SUM: case B2_HASH_PRODUCT:
      if (arrow::is_signed_integer(in.id())) return arrow::int64();
      if (arrow::is_unsigned_integer(in.id())) return arrow::uint64();
      return arrow::float64();
    default: return in.GetSharedPtr();
  }
}

static Result<std::unique_ptr<cp::KernelState>> HashAggInit(cp::KernelContext* ctx, const cp::KernelInitArgs& args) {
  const auto& kd = checked_cast<const HashAggKernelData&>(*args.kernel->data);
  auto st = std::make_unique<HashAggState>();
  st->rt = kd.rt;
  B2HashAggOptions o{1, 1, 0, 0};
  if (kd.kind == B2_HASH_COUNT || kd.kind == B2_HASH_COUNT_DISTINCT) {
    if (auto co = static_cast<const cp::CountOptions*>(args.options))
      o.count_mode = co->mode == cp::CountOptions::ONLY_VALID ? 0 : co->mode == cp::CountOptions::ONLY_NULL ? 1 : 2;
  } else if (kd.kind != B2_HASH_COUNT_ALL) {
    if (auto so = static_cast<const cp::ScalarAggregateOptions*>(args.options)) {
      o.skip_nulls = so->skip_nulls;
      o.min_count = so->min_count;
    }
  }
  int vt = B2_NA;
  const DataType* in_type = nullptr;
  if (kd.kind != B2_HASH_COUNT_ALL) {
    in_type = args.inputs[0].type;
    ARROW_ASSIGN_OR_RAISE(vt, B2TypeId(*in_type));
  }
  B200_RETURN_NOT_OK(b2_hashagg_create(kd.rt->context(), kd.kind, vt, &o, &st->agg));
  st->out_type = in_type ? HashAggOutType(kd.kind, *in_type) : arrow::int64();
  return st;
}

static HashAggState* AggOf(cp::KernelContext* ctx) { return checked_cast<HashAggState*>(ctx->state()); }

static Status HashAggResize(cp::KernelContext* ctx, int64_t num_groups) {
  B200_RETURN_NOT_OK(b2_hashagg_resize(AggOf(ctx)->agg, num_groups, nullptr));
  return Status::OK();
}
static Status HashAggConsume(cp::KernelContext* ctx, const cp::ExecSpan& batch) {
  B2Array v, ids;
  const bool count_all = batch.num_values() == 1;
  if (!count_all) ARROW_RETURN_NOT_OK(SpanToB2(batch[0].array, &v));
  ARROW_RETURN_NOT_OK(SpanToB2(batch[count_all ? 0 : 1].array, &ids));
  B200_RETURN_NOT_OK(b2_hashagg_consume(AggOf(ctx)->agg, count_all ? nullptr : &v, &ids, nullptr));
  return Status::OK();
}
static Status HashAggMerge(cp::KernelContext* ctx, cp::KernelState&& other, const ArrayData& mapping) {
  B2Array m;
  ARROW_RETURN_NOT_OK(DataToB2(mapping, &m));
  B200_RETURN_NOT_OK(b2_hashagg_merge(AggOf(ctx)->agg, checked_cast<HashAggState&>(other).agg, &m, nullptr));
  return Status::OK();
}
static Status HashAggFinalize(cp::KernelContext* ctx, Datum* out) {
  HashAggState* st = AggOf(ctx);
  B2Array o;
  B200_RETURN_NOT_OK(b2_hashagg_finalize(st->agg, &o, nullptr));
  *out = Datum(AdoptOutput(st->rt, o, st->out_type));
  return Status::OK();
}

static Status AddHashAggregate(cp::FunctionRegistry* reg, Runtime* rt, const std::string& name, int kind) {
  static const cp::ScalarAggregateOptions kAggDefaults = cp::ScalarAggregateOptions::Defaults();
  static const cp::CountOptions kCountDefaults = cp::CountOptions::Defaults();
  const bool count_opts = kind == B2_HASH_COUNT || kind == B2_HASH_COUNT_DISTINCT;
  const cp::FunctionOptions* defaults = count_opts ? static_cast<const cp::FunctionOptions*>(&kCountDefaults)
                                        : kind == B2_HASH_COUNT_ALL ? nullptr : &kAggDefaults;
  auto fn = std::make_shared<cp::HashAggregateFunction>(
      name, kind == B2_HASH_COUNT_ALL ? cp::Arity::Unary() : cp::Arity::Binary(),
      kind == B2_HASH_COUNT_ALL ? DocFor({"group_id_array"})
                                : DocFor({"array", "group_id_array"}, count_opts ? "CountOptions" : "ScalarAggregateOptions"),
      defaults);
  auto out_resolver = [kind](cp::KernelContext* ctx, const std::vector<TypeHolder>& types) -> Result<TypeHolder> {
    if (kind == B2_HASH_COUNT_ALL) return TypeHolder(arrow::int64());
    return TypeHolder(HashAggOutType(kind, *types[0].type));
  };
  auto add = [&](std::vector<cp::InputType> in) {
    cp::HashAggregateKernel k(cp::KernelSignature::Make(std::move(in), cp::OutputType(out_resolver)), HashAggInit, HashAggResize,
                              HashAggConsume, HashAggMerge, HashAggFinalize, /*ordered=*/false);
    k.data = std::make_shared<HashAggKernelData>(rt, kind);
    return fn->AddKernel(std::move(k));
  };
  if (kind == B2_HASH_COUNT_ALL) {
    ARROW_RETURN_NOT_OK(add({cp::InputType(arrow::uint32())}));
  } else if (kind == B2_HASH_COUNT) {
    ARROW_RETURN_NOT_OK(add({cp::InputType::Any(), cp::InputType(arrow::uint32())}));
  } else if (kind == B2_HASH_ANY || kind == B2_HASH_ALL) {
    ARROW_RETURN_NOT_OK(add({cp::InputType(arrow::boolean()), cp::InputType(arrow::uint32())}));
  } else if (kind == B2_HASH_COUNT_DISTINCT) {
    for (const auto& ty : NumericTypes()) ARROW_RETURN_NOT_OK(add({cp::InputType(ty), cp::InputType(arrow::uint32())}));
    for (const auto& ty : {arrow::utf8(), arrow::large_utf8(), arrow::binary(), arrow::large_binary()})
      ARROW_RETURN_NOT_OK(add({cp::InputType(ty), cp::InputType(arrow::uint32())}));
  } else {
    for (const auto& ty : NumericTypes()) ARROW_RETURN_NOT_OK(add({cp::InputType(ty), cp::InputType(arrow::uint32())}));
  }
  return reg->AddFunction(std::move(fn), true);
}

// ------------------------------------------------------------------------------------------
// Grouper
// ------------------------------------------------------------------------------------------
class DeviceGrouper : public cp::Grouper {
 public:
  DeviceGrouper(Runtime* rt, std::vector<TypeHolder> key_types, B2Grouper* g)
      : rt_(rt), key_types_(std::move(key_types)), g_(g) {}
  ~DeviceGrouper() override { b2_grouper_destroy(g_); }

  Status Reset() override {
    B200_RETURN_NOT_OK(b2_grouper_reset(g_));
    return Status::OK();
  }
  Result<Datum> Consume(const cp::ExecSpan& batch, int64_t offset, int64_t length) override { return Run(batch, offset, length, true); }
  Result<Datum> Lookup(const cp::ExecSpan& batch, int64_t offset, int64_t length) override { return Run(batch, offset, length, false); }
  Status Populate(const cp::ExecSpan& batch, int64_t offset, int64_t length) override { return Run(batch, offset, length, true).status(); }
  uint32_t num_groups() const override {
    uint32_t n = 0;
    b2_grouper_num_groups(g_, &n);
    return n;
  }
  Result<cp::ExecBatch> GetUniques() override {
    std::vector<B2Array> outs(key_types_.size());
    B200_RETURN_NOT_OK(b2_grouper_uniques(g_, outs.data(), nullptr));
    cp::ExecBatch batch({}, num_groups());
    for (size_t i = 0; i < outs.size(); ++i) batch.values.emplace_back(AdoptOutput(rt_, outs[i], key_types_[i].GetSharedPtr()));
    return batch;
  }

 private:
  Result<Datum> Run(const cp::ExecSpan& batch, int64_t offset, int64_t length, bool insert) {
    if (static_cast<size_t>(batch.num_values()) != key_types_.size())
      return Status::Invalid("expected batch size ", key_types_.size(), " but got ", batch.num_values());
    if (offset < 0 || offset > batch.length) return Status::Invalid("invalid grouper consume offset: ", offset);
    if (length < 0) length = batch.length - offset;
    std::vector<B2Array> keys(key_types_.size());
    for (size_t i = 0; i < keys.size(); ++i) {
      if (!batch[i].is_array()) return Status::NotImplemented("arrow_b200 grouper: scalar key columns");
      if (!batch[i].type()->Equals(*key_types_[i].type))
        return Status::Invalid("expected batch value ", i, " of type ", key_types_[i].type->ToString(), " but got ", batch[i].type()->ToString());
      ARROW_RETURN_NOT_OK(SpanToB2(batch[i].array, &keys[i]));
      keys[i].offset += offset;
      keys[i].length = length;
    }
    B2Array ids;
    B200_RETURN_NOT_OK((insert ? b2_grouper_consume : b2_grouper_lookup)(g_, keys.data(), &ids, nullptr));
    return Datum(AdoptOutput(rt_, ids, arrow::uint32()));
  }
  Runtime* rt_;
  std::vector<TypeHolder> key_types_;
  B2Grouper* g_;
};

Result<std::unique_ptr<cp::Grouper>> MakeGrouper(const std::vector<TypeHolder>& key_types, Runtime* rt) {
  std::vector<int32_t> ids;
  for (const auto& t : key_types) {
    ARROW_ASSIGN_OR_RAISE(int id, B2TypeId(*t.type));
    ids.push_back(id);
  }
  B2Grouper* g = nullptr;
  B200_RETURN_NOT_OK(b2_grouper_create(rt->context(), ids.data(), static_cast<int>(ids.size()), &g));
  return std::unique_ptr<cp::Grouper>(new DeviceGrouper(rt, key_types, g));
}

// ------------------------------------------------------------------------------------------
Status RegisterFunctions(cp::FunctionRegistry* reg, Runtime* rt) {
  const std::pair<const char*, int> arith[] = {{"add", B2_ADD}, {"subtract", B2_SUBTRACT}, {"multiply", B2_MULTIPLY},
                                               {"divide", B2_DIVIDE}, {"add_checked", B2_ADD_CHECKED},
                                               {"subtract_checked", B2_SUBTRACT_CHECKED},
                                               {"multiply_checked", B2_MULTIPLY_CHECKED}, {"divide_checked", B2_DIVIDE_CHECKED}};
  for (const auto& a : arith) ARROW_RETURN_NOT_OK(AddBinaryFunction(reg, rt, a.first, a.second, false));
  const std::pair<const char*, int> cmp[] = {{"equal", B2_EQUAL}, {"not_equal", B2_NOT_EQUAL}, {"greater", B2_GREATER},
                                             {"greater_equal", B2_GREATER_EQUAL}, {"less", B2_LESS}, {"less_equal", B2_LESS_EQUAL}};
  for (const auto& c : cmp) ARROW_RETURN_NOT_OK(AddBinaryFunction(reg, rt, c.first, c.second, true));
  ARROW_RETURN_NOT_OK(AddLogicFunctions(reg, rt));
  ARROW_RETURN_NOT_OK(reg->AddFunction(std::make_shared<CastFunction>(rt), true));
  ARROW_RETURN_NOT_OK(AddSelectionFunctions(reg, rt));
  ARROW_RETURN_NOT_OK(reg->AddFunction(std::make_shared<SortIndicesFunction>(rt), true));
  ARROW_RETURN_NOT_OK(reg->AddFunction(std::make_shared<SelectKFunction>(rt), true));
  ARROW_RETURN_NOT_OK(AddHashFunctions(reg, rt));
  ARROW_RETURN_NOT_OK(AddScalarAggregates(reg, rt));
  const std::pair<const char*, int> aggs[] = {{"hash_sum", B2_HASH_SUM}, {"hash_count", B2_HASH_COUNT},
                                              {"hash_count_all", B2_HASH_COUNT_ALL}, {"hash_mean", B2_HASH_MEAN},
                                              {"hash_min", B2_HASH_MIN}, {"hash_max", B2_HASH_MAX},
                                              {"hash_product", B2_HASH_PRODUCT}, {"hash_any", B2_HASH_ANY}, {"hash_all", B2_HASH_ALL},
                                              {"hash_count_distinct", B2_HASH_COUNT_DISTINCT}};
  for (const auto& a : aggs) ARROW_RETURN_NOT_OK(AddHashAggregate(reg, rt, a.first, a.second));
  return Status::OK();
}

}  // namespace arrow_b200

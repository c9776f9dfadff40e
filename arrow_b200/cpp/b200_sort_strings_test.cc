// b200_sort_strings_test.cc -- parity of the C++ drop-in's sorts over utf8 / binary keys against the reference
// itself: array_sort_indices, sort_indices on a device record batch, select_k_unstable and the b200_order_by Acero
// node go through the stock CPU registry / order_by node and through the nested B200 registry / b200_order_by with
// the same inputs; results (and error texts) must be equal.  Prints one line per check, exits non-zero on a failure.
#include <arrow/acero/exec_plan.h>
#include <arrow/acero/options.h>
#include <arrow/api.h>
#include <arrow/compute/api.h>
#include <arrow/compute/initialize.h>

#include <iostream>
#include <random>

#include "b200_compute.h"

namespace cp = arrow::compute;
namespace ac = arrow::acero;
using arrow::Datum;

static int g_checks = 0;

#define CHECK_OK(expr)                                                         \
  do {                                                                         \
    auto _st = (expr);                                                         \
    if (!_st.ok()) {                                                           \
      std::cout << "FAIL " << __LINE__ << ": " << _st.ToString() << std::endl; \
      std::exit(1);                                                            \
    }                                                                          \
  } while (0)

template <typename T>
T Unwrap(arrow::Result<T> r, int line) {
  if (!r.ok()) {
    std::cout << "FAIL " << line << ": " << r.status().ToString() << std::endl;
    std::exit(1);
  }
  return std::move(r).ValueUnsafe();
}
#define UNWRAP(expr) Unwrap((expr), __LINE__)

static void Fail(const std::string& what) {
  std::cout << "FAIL " << what << std::endl;
  std::exit(1);
}

// n strings over a small alphabet that includes NUL and a byte >= 0x80, lengths 0..max_len, so that prefixes,
// duplicates and ties are common
template <typename Builder>
std::shared_ptr<arrow::Array> RandomStrings(int64_t n, int max_len, double null_p, uint64_t seed) {
  std::mt19937_64 rng(seed);
  std::uniform_real_distribution<double> u(0, 1);
  std::uniform_int_distribution<int> len(0, max_len), ch(0, 3);
  const char alphabet[4] = {'a', 'b', '\0', static_cast<char>(0xc3)};
  Builder b;
  for (int64_t i = 0; i < n; ++i) {
    if (u(rng) < null_p) {
      CHECK_OK(b.AppendNull());
    } else {
      std::string s(len(rng), ' ');
      for (auto& c : s) c = alphabet[ch(rng)];
      CHECK_OK(b.Append(s));
    }
  }
  return UNWRAP(b.Finish());
}

struct Harness {
  arrow_b200::Runtime* rt;
  cp::ExecContext cpu_ctx;
  cp::ExecContext gpu_ctx;
  explicit Harness(arrow_b200::Runtime* r)
      : rt(r), cpu_ctx(arrow::default_memory_pool()), gpu_ctx(arrow::default_memory_pool(), nullptr, r->registry()) {}

  std::shared_ptr<arrow::Array> Dev(const std::shared_ptr<arrow::Array>& a) {
    return arrow::MakeArray(UNWRAP(arrow_b200::ToDevice(*a->data(), rt->memory_manager())));
  }
  std::shared_ptr<arrow::Array> Host(const Datum& d) { return arrow::MakeArray(UNWRAP(arrow_b200::ToHost(*d.array()))); }

  // the same call through both registries: equal results, or the same error
  void Check(const std::string& what, const std::string& fn, const std::vector<Datum>& host_args, const std::vector<Datum>& dev_args,
             const cp::FunctionOptions* opts, bool compare_values_of = false) {
    auto want = cp::CallFunction(fn, host_args, opts, &cpu_ctx);
    auto got = cp::CallFunction(fn, dev_args, opts, &gpu_ctx);
    ++g_checks;
    if (!want.ok() || !got.ok()) {
      if (want.ok() != got.ok() || want.status().code() != got.status().code() || want.status().message() != got.status().message())
        Fail(what + ": reference -> " + want.status().ToString() + " ; device -> " + got.status().ToString());
      std::cout << "OK   " << what << " (same error: " << want.status().message() << ")" << std::endl;
      return;
    }
    if (got->length() > 0 && !arrow_b200::IsOnDevice(*got->array())) Fail(what + ": result is not on the device");
    auto w = want->make_array();
    auto g = Host(*got);
    if (compare_values_of) {  // select_k_unstable: ties may come in any order, the selected values may not
      const auto& values = host_args[0];
      w = UNWRAP(cp::Take(values, w, cp::TakeOptions::Defaults(), &cpu_ctx)).make_array();
      g = UNWRAP(cp::Take(values, g, cp::TakeOptions::Defaults(), &cpu_ctx)).make_array();
    }
    if (!g->Equals(*w))
      Fail(what + ": arrays differ\n  want: " + w->ToString().substr(0, 300) + "\n  got:  " + g->ToString().substr(0, 300));
    std::cout << "OK   " << what << " (" << g->length() << " rows)" << std::endl;
  }
};

int main() {
  CHECK_OK(cp::Initialize());
  auto rt = UNWRAP(arrow_b200::Runtime::Get(0));
  CHECK_OK(arrow_b200::RegisterAceroNodes());
  Harness h(rt);
  const int64_t n = 40000;
  std::vector<std::pair<std::string, std::shared_ptr<arrow::Array>>> cols = {
      {"utf8", RandomStrings<arrow::StringBuilder>(n, 12, 0.1, 0x0ff1ce)},
      {"large_utf8", RandomStrings<arrow::LargeStringBuilder>(n, 20, 0.1, 0x0ff1cf)},
      {"binary", RandomStrings<arrow::BinaryBuilder>(n, 9, 0.0, 0x0ff1d0)},
      {"large_binary", RandomStrings<arrow::LargeBinaryBuilder>(n, 16, 0.3, 0x0ff1d1)},
  };

  // ---- array_sort_indices / sort_indices on one array (sliced: non-zero offsets) ----
  for (auto& [name, full] : cols) {
    auto a = full->Slice(7, n - 20);
    auto d = h.Dev(full)->Slice(7, n - 20);
    for (auto order : {cp::SortOrder::Ascending, cp::SortOrder::Descending}) {
      for (auto np : {cp::NullPlacement::AtEnd, cp::NullPlacement::AtStart}) {
        const std::string tag = std::string(order == cp::SortOrder::Ascending ? " asc" : " desc") + (np == cp::NullPlacement::AtEnd ? " at_end" : " at_start");
        cp::ArraySortOptions o(order, np);
        h.Check("array_sort_indices(" + name + ")" + tag, "array_sort_indices", {a}, {d}, &o);
        cp::SortOptions so({cp::SortKey("not-used", order)}, np);
        h.Check("sort_indices(" + name + ")" + tag, "sort_indices", {a}, {d}, &so);
      }
    }
  }

  // ---- select_k_unstable: the selected values (ties may come in any order) ----
  for (auto& [name, full] : cols) {
    auto d = h.Dev(full);
    for (int64_t k : {int64_t(0), int64_t(1), int64_t(100), int64_t(3000)}) {
      for (auto order : {cp::SortOrder::Ascending, cp::SortOrder::Descending}) {
        cp::SelectKOptions so(k, {cp::SortKey("not-used", order)});
        h.Check("select_k_unstable(" + name + ") k=" + std::to_string(k) + (order == cp::SortOrder::Ascending ? " asc" : " desc"),
                "select_k_unstable", {full}, {d}, &so, /*compare_values_of=*/true);
      }
    }
  }
  {
    cp::SelectKOptions bad(-1, {cp::SortKey("not-used")});
    h.Check("select_k_unstable(utf8) k=-1 error", "select_k_unstable", {cols[0].second}, {h.Dev(cols[0].second)}, &bad);
  }

  // ---- sort_indices over a record batch of device columns: string keys first, last and twice, numeric tie-break ----
  std::shared_ptr<arrow::Array> num;
  {
    std::mt19937_64 rng(0x0ff1d3);
    arrow::Int32Builder b;
    for (int64_t i = 0; i < n; ++i) {
      if (rng() % 10 == 0) CHECK_OK(b.AppendNull());
      else CHECK_OK(b.Append(static_cast<int32_t>(rng() % 5)));
    }
    num = UNWRAP(b.Finish());
  }
  auto schema = arrow::schema({arrow::field("s", arrow::utf8()), arrow::field("t", arrow::large_binary()), arrow::field("i", arrow::int32())});
  auto host_batch = arrow::RecordBatch::Make(schema, n, {cols[0].second, cols[3].second, num});
  auto dev_batch = arrow::RecordBatch::Make(schema, n, {h.Dev(cols[0].second), h.Dev(cols[3].second), h.Dev(num)});
  const std::vector<std::vector<cp::SortKey>> key_sets = {
      {cp::SortKey("s", cp::SortOrder::Ascending), cp::SortKey("i", cp::SortOrder::Descending)},
      {cp::SortKey("i", cp::SortOrder::Ascending), cp::SortKey("s", cp::SortOrder::Descending)},
      {cp::SortKey("t", cp::SortOrder::Descending), cp::SortKey("s", cp::SortOrder::Ascending)},
  };
  for (const auto& keys : key_sets) {
    for (auto np : {cp::NullPlacement::AtEnd, cp::NullPlacement::AtStart}) {
      cp::SortOptions so(keys, np);
      std::string what = "sort_indices(record batch:";
      for (const auto& k : keys) what += " " + k.target.ToString() + (k.order == cp::SortOrder::Ascending ? " asc" : " desc");
      what += np == cp::NullPlacement::AtEnd ? ", at_end)" : ", at_start)";
      h.Check(what, "sort_indices", {Datum(host_batch)}, {Datum(dev_batch)}, &so);
    }
  }
  {
    cp::SortOptions none(std::vector<cp::SortKey>{});
    h.Check("sort_indices(record batch) without keys error", "sort_indices", {Datum(host_batch)}, {Datum(dev_batch)}, &none);
  }

  // ---- Acero: order_by vs b200_order_by with a string key and a numeric tie-break ----
  auto table = arrow::Table::Make(schema, {cols[0].second, cols[3].second, num});
  auto run = [&](const std::string& factory, const cp::Ordering& ord) {
    ac::Declaration plan = ac::Declaration::Sequence({{"table_source", ac::TableSourceNodeOptions(table, 1 << 13)},
                                                      {factory, ac::OrderByNodeOptions(ord)}});
    return UNWRAP(ac::DeclarationToTable(std::move(plan), /*use_threads=*/false));
  };
  for (auto np : {cp::NullPlacement::AtEnd, cp::NullPlacement::AtStart}) {
    cp::Ordering ord({cp::SortKey("s", cp::SortOrder::Descending), cp::SortKey("i", cp::SortOrder::Ascending)}, np);
    auto want = run("order_by", ord), got = run("b200_order_by", ord);
    ++g_checks;
    if (!got->CombineChunks().ValueOrDie()->Equals(*want->CombineChunks().ValueOrDie())) Fail("b200_order_by (s desc, i asc)");
    std::cout << "OK   b200_order_by == order_by (utf8 key descending, int32 tie-break, "
              << (np == cp::NullPlacement::AtEnd ? "nulls last" : "nulls first") << ", " << got->num_rows() << " rows)" << std::endl;
  }
  std::cout << "PASS " << g_checks << " checks; " << b2_launch_count() << " kernels launched by libarrow_b200.so" << std::endl;
  return 0;
}

// C++ tests of the pd:: façade, written the way the reference's Catch2 tests are
// (/root/reference/tests/cudf_examples/dataframe_resample_test.cpp, series_resample_test.cpp,
// dataframe_iterator_test.cpp) so that they read like the reference's own; Catch2 is not installed,
// hence the tiny REQUIRE harness.  Needs a GPU (run by tests/test_facade_gpu.py).
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <filesystem>
#include <iostream>
#include <stdexcept>
#include <string>

#include <arrow/compute/api.h>
#include <arrow/io/api.h>
#include <arrow/ipc/api.h>
#include <arrow/table.h>
#include <parquet/arrow/writer.h>

#include "../../pandasarrow_b200/csrc/host/pd_groupby.h"

using namespace std::string_literals;

static int g_fail = 0, g_checks = 0;
#define REQUIRE(cond)                                                              \
  do {                                                                             \
    ++g_checks;                                                                    \
    if (!(cond)) { ++g_fail; std::printf("FAILED %s:%d  %s\n", __FILE__, __LINE__, #cond); } \
  } while (0)
#define REQUIRE_THROWS(expr)                                  \
  do {                                                        \
    ++g_checks;                                               \
    bool threw__ = false;                                     \
    try { expr; } catch (std::exception const&) { threw__ = true; } \
    if (!threw__) { ++g_fail; std::printf("FAILED %s:%d  expected throw: %s\n", __FILE__, __LINE__, #expr); } \
  } while (0)

static std::string str_at(const pd::ArrayPtr& a, int64_t i) { return pd::ReturnOrThrowOnFailure(a->GetScalar(i))->ToString(); }

static pd::DataFrame people() {
  return pd::DataFrame{pd::range(0L, 10L),
                       std::pair{"id"s, std::vector{"allen"s, "victor"s, "hannah"s, "allen"s, "victor"s, "hannah"s, "allen"s, "victor"s, "hannah"s, "allen"s}},
                       std::pair{"gender"s, std::vector{"male"s, "female"s, "male"s, "male"s, "female"s, "male"s, "male"s, "female"s, "male"s, "male"s}},
                       std::pair{"age"s, std::vector{16, 10, 10, 20, 30, 40, 15, 25, 35, 45}},
                       std::pair{"height"s, std::vector{9, 9, 9, 9, 9, 8, 8, 8, 8, 8}}};
}

// dataframe_resample_test.cpp:8-69 (grouping + order) and :71-250 (aggregates)
static void test_make_groups_and_aggregates() {
  auto df = people();
  pd::GroupBy by_id("id", df);
  REQUIRE(by_id.groupSize() == 3);
  REQUIRE(by_id.unique()->length() == 3);
  REQUIRE(str_at(by_id.unique(), 0) == "allen");
  REQUIRE(str_at(by_id.unique(), 1) == "victor");
  REQUIRE(str_at(by_id.unique(), 2) == "hannah");

  pd::GroupBy groupby("gender", df);
  REQUIRE(groupby.groupSize() == 2);
  REQUIRE(str_at(groupby.unique(), 0) == "male");
  REQUIRE(str_at(groupby.unique(), 1) == "female");

  auto age_mean = pd::ReturnOrThrowOnFailure(groupby.mean("age"));
  REQUIRE(std::fabs(age_mean[0].as<double>() - 25.857) < 1e-3);
  REQUIRE(std::fabs(age_mean[1].as<double>() - 21.667) < 1e-3);
  auto age_height_mean = pd::ReturnOrThrowOnFailure(groupby.mean({"age"s, "height"s}));
  REQUIRE(age_height_mean["age"][0].as<double>() == 25.857142857142858);
  REQUIRE(age_height_mean["age"][1].as<double>() == 21.666666666666668);
  REQUIRE(age_height_mean["height"][0].as<double>() == 8.428571428571429);
  REQUIRE(age_height_mean["height"][1].as<double>() == 8.666666666666666);

  auto age_mm = pd::ReturnOrThrowOnFailure(groupby.min_max("age"));
  REQUIRE(age_mm["min"][0].as<int32_t>() == 10);
  REQUIRE(age_mm["min"][1].as<int32_t>() == 10);
  REQUIRE(age_mm["max"][0].as<int32_t>() == 45);
  REQUIRE(age_mm["max"][1].as<int32_t>() == 30);
  auto ah_mm = pd::ReturnOrThrowOnFailure(groupby.min_max({"age"s, "height"s}));
  REQUIRE(ah_mm["age_min"][0].as<int32_t>() == 10);
  REQUIRE(ah_mm["age_max"][1].as<int32_t>() == 30);
  REQUIRE(ah_mm["height_min"][0].as<int32_t>() == 8);
  REQUIRE(ah_mm["height_max"][1].as<int32_t>() == 9);

  auto age_max = pd::ReturnOrThrowOnFailure(groupby.max("age"));
  REQUIRE(age_max[0].as<int32_t>() == 45);
  REQUIRE(age_max[1].as<int32_t>() == 30);
  auto ah_max = pd::ReturnOrThrowOnFailure(groupby.max({"age"s, "height"s}));
  REQUIRE(ah_max["height"][0].as<int32_t>() == 9);
  REQUIRE(ah_max["height"][1].as<int32_t>() == 9);
  auto age_min = pd::ReturnOrThrowOnFailure(groupby.min("age"));
  REQUIRE(age_min[0].as<int32_t>() == 10);
  REQUIRE(age_min[1].as<int32_t>() == 10);

  auto age_sum = pd::ReturnOrThrowOnFailure(groupby.sum("age"));
  REQUIRE(age_sum[0].as<int64_t>() == 181);
  REQUIRE(age_sum[1].as<int64_t>() == 65);
  REQUIRE(age_sum.dtype()->id() == arrow::Type::INT64);
  auto ah_sum = pd::ReturnOrThrowOnFailure(groupby.sum({"age"s, "height"s}));
  REQUIRE(ah_sum["height"][0].as<int64_t>() == 59);
  REQUIRE(ah_sum["height"][1].as<int64_t>() == 26);

  auto age_count = pd::ReturnOrThrowOnFailure(groupby.count("age"));
  REQUIRE(age_count[0].as<int64_t>() == 7);
  REQUIRE(age_count[1].as<int64_t>() == 3);

  REQUIRE_THROWS(pd::GroupBy("nope", df));                                 // group_by.h:27-30
  REQUIRE(!groupby.sum("nope").ok());
  REQUIRE(groupby.approximate_median("age").status().IsNotImplemented());
}

// dataframe_resample_test.cpp:252-305 — OHLC bars through group_by
static void test_bardata() {
  pd::DataFrame bardata{pd::range(0L, 5L),
                        std::pair("high"s, std::vector<float>{11.1f, 20.2f, 21.f, 15.f, 20.f}),
                        std::pair("low"s, std::vector<float>{9.1f, 9.2f, 10.f, 5.f, 10.f}),
                        std::pair("close"s, std::vector<float>{10.1f, 15.2f, 20.f, 15.f, 15.f}),
                        std::pair("open"s, std::vector<float>{10.f, 20.2f, 10.f, 15.f, 10.f}),
                        std::pair("volume"s, std::vector<uint64_t>{100, 200, 210, 1, 2}),
                        std::pair("day"s, std::vector<int64_t>{1, 1, 2, 2, 5})};
  auto grouper = bardata.group_by("day");
  REQUIRE(grouper.unique()->length() == 3);
  auto open = pd::ReturnOrThrowOnFailure(grouper.first("open"));
  auto close = pd::ReturnOrThrowOnFailure(grouper.last("close"));
  auto high = pd::ReturnOrThrowOnFailure(grouper.max("high"));
  auto low = pd::ReturnOrThrowOnFailure(grouper.min("low"));
  auto volume = pd::ReturnOrThrowOnFailure(grouper.sum("volume"));
  REQUIRE(open.values<float>() == (std::vector<float>{10.f, 10.f, 10.f}));
  REQUIRE(close.values<float>() == (std::vector<float>{15.2f, 15.f, 15.f}));
  REQUIRE(high.values<float>() == (std::vector<float>{20.2f, 21.f, 20.f}));
  REQUIRE(low.values<float>() == (std::vector<float>{9.1f, 5.f, 10.f}));
  REQUIRE(volume.values<uint64_t>() == (std::vector<uint64_t>{300, 211, 2}));
  REQUIRE(open.indexArray() == nullptr);      // dataframe.cpp:1748 quirk: first(string) has no key index
  REQUIRE(close.indexArray() != nullptr);
}

// dataframe_iterator_test.cpp:11-76 — per-group column sums
static void test_apply_sums() {
  auto df = pd::DataFrame(std::map<std::string, std::vector<int32_t>>{{"a", {1, 1, 3, 1, 1, 1, 3, 8, 2, 2}}, {"b", {10, 9, 8, 7, 6, 5, 4, 3, 2, 1}}});
  auto groupby = df.group_by("a"s);
  REQUIRE(groupby.groupSize() == 4);
  auto result = pd::ReturnOrThrowOnFailure(groupby.sum({"a"s, "b"s}));
  REQUIRE(result.num_rows() == 4);
  REQUIRE(result.num_columns() == 2);
  REQUIRE(result["a"].values<int64_t>() == (std::vector<int64_t>{5, 6, 8, 4}));
  REQUIRE(result["b"].values<int64_t>() == (std::vector<int64_t>{37, 12, 3, 3}));
  // group_by(ArrayPtr) (dataframe.cpp:1231-1235) and Series::group_by
  auto g2 = df.group_by(df["a"].array());
  REQUIRE(pd::ReturnOrThrowOnFailure(g2.sum("b")).values<int64_t>() == (std::vector<int64_t>{37, 12, 3, 3}));
  auto g3 = df["b"].group_by(df["a"].array());
  REQUIRE(pd::ReturnOrThrowOnFailure(g3.sum("b")).values<int64_t>() == (std::vector<int64_t>{37, 12, 3, 3}));
}

// dataframe_iterator_test.cpp:11-76 — apply callbacks over materialised groups (+ group(), MakeSubDataFrame,
// orderedGroups from cudf_examples/dataframe_resample_test.cpp:8-69)
static void test_apply_callbacks_and_groups() {
  auto df = pd::DataFrame(std::map<std::string, std::vector<int32_t>>{{"a", {1, 1, 3, 1, 1, 1, 3, 8, 2, 2}}, {"b", {10, 9, 8, 7, 6, 5, 4, 3, 2, 1}}});
  auto groupby = df.group_by("a"s);
  REQUIRE(groupby.groupSize() == 4);
  {
    // apply_chunk (dataframe.cpp:1411-1428): the callback's per-group frames concatenated in group order.  Here: every
    // group reduced to its first row -> one row per group, in first-appearance order of the keys 1, 3, 8, 2
    auto first_rows = pd::ReturnOrThrowOnFailure(groupby.apply_chunk([](pd::DataFrame const& g) {
      return pd::DataFrame(g.array()->Slice(0, 1), g.indexArray()->Slice(0, 1));
    }));
    REQUIRE(first_rows.num_rows() == 4);
    REQUIRE(first_rows["a"].values<int32_t>() == (std::vector<int32_t>{1, 3, 8, 2}));
    REQUIRE(first_rows["b"].values<int32_t>() == (std::vector<int32_t>{10, 8, 3, 2}));
    // identity callback: all rows back, grouped
    auto all = pd::ReturnOrThrowOnFailure(groupby.apply_chunk([](pd::DataFrame const& g) { return g; }));
    REQUIRE(all.num_rows() == 10);
    REQUIRE(all["a"].values<int32_t>() == (std::vector<int32_t>{1, 1, 1, 1, 1, 3, 3, 8, 2, 2}));
    REQUIRE(all["b"].values<int32_t>() == (std::vector<int32_t>{10, 9, 7, 6, 5, 8, 4, 3, 2, 1}));
  }
  auto col_sum = [](pd::Series const& s) -> std::shared_ptr<arrow::Scalar> { return s.sum().scalar; };
  auto result = pd::ReturnOrThrowOnFailure(groupby.apply(col_sum));
  REQUIRE(result.num_rows() == 4);
  REQUIRE(result.num_columns() == 2);
  REQUIRE(result["a"].values<int64_t>() == (std::vector<int64_t>{5, 6, 8, 4}));
  REQUIRE(result["b"].values<int64_t>() == (std::vector<int64_t>{37, 12, 3, 3}));
  auto frame_sum = [](pd::DataFrame const& s) -> std::shared_ptr<arrow::Scalar> { return s.sum().scalar; };
  auto rows = pd::ReturnOrThrowOnFailure(groupby.apply(frame_sum));
  REQUIRE(rows.size() == 4);
  REQUIRE(rows.values<int64_t>() == (std::vector<int64_t>{42, 18, 11, 7}));
  REQUIRE(pd::ReturnOrThrowOnFailure(groupby.apply_async(frame_sum)).values<int64_t>() == (std::vector<int64_t>{42, 18, 11, 7}));
  // per-group row order is the original row order (dataframe_resample_test.cpp:49-52)
  auto g1 = groupby.group(1);
  REQUIRE(g1.size() == 2);
  REQUIRE(g1[1]->length() == 5);
  REQUIRE(pd::Series(g1[1], nullptr).values<int64_t>() == (std::vector<int64_t>{10, 9, 7, 6, 5}));
  auto sub = groupby.MakeSubDataFrame(1, df.array()->schema());      // second group: key 3
  REQUIRE(sub.num_rows() == 2);
  REQUIRE(sub["b"].values<int64_t>() == (std::vector<int64_t>{8, 4}));
  REQUIRE(pd::Series(sub.indexArray(), nullptr).values<int64_t>() == (std::vector<int64_t>{2, 6}));
  REQUIRE_THROWS(groupby.group(77));
  auto ordered = groupby.orderedGroups<int64_t>();
  REQUIRE(ordered.size() == 4);
  REQUIRE(ordered[2].first == 8);
  REQUIRE(ordered[2].second.num_rows() == 1);
  // apply with an array-valued functor: rows come back group by group, indexed by the frame's index
  auto twice = [](pd::DataFrame const& s) -> pd::ArrayPtr {
    return arrow::compute::CallFunction("multiply", {s["b"].array(), arrow::MakeScalar(int32_t(2))}).ValueOrDie().make_array();
  };
  auto doubled = pd::ReturnOrThrowOnFailure(groupby.apply(twice));
  REQUIRE(doubled.size() == 10);
  REQUIRE(doubled.values<int64_t>() == (std::vector<int64_t>{20, 18, 14, 12, 10, 16, 8, 6, 4, 2}));
}

// GROUPBY_AGG(product) / GROUPBY_NUMERIC_AGG(variance|stddev) (dataframe.cpp:1516-1536): expected values from the
// same arrow::compute scalar kernels the reference calls per group
static pd::ArrayPtr int32_array(std::vector<int32_t> const& v) {
  arrow::Int32Builder b;
  pd::ThrowOnFailure(b.AppendValues(v));
  return pd::ReturnOrThrowOnFailure(b.Finish());
}

static void test_second_stage_aggregates() {
  auto df = people();
  pd::GroupBy groupby("gender", df);
  auto male = pd::ReturnOrThrowOnFailure(arrow::compute::CallFunction("variance", {int32_array({16, 10, 20, 40, 15, 35, 45})}));
  auto female = pd::ReturnOrThrowOnFailure(arrow::compute::CallFunction("variance", {int32_array({10, 30, 25})}));
  const double vm = male.scalar_as<arrow::DoubleScalar>().value, vf = female.scalar_as<arrow::DoubleScalar>().value;
  auto var = pd::ReturnOrThrowOnFailure(groupby.variance("age"));
  REQUIRE(std::fabs(var[0].as<double>() - vm) <= 1e-12 * vm);
  REQUIRE(std::fabs(var[1].as<double>() - vf) <= 1e-12 * vf);
  auto sd = pd::ReturnOrThrowOnFailure(groupby.stddev({"age"s, "height"s}));
  REQUIRE(std::fabs(sd["age"][0].as<double>() - std::sqrt(vm)) <= 1e-12 * std::sqrt(vm));
  REQUIRE(sd["height"].size() == 2);
  auto prod = pd::ReturnOrThrowOnFailure(groupby.product("age"));
  REQUIRE(prod[0].as<int64_t>() == int64_t(16) * 10 * 20 * 40 * 15 * 35 * 45);
  REQUIRE(prod[1].as<int64_t>() == int64_t(10) * 30 * 25);
  REQUIRE(!groupby.tdigest("age").ok());                      // still outside the path: NotImplemented, not a crash
  // GROUPBY_NUMERIC_AGG(all|any, bool): a boolean column
  pd::DataFrame flags{pd::range(0L, 6L), std::pair{"k"s, std::vector{1, 1, 2, 2, 3, 3}},
                      std::pair{"b"s, std::vector<bool>{true, true, true, false, false, false}}};
  pd::GroupBy by_k("k", flags);
  auto all = pd::ReturnOrThrowOnFailure(by_k.all("b"));
  auto any = pd::ReturnOrThrowOnFailure(by_k.any("b"));
  REQUIRE(all[0].as<bool>() && !all[1].as<bool>() && !all[2].as<bool>());
  REQUIRE(any[0].as<bool>() && any[1].as<bool>() && !any[2].as<bool>());
  auto nd = pd::ReturnOrThrowOnFailure(groupby.count_distinct("age"));     // male: 16 10 20 40 15 35 45, female: 10 30 25
  REQUIRE(nd[0].as<int64_t>() == 7 && nd[1].as<int64_t>() == 3);
  auto nh = pd::ReturnOrThrowOnFailure(groupby.count_distinct("height"));  // male: 9 9 9 8 8 8 8, female: 9 9 8
  REQUIRE(nh[0].as<int64_t>() == 2 && nh[1].as<int64_t>() == 2);
}

// series_resample_test.cpp:12-70
static void test_resample_series() {
  auto index = pd::date_range(pd::ns_from_ymd(2000, 1, 1), 9);
  auto series = pd::Series(pd::range(0L, 9L), index, "v");
  {
    auto resampler = pd::resample(series, pd::minutes(3));
    auto gi = resampler.index();
    REQUIRE(str_at(gi, 0) == "2000-01-01 00:00:00.000000000");
    REQUIRE(str_at(gi, 1) == "2000-01-01 00:03:00.000000000");
    REQUIRE(str_at(gi, 2) == "2000-01-01 00:06:00.000000000");
    auto sum = pd::ReturnOrThrowOnFailure(resampler.sum());
    REQUIRE(sum.at(0, 0) == int64_t(3));
    REQUIRE(sum.at(1, 0) == int64_t(12));
    REQUIRE(sum.at(2, 0) == int64_t(21));
  }
  {
    auto resampler = pd::resample(series, pd::minutes(3), false, true);
    auto gi = resampler.index();
    REQUIRE(str_at(gi, 0) == "2000-01-01 00:03:00.000000000");
    REQUIRE(str_at(gi, 2) == "2000-01-01 00:09:00.000000000");
    auto sum = pd::ReturnOrThrowOnFailure(resampler.sum());
    REQUIRE(sum.at(2, 0) == int64_t(21));
  }
  {
    auto resampler = pd::resample(series, pd::minutes(3), true, true);
    auto gi = resampler.index();
    REQUIRE(gi->length() == 4);
    REQUIRE(str_at(gi, 0) == "2000-01-01 00:00:00.000000000");
    REQUIRE(str_at(gi, 3) == "2000-01-01 00:09:00.000000000");
    auto sum = pd::ReturnOrThrowOnFailure(resampler.sum());
    REQUIRE(sum.at(0, 0) == int64_t(0));
    REQUIRE(sum.at(1, 0) == int64_t(6));
    REQUIRE(sum.at(2, 0) == int64_t(15));
    REQUIRE(sum.at(3, 0) == int64_t(15));
  }
  {
    auto sum = pd::ReturnOrThrowOnFailure(series.resample("3T").sum());      // string rule, series.cpp:351-359
    REQUIRE(sum.at(1, 0) == int64_t(12));
    REQUIRE_THROWS(pd::resample(series, pd::seconds(30)));                    // upsampling, resample.h:102-105
  }
}

// series_resample_test.cpp:87-130 — DataFrame::downsample
// pd::resample with DateOffset rules (resample.h:62-88 string rule -> makeGroupInfo's DateOffset branch,
// resample.cpp:248-267).  Expected values worked out by hand from the reference code; the same case is held to the
// oracle in tests/test_calendar_cpu.py::test_oracle_calendar_known_answer.
static void test_resample_calendar_rules() {
  // hourly ticks 2020-01-31 22:00 .. 2020-02-02 03:00 (30 of them), values 0..29
  auto index = pd::date_range(pd::ns_from_ymd(2020, 1, 31) + 22LL * 3600 * 1000000000LL, 30, pd::minutes(60));
  auto series = pd::Series(pd::range(0L, 30L), index, "v");
  {
    // "MS": binner 2019-12-01, 2020-01-01, 2020-02-01, 2020-03-01; bucket = (binner + 1 day - 1 ns]: the 26 ticks up to
    // 2020-02-01 23:00 carry the label 2020-01-01, the last 4 carry 2020-02-01; the empty first bucket does not appear
    auto resampler = pd::resample(series, "MS", true);
    auto gi = resampler.index();
    REQUIRE(gi->length() == 2);
    REQUIRE(str_at(gi, 0) == "2020-01-01 00:00:00.000000000");
    REQUIRE(str_at(gi, 1) == "2020-02-01 00:00:00.000000000");
    auto sum = pd::ReturnOrThrowOnFailure(resampler.sum());
    REQUIRE(sum.at(0, 0) == int64_t(25 * 26 / 2));
    REQUIRE(sum.at(1, 0) == int64_t(26 + 27 + 28 + 29));
    auto cnt = pd::ReturnOrThrowOnFailure(resampler.count());
    REQUIRE(cnt.at(0, 0) == int64_t(26));
  }
  {
    // "1D", label right: edges are the midnights themselves; a tick AT midnight closes the bucket that ends there
    auto resampler = pd::resample(series, pd::DateOffset{pd::DateOffset::Day, 1}, true, true);
    auto gi = resampler.index();
    REQUIRE(gi->length() == 3);
    REQUIRE(str_at(gi, 0) == "2020-02-01 00:00:00.000000000");      // ticks 22:00, 23:00, 00:00
    REQUIRE(str_at(gi, 2) == "2020-02-03 00:00:00.000000000");
    auto cnt = pd::ReturnOrThrowOnFailure(resampler.count());
    REQUIRE(cnt.at(0, 0) == int64_t(3));
    REQUIRE(cnt.at(1, 0) == int64_t(24));
    REQUIRE(cnt.at(2, 0) == int64_t(3));
  }
  REQUIRE_THROWS(pd::resample(series, "MS"));             // closed_left is not currently supported by DateOffset
  REQUIRE_THROWS(pd::resample(series, "M", true));        // MonthEnd not supported use arrow month().groupby()
  REQUIRE_THROWS(pd::resample(series, "bogus", true));
}

// SURVEY §8f rank 4: Series::sort / argsort (series.cpp:864-868,978-992), DataFrame::sort_index / sort_values
// (dataframe.cpp:1062-1071,1188-1208), readBinary / readParquet (:757-791, :646-683) and device-resident frames.
// Expected values: arrow's array_sort_indices / Take on the same data (the calls the reference makes).
static void test_sort_and_ingest() {
  auto idx = pd::date_range(pd::ns_from_ymd(2021, 3, 1), 8, pd::minutes(1));
  pd::DataFrame df(idx, std::pair{"k"s, std::vector<int64_t>{5, 3, 5, 1, 3, 9, 1, 5}},
                   std::pair{"v"s, std::vector<double>{1.5, 2.5, 3.5, 4.5, 5.5, 6.5, 7.5, 8.5}});
  {
    auto k = df["k"];
    auto order = k.argsort();
    arrow::compute::ArraySortOptions asc{arrow::compute::SortOrder::Ascending}, desc{arrow::compute::SortOrder::Descending};
    auto want = pd::ReturnOrThrowOnFailure(arrow::compute::CallFunction("array_sort_indices", {k.array()}, &asc)).make_array();
    REQUIRE(order.array()->Equals(want));                      // stable: 3, 6, 1, 4, 0, 2, 7, 5
    auto want_d = pd::ReturnOrThrowOnFailure(arrow::compute::CallFunction("array_sort_indices", {k.array()}, &desc)).make_array();
    REQUIRE(k.argsort(false).array()->Equals(want_d));
    auto sorted = k.sort();
    REQUIRE(sorted.array()->Equals(pd::ReturnOrThrowOnFailure(arrow::compute::Take(*k.array(), *want))));
    REQUIRE(sorted.indexArray()->Equals(pd::ReturnOrThrowOnFailure(arrow::compute::Take(*k.indexArray(), *want))));
    REQUIRE_THROWS(pd::Series(k.array(), nullptr).sort());     // "Cannot sort a Series without an index"
  }
  {
    // sort_index on a reversed frame restores time order in every column
    auto rev = pd::ReturnOrThrowOnFailure(arrow::compute::CallFunction("array_sort_indices", {idx},
                                          std::make_shared<arrow::compute::ArraySortOptions>(arrow::compute::SortOrder::Descending).get())).make_array();
    auto rb = pd::ReturnOrThrowOnFailure(arrow::compute::Take(arrow::Datum(df.array()), arrow::Datum(rev))).record_batch();
    pd::DataFrame shuffled(rb, pd::ReturnOrThrowOnFailure(arrow::compute::Take(*idx, *rev)));
    auto back = shuffled.sort_index();
    REQUIRE(back.indexArray()->Equals(idx));
    REQUIRE(back.array()->Equals(*df.array()));
    auto sv = df.sort_values({"k"});
    REQUIRE(sv["k"].values<int64_t>() == (std::vector<int64_t>{1, 1, 3, 3, 5, 5, 5, 9}));
    REQUIRE(sv["v"].values<double>() == df["v"].values<double>());          // other columns untouched (reference semantics)
    REQUIRE_THROWS(df.sort_values({"nope"}));
  }
  {
    // IPC stream blob -> readBinary(blob, index column)
    auto with_ts = pd::ReturnOrThrowOnFailure(df.array()->AddColumn(0, "ts", pd::ReturnOrThrowOnFailure(idx->View(arrow::int64()))));
    auto sink = pd::ReturnOrThrowOnFailure(arrow::io::BufferOutputStream::Create());
    auto writer = pd::ReturnOrThrowOnFailure(arrow::ipc::MakeStreamWriter(sink, with_ts->schema()));
    pd::ThrowOnFailure(writer->WriteRecordBatch(*with_ts));
    pd::ThrowOnFailure(writer->Close());
    auto buf = pd::ReturnOrThrowOnFailure(sink->Finish());
    auto read = pd::DataFrame::readBinary(std::basic_string_view<uint8_t>(buf->data(), static_cast<size_t>(buf->size())), "ts");
    REQUIRE(read.num_columns() == 2);
    REQUIRE(read.indexArray()->Equals(idx));                   // int64 index column cast to timestamp[ns]
    auto host_sum = pd::ReturnOrThrowOnFailure(read.group_by("k"s).sum("v"));
    // the same frame ingested once: group_by / aggregates / resample use the device copies
    auto dev = read.to_device();
    REQUIRE(dev.on_device());
    auto gb = dev.group_by("k"s);
    auto dev_sum = pd::ReturnOrThrowOnFailure(gb.sum("v"));
    REQUIRE(dev_sum.array()->Equals(host_sum.array()));
    REQUIRE(pd::ReturnOrThrowOnFailure(gb.mean("v")).array()->Equals(pd::ReturnOrThrowOnFailure(read.group_by("k"s).mean("v")).array()));
    auto r_dev = pd::ReturnOrThrowOnFailure(dev.resample("4T").sum());
    auto r_host = pd::ReturnOrThrowOnFailure(read.resample("4T").sum());
    REQUIRE(r_dev.array()->Equals(*r_host.array()));
    REQUIRE(dev["v"].sum().as<double>() == read["v"].sum().as<double>());
    REQUIRE(dev.sort_index(false).array()->Equals(*read.sort_index(false).array()));
  }
  {
    // Parquet file -> readParquet
    auto table = pd::ReturnOrThrowOnFailure(arrow::Table::FromRecordBatches({df.array()}));
    // a directory of our own: a fixed file name in the temp directory may belong to another user of the machine
    std::string dir = (std::filesystem::temp_directory_path() / "pa_b200_facade_XXXXXX").string();
    if (!mkdtemp(dir.data())) throw std::runtime_error("mkdtemp failed for " + dir);
    struct RemoveOnExit {   // also when a call below throws
      std::string dir;
      ~RemoveOnExit() { std::error_code ec; std::filesystem::remove_all(dir, ec); }
    } cleanup{dir};
    const std::string path = dir + "/facade_test.parquet";
    auto out = pd::ReturnOrThrowOnFailure(arrow::io::FileOutputStream::Open(path));
    pd::ThrowOnFailure(parquet::arrow::WriteTable(*table, arrow::default_memory_pool(), out, 1 << 20));
    pd::ThrowOnFailure(out->Close());
    auto pq = pd::DataFrame::readParquet(path);
    REQUIRE(pq.array()->Equals(*df.array()));
    auto s = pd::ReturnOrThrowOnFailure(pq.to_device().group_by("k"s).count("v"));
    REQUIRE(s.values<int64_t>() == (std::vector<int64_t>{3, 2, 2, 1}));
    REQUIRE_THROWS(pd::DataFrame::readParquet(dir + "/does_not_exist.parquet"));
  }
}

static void test_downsample() {
  auto index = pd::date_range(pd::ns_from_ymd(2000, 1, 1), 9);
  pd::DataFrame df(arrow::schema({arrow::field("i", arrow::int64())}), 9, {pd::range(0L, 9L)}, index);
  {
    auto resampler = df.downsample("3T", false);
    auto gi = resampler.index();
    auto sum = pd::ReturnOrThrowOnFailure(resampler.sum());
    REQUIRE(gi->length() == 3);
    REQUIRE(str_at(gi, 1) == "2000-01-01 00:03:00.000000000");
    REQUIRE(sum.at(0, 0) == int64_t(3));
    REQUIRE(sum.at(2, 0) == int64_t(21));
  }
  {
    auto resampler = df.downsample("3T", true);
    auto gi = resampler.index();
    auto sum = pd::ReturnOrThrowOnFailure(resampler.sum());
    REQUIRE(gi->length() == 4);
    REQUIRE(str_at(gi, 3) == "2000-01-01 00:09:00.000000000");
    REQUIRE(sum.at(0, 0) == int64_t(0));
    REQUIRE(sum.at(1, 0) == int64_t(6));
    REQUIRE(sum.at(3, 0) == int64_t(15));
  }
}

int main() {
  try {
    test_make_groups_and_aggregates();
    test_bardata();
    test_apply_sums();
    test_apply_callbacks_and_groups();
    test_second_stage_aggregates();
    test_resample_series();
    test_resample_calendar_rules();
    test_sort_and_ingest();
    test_downsample();
  } catch (std::exception const& e) {
    std::printf("EXCEPTION: %s\n", e.what());
    return 2;
  }
  std::printf("%d checks, %d failed\n", g_checks, g_fail);
  return g_fail ? 1 : 0;
}

// test_plugin_binary.cc — the contract of the drop-in subclass for the binary index types, in the shape of the reference's
// gtest suites (test/unit_test/vector/test_vector_index_binary_{flat,ivf_flat}.cc): status codes, NoData cases, topk 0,
// duplicate ids, the truncated range-search radius, filters, train-on-first-add and the HAMMING distance matrix.
// Needs a GPU; run by tests/test_gpu_binary_plugin_cpp.py.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <random>

#include "vector_index_b200.h"

using namespace dingodb;

static int g_fail = 0;
#define EXPECT(cond)                                                                \
  do {                                                                              \
    if (!(cond)) { ++g_fail; printf("FAIL %s:%d  %s\n", __FILE__, __LINE__, #cond); } \
  } while (0)

static std::vector<uint8_t> fixture(int n, int dim) {  // default-seeded std::mt19937 bytes
  std::mt19937 rng;
  std::vector<uint8_t> x((size_t)n * dim / 8);
  for (auto& b : x) b = (uint8_t)(rng() & 0xFF);
  return x;
}
static int hamming(const uint8_t* a, const uint8_t* b, int dim) {
  int d = 0;
  for (int i = 0; i < dim / 8; ++i) d += __builtin_popcount((unsigned)(a[i] ^ b[i]));
  return d;
}
static pb::common::VectorWithId row(const uint8_t* x, int dim, int64_t id) {
  pb::common::VectorWithId v;
  v.set_id(id);
  v.mutable_vector()->set_dimension(dim);
  v.mutable_vector()->set_value_type(pb::common::ValueType::UINT8);
  for (int j = 0; j < dim / 8; ++j) v.mutable_vector()->add_binary_values(std::string(1, (char)x[j]));
  return v;
}
static std::vector<pb::common::VectorWithId> to_pb(const std::vector<uint8_t>& x, int n, int dim, int64_t first_id) {
  std::vector<pb::common::VectorWithId> out;
  for (int i = 0; i < n; ++i) out.push_back(row(x.data() + (size_t)i * dim / 8, dim, first_id + i));
  return out;
}
static std::shared_ptr<VectorIndexB200> make(pb::common::VectorIndexType t, int dim, int nlist = 0,
                                             pb::common::MetricType m = pb::common::METRIC_TYPE_HAMMING) {
  pb::common::VectorIndexParameter p;
  p.set_vector_index_type(t);
  if (t == pb::common::VECTOR_INDEX_TYPE_BINARY_FLAT) { auto* q = p.mutable_binary_flat_parameter(); q->dimension_ = dim; q->metric_type_ = m; }
  if (t == pb::common::VECTOR_INDEX_TYPE_BINARY_IVF_FLAT) {
    auto* q = p.mutable_binary_ivf_flat_parameter(); q->dimension_ = dim; q->metric_type_ = m; q->ncentroids_ = nlist;
  }
  return std::make_shared<VectorIndexB200>(1, p, pb::common::RegionEpoch(), pb::common::Range(), nullptr);
}
static bool created(const std::shared_ptr<VectorIndexB200>& ix) { int64_t c = 0; return ix->GetCount(c).ok(); }

// the result contract shared by both types: one entry per query, UINT8 rows, HAMMING, ascending integer distances that
// equal a host recomputation, hits inside the id filter
static void check_results(const std::vector<pb::index::VectorWithDistanceResult>& results, const std::vector<uint8_t>& x, int dim,
                          int64_t first_id, const std::vector<uint8_t>& q, int nq, int64_t lo = INT64_MIN, int64_t hi = INT64_MAX) {
  EXPECT((int)results.size() == nq);
  for (int r = 0; r < (int)results.size(); ++r) {
    float prev = -1;
    for (const auto& h : results[r].vector_with_distances()) {
      const int64_t id = h.vector_with_id().id();
      EXPECT(id >= lo && id < hi);
      EXPECT(h.vector_with_id().vector().value_type() == pb::common::ValueType::UINT8);
      EXPECT(h.vector_with_id().vector().dimension() == dim);
      EXPECT(h.metric_type() == pb::common::METRIC_TYPE_HAMMING);
      EXPECT(h.distance() >= prev);
      prev = h.distance();
      EXPECT(h.distance() == (float)hamming(q.data() + (size_t)r * dim / 8, x.data() + (size_t)(id - first_id) * dim / 8, dim));
    }
  }
}

static void test_create() {
  EXPECT(created(make(pb::common::VECTOR_INDEX_TYPE_BINARY_FLAT, 64)));
  EXPECT(created(make(pb::common::VECTOR_INDEX_TYPE_BINARY_IVF_FLAT, 64, 0)));  // ncentroids 0 -> 2048
  EXPECT(!created(make(pb::common::VECTOR_INDEX_TYPE_BINARY_FLAT, 64, 0, pb::common::METRIC_TYPE_L2)));
  EXPECT(!created(make(pb::common::VECTOR_INDEX_TYPE_BINARY_FLAT, 12)));
  EXPECT(!created(make(pb::common::VECTOR_INDEX_TYPE_BINARY_IVF_FLAT, 0, 10)));
}

static void test_binary_flat() {
  const int n = 1000, dim = 64;
  auto x = fixture(n, dim);
  auto vs = to_pb(x, n, dim, 1);
  auto ix = make(pb::common::VECTOR_INDEX_TYPE_BINARY_FLAT, dim);
  if (!created(ix)) { printf("cannot create the index: %s\n", b200vs_last_error()); exit(2); }
  std::vector<pb::index::VectorWithDistanceResult> results;
  pb::common::VectorSearchParameter sp;
  EXPECT(!ix->NeedTrain() && ix->IsTrained());
  std::vector<uint8_t> none;
  EXPECT(ix->Train(none).ok());  // Flat: no-op
  // empty add / search -> EILLEGAL_PARAMTETERS
  EXPECT(ix->Add({}).error_code() == pb::error::EILLEGAL_PARAMTETERS);
  EXPECT(ix->Search({}, 3, {}, false, sp, results).error_code() == pb::error::EILLEGAL_PARAMTETERS);
  // NoData: search of an empty index -> OK, one empty result per query
  EXPECT(ix->Search({vs[0]}, 3, {}, false, sp, results).ok() && results.size() == 1 && results[0].vector_with_distances_size() == 0);
  // wrong byte count, wrong dimension field, float rows -> EVECTOR_INVALID
  auto bad = vs[0];
  bad.mutable_vector()->add_binary_values(std::string(1, 'x'));
  EXPECT(ix->Add({bad}).error_code() == pb::error::EVECTOR_INVALID);
  bad = vs[0];
  bad.mutable_vector()->set_dimension(dim - 8);
  EXPECT(ix->Add({bad}).error_code() == pb::error::EVECTOR_INVALID);
  bad = vs[0];
  bad.mutable_vector()->set_value_type(pb::common::ValueType::FLOAT);
  EXPECT(ix->Add({bad}).error_code() == pb::error::EVECTOR_INVALID);
  results.clear();
  EXPECT(ix->Search({bad}, 3, {}, false, sp, results).error_code() == pb::error::EVECTOR_INVALID);
  // duplicate ids in one batch -> EVECTOR_ID_DUPLICATED
  EXPECT(ix->Add({vs[0], vs[0]}).error_code() == pb::error::EVECTOR_ID_DUPLICATED);
  EXPECT(ix->Add(vs).ok());
  int64_t c = -1;
  EXPECT(ix->GetCount(c).ok() && c == n);
  // topk 0 -> OK, nothing appended
  results.clear();
  EXPECT(ix->Search({vs[3]}, 0, {}, false, sp, results).ok() && results.empty());
  // self match at rank 0, distance 0
  std::vector<uint8_t> q(x.begin(), x.begin() + 5 * dim / 8);
  results.clear();
  EXPECT(ix->Search({vs[0], vs[1], vs[2], vs[3], vs[4]}, 10, {}, false, sp, results).ok());
  for (int r = 0; r < 5 && r < (int)results.size(); ++r)
    EXPECT(results[r].vector_with_distances_size() == 10 && results[r].vector_with_distances(0).vector_with_id().id() == r + 1 &&
           results[r].vector_with_distances(0).distance() == 0.f);
  check_results(results, x, dim, 1, q, 5);
  // range filter and id-list filter (and its negation)
  results.clear();
  std::vector<std::shared_ptr<VectorIndex::FilterFunctor>> filt{std::make_shared<VectorIndex::RangeFilterFunctor>(100, 300)};
  EXPECT(ix->Search({vs[0], vs[1], vs[2], vs[3], vs[4]}, 20, filt, false, sp, results).ok());
  check_results(results, x, dim, 1, q, 5, 100, 300);
  std::vector<int64_t> allow{7, 9, 11, 500};
  results.clear();
  filt = {std::make_shared<VectorIndex::SortFilterFunctor>(allow)};
  EXPECT(ix->Search({vs[0]}, 10, filt, false, sp, results).ok() && results[0].vector_with_distances_size() == 4);
  // range search: the radius is truncated to int, hits have distance < 10
  results.clear();
  EXPECT(ix->RangeSearch({vs[0], vs[1], vs[2], vs[3], vs[4]}, 10.1f, {}, false, sp, results).ok());
  check_results(results, x, dim, 1, q, 5);
  for (int r = 0; r < (int)results.size(); ++r) {
    int expect = 0;
    for (int i = 0; i < n; ++i) expect += hamming(q.data() + (size_t)r * dim / 8, x.data() + (size_t)i * dim / 8, dim) < 10;
    EXPECT(results[r].vector_with_distances_size() == expect);
    for (const auto& h : results[r].vector_with_distances()) EXPECT(h.distance() < 10.f);
  }
  // delete (unknown ids ignored), upsert replaces
  EXPECT(ix->Delete({1, 2, 3, 100000}).ok());
  EXPECT(ix->GetCount(c).ok() && c == n - 3);
  auto up = row(x.data() + 10 * dim / 8, dim, 5);  // id 5 now holds row 10's bits
  EXPECT(ix->Upsert({up}).ok());
  EXPECT(ix->GetCount(c).ok() && c == n - 3);
  results.clear();
  EXPECT(ix->Search({vs[10]}, 2, {}, false, sp, results).ok());
  if (!results.empty() && results[0].vector_with_distances_size() == 2) {
    EXPECT(results[0].vector_with_distances(0).vector_with_id().id() == 5);  // (distance 0, id 5) before (0, 11)
    EXPECT(results[0].vector_with_distances(1).vector_with_id().id() == 11);
  }
}

static void test_binary_ivf_flat() {
  const int n = 2000, dim = 128, nlist = 10;
  auto x = fixture(n, dim);
  auto vs = to_pb(x, n, dim, 1);
  auto ix = make(pb::common::VECTOR_INDEX_TYPE_BINARY_IVF_FLAT, dim, nlist);
  std::vector<pb::index::VectorWithDistanceResult> results;
  pb::common::VectorSearchParameter sp;
  EXPECT(ix->NeedTrain() && !ix->IsTrained());
  // untrained: search -> OK with empty results, delete -> OK
  EXPECT(ix->Search({vs[0]}, 3, {}, false, sp, results).ok() && results.size() == 1 && results[0].vector_with_distances_size() == 0);
  EXPECT(ix->Delete({1, 2}).ok());
  // Train(uint8): no data / ragged data -> EILLEGAL_PARAMTETERS
  std::vector<uint8_t> empty, ragged(dim / 8 + 1, 0);
  EXPECT(ix->Train(empty).error_code() == pb::error::EILLEGAL_PARAMTETERS);
  EXPECT(ix->Train(ragged).error_code() == pb::error::EILLEGAL_PARAMTETERS);
  // the first Add trains on its own batch and retries (ivf_flat.cc:133-150)
  EXPECT(ix->Add(vs).ok());
  EXPECT(ix->IsTrained());
  int64_t c = -1;
  EXPECT(ix->GetCount(c).ok() && c == n);
  // delete of unknown ids -> EVECTOR_INVALID
  EXPECT(ix->Delete({100000}).error_code() == pb::error::EVECTOR_INVALID);
  // nprobe comes from binary_ivf_flat(): all lists probed = exact answer, self match at rank 0
  sp.mutable_binary_ivf_flat()->set_nprobe(nlist);
  std::vector<uint8_t> q(x.begin(), x.begin() + 4 * dim / 8);
  results.clear();
  EXPECT(ix->Search({vs[0], vs[1], vs[2], vs[3]}, 10, {}, false, sp, results).ok());
  check_results(results, x, dim, 1, q, 4);
  for (int r = 0; r < 4 && r < (int)results.size(); ++r)
    EXPECT(results[r].vector_with_distances_size() == 10 && results[r].vector_with_distances(0).vector_with_id().id() == r + 1);
  results.clear();
  EXPECT(ix->Search({vs[0]}, 0, {}, false, sp, results).ok() && results.empty());
  results.clear();
  std::vector<std::shared_ptr<VectorIndex::FilterFunctor>> filt{std::make_shared<VectorIndex::RangeFilterFunctor>(500, 900)};
  EXPECT(ix->Search({vs[0], vs[1], vs[2], vs[3]}, 10, filt, false, sp, results).ok());
  check_results(results, x, dim, 1, q, 4, 500, 900);
  results.clear();
  EXPECT(ix->RangeSearch({vs[0], vs[1], vs[2], vs[3]}, 50.7f, {}, false, sp, results).ok());
  check_results(results, x, dim, 1, q, 4);
  for (int r = 0; r < (int)results.size(); ++r) {
    int expect = 0;
    for (int i = 0; i < n; ++i) expect += hamming(q.data() + (size_t)r * dim / 8, x.data() + (size_t)i * dim / 8, dim) < 50;
    EXPECT(results[r].vector_with_distances_size() == expect);
  }
  // fewer training rows than ncentroids: nlist degenerates to 1 and the index still serves
  auto iy = make(pb::common::VECTOR_INDEX_TYPE_BINARY_IVF_FLAT, dim, nlist);
  std::vector<uint8_t> few(x.begin(), x.begin() + (size_t)(nlist - 1) * dim / 8);
  EXPECT(iy->Train(few).ok() && iy->IsTrained());
  EXPECT(iy->Add(vs).ok());
  results.clear();
  EXPECT(iy->Search({vs[7]}, 1, {}, false, pb::common::VectorSearchParameter(), results).ok() &&
         results[0].vector_with_distances_size() == 1 && results[0].vector_with_distances(0).vector_with_id().id() == 8);
}

static void test_calc_distance() {
  auto x = fixture(5, 64);
  std::vector<pb::common::Vector> left, right;
  for (int i = 0; i < 2; ++i) left.push_back(row(x.data() + i * 8, 64, i).vector());
  for (int i = 0; i < 5; ++i) right.push_back(row(x.data() + i * 8, 64, i).vector());
  std::vector<std::vector<float>> d;
  std::vector<pb::common::Vector> lo, ro;
  EXPECT(VectorIndexB200Utils::CalcDistance(B200VS_ALGORITHM_FAISS, pb::common::METRIC_TYPE_HAMMING, left, right, true, d, lo, ro).ok());
  EXPECT(d.size() == 2 && d[0].size() == 5);
  for (int i = 0; i < 2 && i < (int)d.size(); ++i)
    for (int j = 0; j < 5 && j < (int)d[i].size(); ++j) EXPECT(d[i][j] == (float)hamming(x.data() + i * 8, x.data() + j * 8, 64));
  EXPECT(lo.size() == 2 && lo[0].dimension() == 64 && lo[0].value_type() == pb::common::ValueType::UINT8 && ro.size() == 5);
  EXPECT(VectorIndexB200Utils::CalcDistance(0, pb::common::METRIC_TYPE_HAMMING, left, right, false, d, lo, ro).error_code() ==
         pb::error::EILLEGAL_PARAMTETERS);
}

int main() {
  test_create();
  test_binary_flat();
  test_binary_ivf_flat();
  test_calc_distance();
  if (g_fail) { printf("%d BINARY PLUGIN CHECKS FAILED\n", g_fail); return 1; }
  printf("BINARY PLUGIN TESTS OK\n");
  return 0;
}

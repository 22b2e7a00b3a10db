// vector_index_b200.cc — see vector_index_b200.h.
#include "vector_index_b200.h"

#include <algorithm>
#include <cstdint>
#include <cstring>
#include <string>
#include <unordered_set>

namespace dingodb {

int32_t VectorIndexB200::max_range_search_result_count = 1024;

namespace {

// CheckVectorDimension, src/vector/vector_index_utils.cc:502-530, plus ExtractVectorValue's value-type check (:563-600):
// float indexes take FLOAT rows of `dimension` values, binary indexes UINT8 rows of dimension / 8 bytes
butil::Status CheckVectorDimension(const std::vector<pb::common::VectorWithId>& vs, int dimension, bool binary = false) {
  const pb::common::ValueType want = binary ? pb::common::ValueType::UINT8 : pb::common::ValueType::FLOAT;
  for (const auto& v : vs) {
    if (v.vector().value_type() != want)
      return butil::Status(pb::error::Errno::EVECTOR_INVALID, "invalid value type");
    if (!binary && (int)v.vector().float_values().size() != dimension)
      return butil::Status(pb::error::Errno::EVECTOR_INVALID, "vector dimension not match, " + std::to_string(v.vector().float_values_size()) + " " + std::to_string(dimension));
    if (binary && (int)v.vector().binary_values().size() != dimension / 8)
      return butil::Status(pb::error::Errno::EVECTOR_INVALID, "binary vector dimension not match, " + std::to_string(v.vector().binary_values_size()) + " " + std::to_string(dimension) + "/bit");
    if (v.vector().dimension() != dimension)
      return butil::Status(pb::error::Errno::EVECTOR_INVALID, "vector dimension not match, " + std::to_string(v.vector().dimension()) + " " + std::to_string(dimension));
  }
  return butil::Status::OK();
}

// ExtractVectorValue<float> (memcpy into one row-major array; normalisation happens on the device), utils.cc:563-609
std::vector<float> ExtractVectorValue(const std::vector<pb::common::VectorWithId>& vs, int dimension) {
  std::vector<float> out(vs.size() * (size_t)dimension);
  for (size_t i = 0; i < vs.size(); ++i) memcpy(out.data() + i * dimension, vs[i].vector().float_values().data(), (size_t)dimension * sizeof(float));
  return out;
}

// ExtractVectorValue<uint8_t>: each binary_values element is one byte, read as val[0] (utils.cc:590-600)
std::vector<uint8_t> ExtractBinaryValue(const std::vector<pb::common::VectorWithId>& vs, int dimension) {
  const size_t code = (size_t)dimension / 8;
  std::vector<uint8_t> out(vs.size() * code);
  for (size_t i = 0; i < vs.size(); ++i) {
    const auto& b = vs[i].vector().binary_values();
    for (size_t j = 0; j < code; ++j) out[i * code + j] = b[j].empty() ? 0 : static_cast<uint8_t>(b[j][0]);
  }
  return out;
}

struct LoweredFilters {
  b200vs_search_params sp;
  std::vector<int64_t> ids;  // keeps sorted_ids alive
};

}  // namespace

VectorIndexB200::VectorIndexB200(int64_t id, const pb::common::VectorIndexParameter& p, const pb::common::RegionEpoch& epoch,
                                 const pb::common::Range& range, ThreadPoolPtr thread_pool, int device)
    : VectorIndex(id, p, epoch, range, std::move(thread_pool)) {
  b200vs_params bp;
  memset(&bp, 0, sizeof(bp));
  bp.device = device;
  b200vs_type type = B200VS_FLAT;
  switch (p.vector_index_type()) {
    case pb::common::VECTOR_INDEX_TYPE_FLAT:
      type = B200VS_FLAT; dimension_ = p.flat_parameter().dimension(); metric_type_ = p.flat_parameter().metric_type(); break;
    case pb::common::VECTOR_INDEX_TYPE_IVF_FLAT:
      type = B200VS_IVF_FLAT; dimension_ = p.ivf_flat_parameter().dimension(); metric_type_ = p.ivf_flat_parameter().metric_type();
      bp.nlist = p.ivf_flat_parameter().ncentroids(); break;
    case pb::common::VECTOR_INDEX_TYPE_IVF_PQ:
      type = B200VS_IVF_PQ; dimension_ = p.ivf_pq_parameter().dimension(); metric_type_ = p.ivf_pq_parameter().metric_type();
      bp.nlist = p.ivf_pq_parameter().ncentroids(); bp.pq_m = p.ivf_pq_parameter().nsubvector(); bp.pq_nbits = p.ivf_pq_parameter().nbits_per_idx(); break;
    case pb::common::VECTOR_INDEX_TYPE_HNSW:
      type = B200VS_HNSW; dimension_ = p.hnsw_parameter().dimension(); metric_type_ = p.hnsw_parameter().metric_type();
      bp.hnsw_m = p.hnsw_parameter().nlinks(); bp.hnsw_efc = p.hnsw_parameter().efconstruction(); bp.max_elements = p.hnsw_parameter().max_elements(); break;
    case pb::common::VECTOR_INDEX_TYPE_BINARY_FLAT:  // factory.cc:73-76
      type = B200VS_BINARY_FLAT; dimension_ = p.binary_flat_parameter().dimension(); metric_type_ = p.binary_flat_parameter().metric_type();
      binary_ = true; break;
    case pb::common::VECTOR_INDEX_TYPE_BINARY_IVF_FLAT:  // factory.cc:77-80
      type = B200VS_BINARY_IVF_FLAT; dimension_ = p.binary_ivf_flat_parameter().dimension(); metric_type_ = p.binary_ivf_flat_parameter().metric_type();
      bp.nlist = p.binary_ivf_flat_parameter().ncentroids(); binary_ = true; break;
    default: break;
  }
  // "not support metric type, use L2" — flat.cc:91-96.  Binary types need HAMMING; any other metric fails the create.
  b200vs_metric m = metric_type_ == pb::common::METRIC_TYPE_INNER_PRODUCT ? B200VS_IP : metric_type_ == pb::common::METRIC_TYPE_COSINE ? B200VS_COSINE : B200VS_L2;
  if (metric_type_ == pb::common::METRIC_TYPE_HAMMING) m = B200VS_HAMMING;
  b200vs_create(type, m, dimension_, &bp, &index_);  // a failed create leaves index_ null: every call then returns EINTERNAL
}

VectorIndexB200::~VectorIndexB200() { b200vs_destroy(index_); }

butil::Status VectorIndexB200::ToStatus(int rc) const {
  if (rc == B200VS_OK) return butil::Status::OK();
  pb::error::Errno e = pb::error::EINTERNAL;
  switch (rc) {
    case B200VS_EILLEGAL_PARAMETERS: e = pb::error::EILLEGAL_PARAMTETERS; break;
    case B200VS_EVECTOR_INVALID: e = pb::error::EVECTOR_INVALID; break;
    case B200VS_EVECTOR_NOT_TRAIN: e = pb::error::EVECTOR_NOT_TRAIN; break;
    case B200VS_EVECTOR_NOT_SUPPORT: e = pb::error::EVECTOR_NOT_SUPPORT; break;
    case B200VS_EVECTOR_ID_DUPLICATED: e = pb::error::EVECTOR_ID_DUPLICATED; break;
    default: break;
  }
  return butil::Status(e, b200vs_last_error());
}

butil::Status VectorIndexB200::GetCount(int64_t& count) { return ToStatus(index_ ? b200vs_count(index_, &count) : B200VS_EINTERNAL); }
butil::Status VectorIndexB200::GetDeletedCount(int64_t& c) { return ToStatus(index_ ? b200vs_deleted_count(index_, &c) : B200VS_EINTERNAL); }
butil::Status VectorIndexB200::GetMemorySize(int64_t& m) { return ToStatus(index_ ? b200vs_memory_size(index_, &m) : B200VS_EINTERNAL); }

bool VectorIndexB200::IsExceedsMaxElements(int64_t vector_size) {  // hnsw.cc:540-550; faiss types: never
  if (vector_index_type != pb::common::VECTOR_INDEX_TYPE_HNSW) return false;
  // hnswlib's cur_element_count includes tombstoned nodes (markDelete frees nothing) and so does the library's own
  // capacity check: gate on live + deleted so the service never admits a write the index then rejects
  int64_t count = 0, deleted = 0;
  if (!index_ || b200vs_count(index_, &count) != B200VS_OK || b200vs_deleted_count(index_, &deleted) != B200VS_OK) return true;
  return count + deleted + vector_size > vector_index_parameter.hnsw_parameter().max_elements();
}

butil::Status VectorIndexB200::AddOrUpsert(const std::vector<pb::common::VectorWithId>& vs, bool is_upsert) {
  if (vs.empty()) return butil::Status(pb::error::EILLEGAL_PARAMTETERS, "vector_with_ids is empty");  // flat.cc:123-125
  auto status = CheckVectorDimension(vs, dimension_, binary_);
  if (!status.ok()) return status;
  if (!index_) return ToStatus(B200VS_EINTERNAL);
  std::vector<int64_t> ids(vs.size());
  for (size_t i = 0; i < vs.size(); ++i) ids[i] = vs[i].id();
  std::vector<float> x;
  std::vector<uint8_t> xb;
  if (binary_) xb = ExtractBinaryValue(vs, dimension_);
  else x = ExtractVectorValue(vs, dimension_);
  auto add = [&]() {
    return binary_ ? b200vs_add_binary_with_ids(index_, (int64_t)vs.size(), xb.data(), ids.data(), is_upsert ? 1 : 0)
                   : b200vs_add_with_ids(index_, (int64_t)vs.size(), x.data(), ids.data(), is_upsert ? 1 : 0);
  };
  std::shared_lock<std::shared_mutex> gate(write_gate_);
  int rc = add();
  if (rc == B200VS_EVECTOR_NOT_TRAIN) {  // "train with this batch and try again", ivf_flat.cc:133-150
    status = Train(vs);
    if (!status.ok()) return status;
    rc = add();
  }
  return ToStatus(rc);
}
butil::Status VectorIndexB200::Add(const std::vector<pb::common::VectorWithId>& vs) { return AddOrUpsert(vs, false); }
butil::Status VectorIndexB200::Upsert(const std::vector<pb::common::VectorWithId>& vs) { return AddOrUpsert(vs, true); }

butil::Status VectorIndexB200::Delete(const std::vector<int64_t>& delete_ids) {
  if (delete_ids.empty()) return butil::Status::OK();  // flat.cc:172-174
  if (!index_) return ToStatus(B200VS_EINTERNAL);
  std::shared_lock<std::shared_mutex> gate(write_gate_);
  int64_t removed = 0;
  return ToStatus(b200vs_remove_ids(index_, (int64_t)delete_ids.size(), delete_ids.data(), &removed));
}

butil::Status VectorIndexB200::Save(const std::string& path) { return ToStatus(index_ ? b200vs_save(index_, path.c_str()) : B200VS_EINTERNAL); }
butil::Status VectorIndexB200::Load(const std::string& path) { return ToStatus(index_ ? b200vs_load(index_, path.c_str()) : B200VS_EINTERNAL); }

// Lower the reference's host-side functors (vector_index.h:67-146) to the device form.  RangeFilterFunctor and
// SortFilterFunctor — the only two ever constructed in src/ (vector_index.cc:1342, vector_reader.cc:1777) — map
// directly; any other functor is evaluated over the index's ids on the host into a sorted allow-list.
static butil::Status LowerFilters(b200vs_index* index, const std::vector<std::shared_ptr<VectorIndex::FilterFunctor>>& filters,
                                  LoweredFilters& out) {
  memset(&out.sp, 0, sizeof(out.sp));
  bool have_list = false;
  std::vector<VectorIndex::FilterFunctor*> generic;
  for (const auto& f : filters) {
    if (!f) continue;
    if (auto* r = dynamic_cast<VectorIndex::RangeFilterFunctor*>(f.get())) {
      const int64_t lo = r->MinVectorId(), hi = r->MaxVectorId();
      if (!out.sp.has_range) { out.sp.has_range = 1; out.sp.range_min = lo; out.sp.range_max = hi; }
      else { out.sp.range_min = std::max<int64_t>(out.sp.range_min, lo); out.sp.range_max = std::min<int64_t>(out.sp.range_max, hi); }
    } else if (auto* s = dynamic_cast<VectorIndex::SortFilterFunctor*>(f.get()); s && !have_list) {
      out.ids = s->VectorIds();
      out.sp.negate = s->IsNegation() ? 1 : 0;
      have_list = true;
    } else {
      generic.push_back(f.get());
    }
  }
  if (!generic.empty()) {  // generic fallback: Check() over every id held by the index
    int64_t n = 0;
    if (b200vs_count(index, &n) != B200VS_OK) return butil::Status(pb::error::EINTERNAL, b200vs_last_error());
    std::vector<int64_t> all((size_t)n);
    if (n && b200vs_export_lists(index, nullptr, nullptr, nullptr, all.data()) != B200VS_OK) return butil::Status(pb::error::EINTERNAL, b200vs_last_error());
    std::vector<int64_t> allow;
    for (int64_t id : all) {
      bool ok = true;
      for (auto* g : generic) ok = ok && g->Check(id);
      if (ok && have_list) { const bool in = std::binary_search(out.ids.begin(), out.ids.end(), id); ok = out.sp.negate ? !in : in; }
      if (ok) allow.push_back(id);
    }
    std::sort(allow.begin(), allow.end());
    out.ids.swap(allow);
    out.sp.negate = 0;
    have_list = true;
  }
  if (have_list) { out.sp.sorted_ids = out.ids.data(); out.sp.n_ids = (int64_t)out.ids.size(); }
  return butil::Status::OK();
}

butil::Status VectorIndexB200::Search(const std::vector<pb::common::VectorWithId>& vs, uint32_t topk,
                                      const std::vector<std::shared_ptr<FilterFunctor>>& filters, bool reconstruct,
                                      const pb::common::VectorSearchParameter& parameter,
                                      std::vector<pb::index::VectorWithDistanceResult>& results) {
  if (vs.empty()) return butil::Status(pb::error::EILLEGAL_PARAMTETERS, "vector_with_ids is empty");  // flat.cc:208-210
  if (topk <= 0) return butil::Status::OK();                                                            // flat.cc:212
  if (vector_index_type == pb::common::VECTOR_INDEX_TYPE_HNSW &&
      (parameter.hnsw().efsearch() < 0 || parameter.hnsw().efsearch() > 1024))                           // hnsw.cc:332-336
    return butil::Status(pb::error::EILLEGAL_PARAMTETERS, "efsearch is illegal, " + std::to_string(parameter.hnsw().efsearch()) + ", must between 0 and 1024");
  auto status = CheckVectorDimension(vs, dimension_, binary_);
  if (!status.ok()) return status;
  if (!index_) return ToStatus(B200VS_EINTERNAL);
  LoweredFilters lf;
  status = LowerFilters(index_, filters, lf);
  if (!status.ok()) return status;
  lf.sp.nprobe = SearchNprobe(parameter);
  lf.sp.efsearch = parameter.hnsw().efsearch();
  std::vector<float> distances((size_t)topk * vs.size(), 0.0f);
  std::vector<int64_t> labels((size_t)topk * vs.size(), -1);  // flat.cc:218-219
  int rc;
  if (binary_) {
    const std::vector<uint8_t> xb = ExtractBinaryValue(vs, dimension_);
    rc = b200vs_search_binary(index_, (int64_t)vs.size(), xb.data(), (int32_t)topk, &lf.sp, distances.data(), labels.data());
  } else {
    const std::vector<float> x = ExtractVectorValue(vs, dimension_);
    rc = b200vs_search(index_, (int64_t)vs.size(), x.data(), (int32_t)topk, &lf.sp, distances.data(), labels.data());
  }
  if (rc != B200VS_OK) return ToStatus(rc);
  // reconstruct: only the HNSW plugin honours it, and never for cosine (hnsw.cc:383-395, :469-472 "force reconstruct false");
  // the faiss plugins ignore the flag (flat.cc:205, ivf_flat.cc:191)
  std::vector<float> stored;
  std::vector<uint8_t> found;
  if (reconstruct && vector_index_type == pb::common::VECTOR_INDEX_TYPE_HNSW && metric_type_ != pb::common::METRIC_TYPE_COSINE) {
    stored.resize(labels.size() * (size_t)dimension_);
    found.assign(labels.size(), 0);
    std::vector<int64_t> ask(labels);
    for (auto& l : ask) if (l < 0) l = INT64_MIN;  // never a stored id
    const int rrc = b200vs_reconstruct(index_, (int64_t)ask.size(), ask.data(), stored.data(), found.data());
    if (rrc != B200VS_OK) return ToStatus(rrc);
  }
  // FillSearchResult, utils.cc:611-655: one result per query appended; label < 0 skipped; distances arrive in API semantics
  // (HAMMING: float of the integer distance, value type UINT8, :640-648)
  for (size_t row = 0; row < vs.size(); ++row) {
    auto& result = results.emplace_back();
    for (size_t i = 0; i < topk; ++i) {
      const size_t pos = row * topk + i;
      if (labels[pos] < 0) continue;
      auto* vwd = result.add_vector_with_distances();
      auto* vwi = vwd->mutable_vector_with_id();
      vwi->set_id(labels[pos]);
      vwi->mutable_vector()->set_dimension(dimension_);
      vwi->mutable_vector()->set_value_type(binary_ ? pb::common::ValueType::UINT8 : pb::common::ValueType::FLOAT);
      if (!found.empty()) {
        if (!found[pos]) return butil::Status(pb::error::EINTERNAL, "getDataByLabel failed, label: " + std::to_string(labels[pos]));  // hnsw.cc:389-394
        for (int32_t j = 0; j < dimension_; ++j) vwi->mutable_vector()->add_float_values(stored[pos * (size_t)dimension_ + j]);
      }
      vwd->set_distance(distances[pos]);
      vwd->set_metric_type(metric_type_);
    }
  }
  return butil::Status::OK();
}

// VectorIndexIvfPq::VectorIndexSubType (vector_index_ivf_pq.cc:474): FLAT while the inner Flat index serves, IVF_PQ after.
pb::common::VectorIndexType VectorIndexB200::VectorIndexSubType() {
  if (vector_index_type != pb::common::VECTOR_INDEX_TYPE_IVF_PQ || !index_) return pb::common::VECTOR_INDEX_TYPE_NONE;  // base default, vector_index.h:238
  switch (b200vs_sub_type(index_)) {
    case B200VS_FLAT: return pb::common::VECTOR_INDEX_TYPE_FLAT;
    case B200VS_IVF_PQ: return pb::common::VECTOR_INDEX_TYPE_IVF_PQ;
    default: return pb::common::VECTOR_INDEX_TYPE_NONE;
  }
}

butil::Status VectorIndexB200::RangeSearch(const std::vector<pb::common::VectorWithId>& vs, float radius,
                                           const std::vector<std::shared_ptr<FilterFunctor>>& filters, bool /*reconstruct*/,
                                           const pb::common::VectorSearchParameter& parameter,
                                           std::vector<pb::index::VectorWithDistanceResult>& results) {
  if (vector_index_type == pb::common::VECTOR_INDEX_TYPE_HNSW)
    return butil::Status(pb::error::Errno::EVECTOR_NOT_SUPPORT, "RangeSearch not support in Hnsw!!!");  // hnsw.cc:487-493
  if (vs.empty()) return butil::Status(pb::error::EILLEGAL_PARAMTETERS, "vector_with_ids is empty");   // flat.cc:271-273
  auto status = CheckVectorDimension(vs, dimension_, binary_);
  if (!status.ok()) return status;
  if (!index_) return ToStatus(B200VS_EINTERNAL);
  LoweredFilters lf;
  status = LowerFilters(index_, filters, lf);
  if (!status.ok()) return status;
  lf.sp.nprobe = SearchNprobe(parameter);
  const int32_t cap = max_range_search_result_count;
  std::vector<float> distances((size_t)cap * vs.size());
  std::vector<int64_t> labels((size_t)cap * vs.size());
  std::vector<int32_t> counts(vs.size());
  int rc;
  if (binary_) {  // the radius is truncated to int inside (faiss binary range_search, flat.cc:282-311)
    const std::vector<uint8_t> xb = ExtractBinaryValue(vs, dimension_);
    rc = b200vs_range_search_binary(index_, (int64_t)vs.size(), xb.data(), radius, cap, &lf.sp, distances.data(), labels.data(), counts.data());
  } else {
    const std::vector<float> x = ExtractVectorValue(vs, dimension_);
    rc = b200vs_range_search(index_, (int64_t)vs.size(), x.data(), radius, cap, &lf.sp, distances.data(), labels.data(), counts.data());
  }
  if (rc != B200VS_OK) return ToStatus(rc);
  for (size_t row = 0; row < vs.size(); ++row) {  // FillRangeSearchResult, utils.cc:657-700
    auto& result = results.emplace_back();
    for (int32_t i = 0; i < counts[row]; ++i) {
      const size_t pos = row * cap + i;
      auto* vwd = result.add_vector_with_distances();
      auto* vwi = vwd->mutable_vector_with_id();
      vwi->set_id(labels[pos]);
      vwi->mutable_vector()->set_dimension(dimension_);
      vwi->mutable_vector()->set_value_type(binary_ ? pb::common::ValueType::UINT8 : pb::common::ValueType::FLOAT);
      vwd->set_distance(distances[pos]);
      vwd->set_metric_type(metric_type_);
    }
  }
  return butil::Status::OK();
}

// nprobe of the search parameter the index type reads: ivf_pq() (raw_ivf_pq.cc:170), binary_ivf_flat() (ivf_flat.cc:207-209),
// else ivf_flat() (ivf_flat.cc:211)
int32_t VectorIndexB200::SearchNprobe(const pb::common::VectorSearchParameter& parameter) const {
  if (vector_index_type == pb::common::VECTOR_INDEX_TYPE_IVF_PQ) return parameter.ivf_pq().nprobe();
  if (vector_index_type == pb::common::VECTOR_INDEX_TYPE_BINARY_IVF_FLAT) return parameter.binary_ivf_flat().nprobe();
  return parameter.ivf_flat().nprobe();
}

butil::Status VectorIndexB200::Train(std::vector<float>& train_datas) {
  if (vector_index_type == pb::common::VECTOR_INDEX_TYPE_FLAT || vector_index_type == pb::common::VECTOR_INDEX_TYPE_HNSW ||
      vector_index_type == pb::common::VECTOR_INDEX_TYPE_BINARY_FLAT)
    return butil::Status::OK();  // flat.cc:464-466, hnsw.cc:560
  const size_t data_size = dimension_ > 0 ? train_datas.size() / dimension_ : 0;
  if (data_size == 0) return butil::Status(pb::error::EILLEGAL_PARAMTETERS, "data size invalid");  // ivf_flat.cc:646-649
  if (train_datas.size() % dimension_ != 0)
    return butil::Status(pb::error::EILLEGAL_PARAMTETERS, "dimension not match " + std::to_string(train_datas.size()) + " " + std::to_string(dimension_));
  if (!index_) return ToStatus(B200VS_EINTERNAL);
  return ToStatus(b200vs_train(index_, (int64_t)data_size, train_datas.data()));
}

// VectorIndexIvfFlat<faiss::IndexBinary>::Train(std::vector<uint8_t>&), ivf_flat.cc:578-640; Flat: no-op
butil::Status VectorIndexB200::Train(std::vector<uint8_t>& train_datas) {
  if (vector_index_type != pb::common::VECTOR_INDEX_TYPE_BINARY_IVF_FLAT) return butil::Status::OK();
  const size_t code = (size_t)dimension_ / 8;
  const size_t data_size = code > 0 ? train_datas.size() / code : 0;
  if (data_size == 0) return butil::Status(pb::error::EILLEGAL_PARAMTETERS, "data size invalid");
  if (train_datas.size() % code != 0)
    return butil::Status(pb::error::EILLEGAL_PARAMTETERS, "dimension not match " + std::to_string(train_datas.size()) + " * CHAR_BIT(8) " + std::to_string(dimension_));
  if (!index_) return ToStatus(B200VS_EINTERNAL);
  return ToStatus(b200vs_train_binary(index_, (int64_t)data_size, train_datas.data()));
}

butil::Status VectorIndexB200::Train(const std::vector<pb::common::VectorWithId>& vectors) {  // ivf_flat.cc:714-742
  if (binary_) {
    std::vector<uint8_t> train_datas;
    train_datas.reserve((size_t)dimension_ / 8 * vectors.size());
    for (const auto& v : vectors) {
      if ((int)v.vector().binary_values().size() != dimension_ / 8)
        return butil::Status(pb::error::EINTERNAL, "dimension not match " + std::to_string(v.vector().binary_values_size()) + " * CHAR_BIT(8) " + std::to_string(dimension_));
      for (const auto& b : v.vector().binary_values()) train_datas.push_back(b.empty() ? 0 : static_cast<uint8_t>(b[0]));
    }
    return Train(train_datas);
  }
  std::vector<float> train_datas;
  train_datas.reserve((size_t)dimension_ * vectors.size());
  for (const auto& v : vectors) {
    if ((int)v.vector().float_values().size() != dimension_)
      return butil::Status(pb::error::EINTERNAL, "ivf_flat index dimension not match");
    train_datas.insert(train_datas.end(), v.vector().float_values().begin(), v.vector().float_values().end());
  }
  return Train(train_datas);
}

bool VectorIndexB200::NeedTrain() {
  return vector_index_type == pb::common::VECTOR_INDEX_TYPE_IVF_FLAT || vector_index_type == pb::common::VECTOR_INDEX_TYPE_IVF_PQ ||
         vector_index_type == pb::common::VECTOR_INDEX_TYPE_BINARY_IVF_FLAT;
}
bool VectorIndexB200::IsTrained() { return index_ && b200vs_is_trained(index_) != 0; }
bool VectorIndexB200::NeedToSave(int64_t last_save_log_behind) { return SupportSave() && last_save_log_behind > 10000; }  // flat.cc:515-531

namespace {
butil::Status AbiStatus(int rc) {
  if (rc == B200VS_OK) return butil::Status::OK();
  pb::error::Errno e = pb::error::EINTERNAL;
  if (rc == B200VS_EILLEGAL_PARAMETERS) e = pb::error::EILLEGAL_PARAMTETERS;
  else if (rc == B200VS_EVECTOR_INVALID) e = pb::error::EVECTOR_INVALID;
  else if (rc == B200VS_EVECTOR_ID_DUPLICATED) e = pb::error::EVECTOR_ID_DUPLICATED;
  else if (rc == B200VS_EVECTOR_NOT_SUPPORT) e = pb::error::EVECTOR_NOT_SUPPORT;
  return butil::Status(e, b200vs_last_error());
}
b200vs_metric AbiMetric(pb::common::MetricType m) {
  return m == pb::common::METRIC_TYPE_INNER_PRODUCT ? B200VS_IP : m == pb::common::METRIC_TYPE_COSINE ? B200VS_COSINE : B200VS_L2;
}
}  // namespace

butil::Status VectorIndexB200Utils::CalcDistance(int algorithm_type, pb::common::MetricType metric_type,
                                                 const std::vector<pb::common::Vector>& op_left_vectors,
                                                 const std::vector<pb::common::Vector>& op_right_vectors, bool is_return_normlize,
                                                 std::vector<std::vector<float>>& distances,
                                                 std::vector<pb::common::Vector>& result_op_left_vectors,
                                                 std::vector<pb::common::Vector>& result_op_right_vectors, int device) {
  if (algorithm_type != B200VS_ALGORITHM_FAISS && algorithm_type != B200VS_ALGORITHM_HNSWLIB)
    return butil::Status(pb::error::EILLEGAL_PARAMTETERS, "invalid algorithm type : ALGORITHM_NONE");     // utils.cc:70-76
  if (metric_type == pb::common::METRIC_TYPE_HAMMING)
    return CalcHammingDistance(algorithm_type, op_left_vectors, op_right_vectors, is_return_normlize, distances, result_op_left_vectors,
                               result_op_right_vectors, device);
  if (metric_type != pb::common::METRIC_TYPE_L2 && metric_type != pb::common::METRIC_TYPE_INNER_PRODUCT && metric_type != pb::common::METRIC_TYPE_COSINE)
    return butil::Status(pb::error::EILLEGAL_PARAMTETERS, "invalid metric_type type : METRIC_TYPE_NONE");  // utils.cc:151-157
  distances.clear();
  distances.resize(op_left_vectors.size());  // CalcDistanceCore, utils.cc:86-88
  if (op_left_vectors.empty() || op_right_vectors.empty()) return butil::Status::OK();
  const size_t d = op_left_vectors[0].float_values().size();
  for (const auto& v : op_left_vectors) if (v.float_values().size() != d) return butil::Status(pb::error::EILLEGAL_PARAMTETERS, "op_left_vectors dimension not match");
  for (const auto& v : op_right_vectors) if (v.float_values().size() != d) return butil::Status(pb::error::EILLEGAL_PARAMTETERS, "op_right_vectors dimension not match");
  const size_t nl = op_left_vectors.size(), nr = op_right_vectors.size();
  std::vector<float> left(nl * d), right(nr * d), out(nl * nr), lo, ro;
  for (size_t i = 0; i < nl; ++i) memcpy(left.data() + i * d, op_left_vectors[i].float_values().data(), d * sizeof(float));
  for (size_t i = 0; i < nr; ++i) memcpy(right.data() + i * d, op_right_vectors[i].float_values().data(), d * sizeof(float));
  if (is_return_normlize) { lo.resize(nl * d); ro.resize(nr * d); }
  const int rc = b200vs_calc_distance(device, algorithm_type, AbiMetric(metric_type), (int32_t)d, (int64_t)nl, left.data(), (int64_t)nr, right.data(),
                                      out.data(), is_return_normlize ? lo.data() : nullptr, is_return_normlize ? ro.data() : nullptr);
  if (rc != B200VS_OK) return AbiStatus(rc);
  for (size_t i = 0; i < nl; ++i) distances[i].assign(out.begin() + i * nr, out.begin() + (i + 1) * nr);
  if (is_return_normlize) {  // ResultOpVectorAssignment, utils.cc:421-426
    auto fill = [&](std::vector<pb::common::Vector>& dst, const std::vector<float>& src, size_t n) {
      dst.clear();
      dst.resize(n);
      for (size_t i = 0; i < n; ++i) {
        dst[i].mutable_float_values()->assign(src.begin() + i * d, src.begin() + (i + 1) * d);
        dst[i].set_dimension((int32_t)d);
        dst[i].set_value_type(pb::common::ValueType::FLOAT);
      }
    };
    fill(result_op_left_vectors, lo, nl);
    fill(result_op_right_vectors, ro, nr);
  }
  return butil::Status::OK();
}

// The HAMMING branch of CalcDistanceByFaiss (utils.cc:146-149, :333-356): popcount(a ^ b) over the operands' binary_values.
// CalcDistanceByHnswlib has no HAMMING case (utils.cc:160-192): it computes nothing and returns OK, as here.
butil::Status VectorIndexB200Utils::CalcHammingDistance(int algorithm_type, const std::vector<pb::common::Vector>& op_left_vectors,
                                                        const std::vector<pb::common::Vector>& op_right_vectors, bool is_return_normlize,
                                                        std::vector<std::vector<float>>& distances,
                                                        std::vector<pb::common::Vector>& result_op_left_vectors,
                                                        std::vector<pb::common::Vector>& result_op_right_vectors, int device) {
  distances.clear();
  distances.resize(op_left_vectors.size());
  if (algorithm_type != B200VS_ALGORITHM_FAISS || op_left_vectors.empty() || op_right_vectors.empty()) return butil::Status::OK();
  const size_t code = op_left_vectors[0].binary_values().size();
  for (const auto& v : op_left_vectors) if (v.binary_values().size() != code) return butil::Status(pb::error::EILLEGAL_PARAMTETERS, "op_left_vectors dimension not match");
  for (const auto& v : op_right_vectors) if (v.binary_values().size() != code) return butil::Status(pb::error::EILLEGAL_PARAMTETERS, "op_right_vectors dimension not match");
  const size_t nl = op_left_vectors.size(), nr = op_right_vectors.size();
  auto pack = [&](const std::vector<pb::common::Vector>& vs) {
    std::vector<uint8_t> out(vs.size() * code);
    for (size_t i = 0; i < vs.size(); ++i)
      for (size_t j = 0; j < code; ++j) out[i * code + j] = vs[i].binary_values()[j].empty() ? 0 : static_cast<uint8_t>(vs[i].binary_values()[j][0]);
    return out;
  };
  const std::vector<uint8_t> left = pack(op_left_vectors), right = pack(op_right_vectors);
  std::vector<float> out(nl * nr);
  const int rc = b200vs_calc_distance_binary(device, (int32_t)(code * 8), (int64_t)nl, left.data(), (int64_t)nr, right.data(), out.data());
  if (rc != B200VS_OK) return AbiStatus(rc);
  for (size_t i = 0; i < nl; ++i) distances[i].assign(out.begin() + i * nr, out.begin() + (i + 1) * nr);
  if (is_return_normlize) {  // ResultOpBinaryVectorAssignment, utils.cc:439-444: the operands, dimension in bits, UINT8
    auto fill = [&](std::vector<pb::common::Vector>& dst, const std::vector<pb::common::Vector>& src) {
      dst = src;
      for (auto& v : dst) { v.set_dimension((int32_t)(code * 8)); v.set_value_type(pb::common::ValueType::UINT8); }
    };
    fill(result_op_left_vectors, op_left_vectors);
    fill(result_op_right_vectors, op_right_vectors);
  }
  return butil::Status::OK();
}

BruteForceScannerB200::BruteForceScannerB200(pb::common::MetricType metric_type, int32_t dimension,
                                             const std::vector<pb::common::VectorWithId>& vector_with_ids, uint32_t topk, int device)
    : metric_type_(metric_type), dimension_(dimension), nq_(vector_with_ids.size()), topk_(topk) {
  if (dimension <= 0) { init_status_ = butil::Status(pb::error::EVECTOR_INVALID, "vector index dimension is invalid"); return; }  // reader.cc:1889-1894
  if (vector_with_ids.empty()) { init_status_ = butil::Status(pb::error::EILLEGAL_PARAMTETERS, "vector_with_ids is empty"); return; }
  init_status_ = CheckVectorDimension(vector_with_ids, dimension);
  if (!init_status_.ok() || topk == 0) return;
  const std::vector<float> x = ExtractVectorValue(vector_with_ids, dimension);
  init_status_ = AbiStatus(b200vs_scan_begin(device, AbiMetric(metric_type), dimension, (int64_t)nq_, x.data(), (int32_t)topk, nullptr, &scan_));
}
BruteForceScannerB200::~BruteForceScannerB200() { if (scan_) b200vs_scan_abort(scan_); }

butil::Status BruteForceScannerB200::Push(const std::vector<pb::common::VectorWithId>& batch) {
  if (!init_status_.ok()) return init_status_;
  if (batch.empty() || topk_ == 0) return butil::Status::OK();
  auto status = CheckVectorDimension(batch, dimension_);
  if (!status.ok()) return status;
  std::vector<int64_t> ids(batch.size());
  for (size_t i = 0; i < batch.size(); ++i) ids[i] = batch[i].id();
  const std::vector<float> x = ExtractVectorValue(batch, dimension_);
  return AbiStatus(b200vs_scan_push(scan_, (int64_t)batch.size(), x.data(), ids.data()));
}

butil::Status BruteForceScannerB200::Finish(std::vector<pb::index::VectorWithDistanceResult>& results) {
  if (!init_status_.ok()) return init_status_;
  results.resize(nq_);  // reader.cc:2022
  if (topk_ == 0) return butil::Status::OK();
  std::vector<float> distances(nq_ * topk_, 0.0f);
  std::vector<int64_t> labels(nq_ * topk_, -1);
  b200vs_scan* s = scan_;
  scan_ = nullptr;  // finish frees the handle
  const int rc = b200vs_scan_finish(s, distances.data(), labels.data());
  if (rc != B200VS_OK) return AbiStatus(rc);
  for (size_t row = 0; row < nq_; ++row)
    for (uint32_t i = 0; i < topk_; ++i) {
      const size_t pos = row * topk_ + i;
      if (labels[pos] < 0) continue;
      auto* vwd = results[row].add_vector_with_distances();
      vwd->mutable_vector_with_id()->set_id(labels[pos]);
      vwd->mutable_vector_with_id()->mutable_vector()->set_dimension(dimension_);
      vwd->mutable_vector_with_id()->mutable_vector()->set_value_type(pb::common::ValueType::FLOAT);
      vwd->set_distance(distances[pos]);
      vwd->set_metric_type(metric_type_);
    }
  return butil::Status::OK();
}

}  // namespace dingodb

// dingo_shim.h — minimal stand-ins for the dingo-store / brpc / protobuf types that appear in the VectorIndex
// plugin interface (src/vector/vector_index.h:56-279), so the drop-in subclass in vector_index_b200.{h,cc} can be
// compiled and tested in this repository, where proto/*.pb.h, butil and faiss are not available
// (SURVEY.md §0).  In a dingo-store checkout this header is NOT used: define B200VS_WITH_DINGO_HEADERS and the
// subclass compiles against the real "vector/vector_index.h" (see INTEGRATION.md).
// Only the accessors the plugin code touches are reproduced, with the generated-protobuf spelling.
#pragma once
#include <cstdint>
#include <memory>
#include <string>
#include <utility>
#include <vector>

namespace butil {
class Status {
 public:
  Status() = default;
  Status(int code, const std::string& msg) : code_(code), msg_(msg) {}
  static Status OK() { return Status(); }
  bool ok() const { return code_ == 0; }
  int error_code() const { return code_; }
  const char* error_cstr() const { return msg_.c_str(); }
  const std::string& error_str() const { return msg_; }
 private:
  int code_ = 0;
  std::string msg_;
};
}  // namespace butil

namespace dingodb {
namespace pb {
namespace error {
// numeric values are internal to this shim; the real enum lives in proto/error.pb.h
enum Errno { OK = 0, EINTERNAL = 10000, EILLEGAL_PARAMTETERS = 10010, EVECTOR_INVALID = 30003, EVECTOR_NOT_SUPPORT = 30001,
             EVECTOR_NOT_TRAIN = 30012, EVECTOR_ID_DUPLICATED = 30004, EVECTOR_INDEX_NOT_FOUND = 30008 };
}  // namespace error
namespace common {
enum ValueType { FLOAT = 0, UINT8 = 1 };
enum MetricType { METRIC_TYPE_NONE = 0, METRIC_TYPE_L2 = 1, METRIC_TYPE_INNER_PRODUCT = 2, METRIC_TYPE_COSINE = 3,
                  METRIC_TYPE_HAMMING = 4 };
// numeric values are internal to this shim; the real enum lives in proto/common.pb.h
enum VectorIndexType { VECTOR_INDEX_TYPE_NONE = 0, VECTOR_INDEX_TYPE_FLAT = 1, VECTOR_INDEX_TYPE_IVF_FLAT = 2,
                       VECTOR_INDEX_TYPE_IVF_PQ = 3, VECTOR_INDEX_TYPE_HNSW = 4, VECTOR_INDEX_TYPE_BINARY_FLAT = 6,
                       VECTOR_INDEX_TYPE_BINARY_IVF_FLAT = 7 };

class Vector {
 public:
  int32_t dimension() const { return dimension_; }
  void set_dimension(int32_t d) { dimension_ = d; }
  ValueType value_type() const { return value_type_; }
  void set_value_type(ValueType t) { value_type_ = t; }
  const std::vector<float>& float_values() const { return float_values_; }
  std::vector<float>* mutable_float_values() { return &float_values_; }
  int float_values_size() const { return (int)float_values_.size(); }
  void add_float_values(float v) { float_values_.push_back(v); }
  // repeated bytes binary_values: one byte per element for the binary index types (vector_index_utils.cc:590-600)
  const std::vector<std::string>& binary_values() const { return binary_values_; }
  int binary_values_size() const { return (int)binary_values_.size(); }
  void add_binary_values(std::string v) { binary_values_.push_back(std::move(v)); }
 private:
  int32_t dimension_ = 0;
  ValueType value_type_ = FLOAT;
  std::vector<float> float_values_;
  std::vector<std::string> binary_values_;
};
class VectorWithId {
 public:
  int64_t id() const { return id_; }
  void set_id(int64_t v) { id_ = v; }
  const Vector& vector() const { return vector_; }
  Vector* mutable_vector() { return &vector_; }
 private:
  int64_t id_ = 0;
  Vector vector_;
};
struct SearchFlatParam {};
struct SearchIvfParam { int32_t nprobe_ = 0; int32_t nprobe() const { return nprobe_; } void set_nprobe(int32_t v) { nprobe_ = v; } };
struct SearchHnswParam { int32_t efsearch_ = 0; int32_t efsearch() const { return efsearch_; } void set_efsearch(int32_t v) { efsearch_ = v; } };
class VectorSearchParameter {
 public:
  const SearchIvfParam& ivf_flat() const { return ivf_flat_; }
  SearchIvfParam* mutable_ivf_flat() { return &ivf_flat_; }
  const SearchIvfParam& ivf_pq() const { return ivf_pq_; }
  SearchIvfParam* mutable_ivf_pq() { return &ivf_pq_; }
  const SearchHnswParam& hnsw() const { return hnsw_; }
  SearchHnswParam* mutable_hnsw() { return &hnsw_; }
  const SearchIvfParam& binary_ivf_flat() const { return binary_ivf_flat_; }
  SearchIvfParam* mutable_binary_ivf_flat() { return &binary_ivf_flat_; }
 private:
  SearchIvfParam ivf_flat_, ivf_pq_, binary_ivf_flat_;
  SearchHnswParam hnsw_;
};
struct CreateFlatParam { int32_t dimension_ = 0; MetricType metric_type_ = METRIC_TYPE_L2;
  int32_t dimension() const { return dimension_; } MetricType metric_type() const { return metric_type_; } };
struct CreateIvfFlatParam : CreateFlatParam { int32_t ncentroids_ = 0; int32_t ncentroids() const { return ncentroids_; } };
struct CreateIvfPqParam : CreateIvfFlatParam { int32_t nsubvector_ = 0, nbits_per_idx_ = 0;
  int32_t nsubvector() const { return nsubvector_; } int32_t nbits_per_idx() const { return nbits_per_idx_; } };
struct CreateHnswParam : CreateFlatParam { int32_t efconstruction_ = 0, nlinks_ = 0; int64_t max_elements_ = 0;
  int32_t efconstruction() const { return efconstruction_; } int32_t nlinks() const { return nlinks_; } int64_t max_elements() const { return max_elements_; } };
class VectorIndexParameter {
 public:
  VectorIndexType vector_index_type() const { return type_; }
  void set_vector_index_type(VectorIndexType t) { type_ = t; }
  const CreateFlatParam& flat_parameter() const { return flat_; }
  CreateFlatParam* mutable_flat_parameter() { return &flat_; }
  const CreateIvfFlatParam& ivf_flat_parameter() const { return ivf_flat_; }
  CreateIvfFlatParam* mutable_ivf_flat_parameter() { return &ivf_flat_; }
  const CreateIvfPqParam& ivf_pq_parameter() const { return ivf_pq_; }
  CreateIvfPqParam* mutable_ivf_pq_parameter() { return &ivf_pq_; }
  const CreateHnswParam& hnsw_parameter() const { return hnsw_; }
  CreateHnswParam* mutable_hnsw_parameter() { return &hnsw_; }
  const CreateFlatParam& binary_flat_parameter() const { return binary_flat_; }  // dimension in bits, metric HAMMING
  CreateFlatParam* mutable_binary_flat_parameter() { return &binary_flat_; }
  const CreateIvfFlatParam& binary_ivf_flat_parameter() const { return binary_ivf_flat_; }
  CreateIvfFlatParam* mutable_binary_ivf_flat_parameter() { return &binary_ivf_flat_; }
 private:
  VectorIndexType type_ = VECTOR_INDEX_TYPE_NONE;
  CreateFlatParam flat_; CreateIvfFlatParam ivf_flat_; CreateIvfPqParam ivf_pq_; CreateHnswParam hnsw_;
  CreateFlatParam binary_flat_; CreateIvfFlatParam binary_ivf_flat_;
};
struct RegionEpoch { int64_t conf_version = 0, version = 0; };
struct Range { std::string start_key, end_key; };
}  // namespace common
namespace index {
class VectorWithDistance {
 public:
  const common::VectorWithId& vector_with_id() const { return vwi_; }
  common::VectorWithId* mutable_vector_with_id() { return &vwi_; }
  float distance() const { return distance_; }
  void set_distance(float d) { distance_ = d; }
  common::MetricType metric_type() const { return metric_; }
  void set_metric_type(common::MetricType m) { metric_ = m; }
 private:
  common::VectorWithId vwi_;
  float distance_ = 0;
  common::MetricType metric_ = common::METRIC_TYPE_NONE;
};
class VectorWithDistanceResult {
 public:
  VectorWithDistance* add_vector_with_distances() { v_.emplace_back(); return &v_.back(); }
  int vector_with_distances_size() const { return (int)v_.size(); }
  const VectorWithDistance& vector_with_distances(int i) const { return v_[i]; }
  const std::vector<VectorWithDistance>& vector_with_distances() const { return v_; }
  void Swap(VectorWithDistanceResult* o) { v_.swap(o->v_); }
 private:
  std::vector<VectorWithDistance> v_;
};
}  // namespace index
}  // namespace pb

class ThreadPool;
using ThreadPoolPtr = std::shared_ptr<ThreadPool>;

// The plugin base class, reduced to the members the subclass overrides or uses (vector_index.h:56-279).
class VectorIndex {
 public:
  VectorIndex(int64_t id, const pb::common::VectorIndexParameter& p, const pb::common::RegionEpoch& e, const pb::common::Range& r,
              ThreadPoolPtr tp)
      : id(id), vector_index_type(p.vector_index_type()), epoch(e), range(r), vector_index_parameter(p), thread_pool(std::move(tp)) {}
  virtual ~VectorIndex() = default;

  class FilterFunctor {
   public:
    virtual ~FilterFunctor() = default;
    virtual bool Check(int64_t vector_id) = 0;
  };
  class RangeFilterFunctor : public FilterFunctor {  // vector_index.h:75-84 (+ accessors, see INTEGRATION.md)
   public:
    RangeFilterFunctor(int64_t min_vector_id, int64_t max_vector_id) : min_vector_id_(min_vector_id), max_vector_id_(max_vector_id) {}
    bool Check(int64_t vector_id) override { return vector_id >= min_vector_id_ && vector_id < max_vector_id_; }
    int64_t MinVectorId() const { return min_vector_id_; }
    int64_t MaxVectorId() const { return max_vector_id_; }
   private:
    int64_t min_vector_id_, max_vector_id_;
  };
  class SortFilterFunctor : public FilterFunctor {  // vector_index.h:112-146 (+ accessors)
   public:
    explicit SortFilterFunctor(std::vector<int64_t>& vector_ids, bool is_negation = false) : is_negation_(is_negation) { vector_ids_.swap(vector_ids); }
    bool Check(int64_t vector_id) override {
      int64_t begin = 0, end = (int64_t)vector_ids_.size() - 1;
      bool exist = false;
      while (begin <= end) {
        int64_t mid = (begin + end) / 2;
        if (vector_id == vector_ids_[mid]) { exist = true; break; }
        if (vector_id < vector_ids_[mid]) end = mid - 1; else begin = mid + 1;
      }
      return !is_negation_ ? exist : !exist;
    }
    const std::vector<int64_t>& VectorIds() const { return vector_ids_; }
    bool IsNegation() const { return is_negation_; }
   private:
    bool is_negation_;
    std::vector<int64_t> vector_ids_;
  };

  virtual int32_t GetDimension() = 0;
  virtual pb::common::MetricType GetMetricType() = 0;
  virtual butil::Status GetCount(int64_t& count) = 0;
  virtual butil::Status GetDeletedCount(int64_t& deleted_count) = 0;
  virtual butil::Status GetMemorySize(int64_t& memory_size) = 0;
  virtual bool IsExceedsMaxElements(int64_t vector_size) = 0;
  virtual butil::Status Add(const std::vector<pb::common::VectorWithId>& vector_with_ids) = 0;
  virtual butil::Status Upsert(const std::vector<pb::common::VectorWithId>& vector_with_ids) = 0;
  virtual butil::Status Delete(const std::vector<int64_t>& delete_ids) = 0;
  virtual butil::Status Save(const std::string& path) = 0;
  virtual butil::Status Load(const std::string& path) = 0;
  virtual butil::Status Search(const std::vector<pb::common::VectorWithId>& vector_with_ids, uint32_t topk,
                               const std::vector<std::shared_ptr<FilterFunctor>>& filters, bool reconstruct,
                               const pb::common::VectorSearchParameter& parameter,
                               std::vector<pb::index::VectorWithDistanceResult>& results) = 0;
  virtual butil::Status RangeSearch(const std::vector<pb::common::VectorWithId>& vector_with_ids, float radius,
                                    const std::vector<std::shared_ptr<FilterFunctor>>& filters, bool reconstruct,
                                    const pb::common::VectorSearchParameter& parameter,
                                    std::vector<pb::index::VectorWithDistanceResult>& results) = 0;
  virtual void LockWrite() = 0;
  virtual void UnlockWrite() = 0;
  virtual butil::Status Train(std::vector<float>& train_datas) = 0;
  virtual butil::Status Train(std::vector<uint8_t>& /*train_datas*/) { return butil::Status::OK(); }  // vector_index.h:195
  virtual butil::Status Train(const std::vector<pb::common::VectorWithId>& vectors) = 0;
  virtual bool NeedToRebuild() = 0;
  virtual bool NeedTrain() { return false; }
  virtual bool IsTrained() { return true; }
  virtual bool NeedToSave(int64_t last_save_log_behind) = 0;
  virtual bool SupportSave() { return false; }
  virtual uint32_t WriteOpParallelNum() { return 1; }
  virtual pb::common::VectorIndexType VectorIndexSubType() { return pb::common::VECTOR_INDEX_TYPE_NONE; }  // vector_index.h:238

  int64_t Id() const { return id; }
  pb::common::VectorIndexType VectorIndexType() { return vector_index_type; }

 protected:
  int64_t id;
  pb::common::VectorIndexType vector_index_type;
  pb::common::RegionEpoch epoch;
  pb::common::Range range;
  pb::common::VectorIndexParameter vector_index_parameter;
  ThreadPoolPtr thread_pool;
};
using VectorIndexPtr = std::shared_ptr<VectorIndex>;

}  // namespace dingodb

// vector_index_b200.h — drop-in subclass of dingodb::VectorIndex backed by libb200vs (include/b200vs.h).
//
// One class serves the six plugin types; VectorIndexFactory::New{Flat,IvfFlat,IvfPq,Hnsw,BinaryFlat,BinaryIvfFlat}
// (src/vector/vector_index_factory.cc:40-95) would return it instead of VectorIndexFlat / VectorIndexIvfFlat /
// VectorIndexIvfPq / VectorIndexHnsw and their faiss::IndexBinary instantiations.  The class does only what the reference plugins do around their faiss /
// hnswlib calls: argument checks with the same status codes, pb -> flat-array marshalling
// (CheckVectorDimension / ExtractVectorValue / FillSearchResult, src/vector/vector_index_utils.cc:502-655), filter
// lowering, and the write lock bookkeeping; all arithmetic is behind the C ABI.
#pragma once
#ifdef B200VS_WITH_DINGO_HEADERS
#include "vector/vector_index.h"
#else
#include "dingo_shim.h"
#endif

#include <shared_mutex>

#include "../../include/b200vs.h"

namespace dingodb {

class VectorIndexB200 : public VectorIndex {
 public:
  VectorIndexB200(int64_t id, const pb::common::VectorIndexParameter& vector_index_parameter, const pb::common::RegionEpoch& epoch,
                  const pb::common::Range& range, ThreadPoolPtr thread_pool, int device = 0);
  ~VectorIndexB200() override;

  VectorIndexB200(const VectorIndexB200&) = delete;
  VectorIndexB200& operator=(const VectorIndexB200&) = delete;

  int32_t GetDimension() override { return dimension_; }
  pb::common::MetricType GetMetricType() override { return metric_type_; }
  butil::Status GetCount(int64_t& count) override;
  butil::Status GetDeletedCount(int64_t& deleted_count) override;
  butil::Status GetMemorySize(int64_t& memory_size) override;
  bool IsExceedsMaxElements(int64_t vector_size) override;

  butil::Status Add(const std::vector<pb::common::VectorWithId>& vector_with_ids) override;
  butil::Status Upsert(const std::vector<pb::common::VectorWithId>& vector_with_ids) override;
  butil::Status Delete(const std::vector<int64_t>& delete_ids) override;

  butil::Status Save(const std::string& path) override;
  butil::Status Load(const std::string& path) override;

  butil::Status Search(const std::vector<pb::common::VectorWithId>& vector_with_ids, uint32_t topk,
                       const std::vector<std::shared_ptr<FilterFunctor>>& filters, bool reconstruct,
                       const pb::common::VectorSearchParameter& parameter,
                       std::vector<pb::index::VectorWithDistanceResult>& results) override;
  butil::Status RangeSearch(const std::vector<pb::common::VectorWithId>& vector_with_ids, float radius,
                            const std::vector<std::shared_ptr<FilterFunctor>>& filters, bool reconstruct,
                            const pb::common::VectorSearchParameter& parameter,
                            std::vector<pb::index::VectorWithDistanceResult>& results) override;

  void LockWrite() override { write_gate_.lock(); }
  void UnlockWrite() override { write_gate_.unlock(); }
  butil::Status Train(std::vector<float>& train_datas) override;
  butil::Status Train(const std::vector<pb::common::VectorWithId>& vectors) override;
  butil::Status Train(std::vector<uint8_t>& train_datas) override;  // binary types: dim / 8 bytes per row
  bool NeedToRebuild() override { return false; }
  bool NeedTrain() override;
  bool IsTrained() override;
  bool NeedToSave(int64_t last_save_log_behind) override;
  // fork()-based saving (vector_index_snapshot_manager.cc:583-608) cannot carry a CUDA context into the child:
  // report "no save support" like the DiskANN plugin (vector_index_diskann.cc:267); the server rebuilds from RocksDB.
  bool SupportSave() override { return false; }
  pb::common::VectorIndexType VectorIndexSubType() override;  // vector_index.h:238

  // largest result count RangeSearch keeps per query (FLAGS_vector_index_max_range_search_result_count, vector_reader.cc:60)
  static int32_t max_range_search_result_count;

 private:
  butil::Status AddOrUpsert(const std::vector<pb::common::VectorWithId>& vector_with_ids, bool is_upsert);
  butil::Status ToStatus(int rc) const;
  int32_t SearchNprobe(const pb::common::VectorSearchParameter& parameter) const;

  b200vs_index* index_ = nullptr;
  int32_t dimension_ = 0;  // bits for the binary types
  bool binary_ = false;     // BINARY_FLAT / BINARY_IVF_FLAT: rows are UINT8 binary_values
  pb::common::MetricType metric_type_ = pb::common::METRIC_TYPE_NONE;
  std::shared_mutex write_gate_;  // LockWrite/UnlockWrite of the snapshot path; reads and writes lock inside the library
};

// VectorIndexUtils::CalcDistanceEntry (src/vector/vector_index_utils.cc:48-76) over the C ABI: same operand meaning
// (algorithm_type = pb::index::AlgorithmType: 1 FAISS, 2 HNSWLIB; metric; is_return_normlize) and the same error codes.
// METRIC_TYPE_HAMMING reads the operands' binary_values (utils.cc:146-149, :333-356).
class VectorIndexB200Utils {
 public:
  static butil::Status CalcDistance(int algorithm_type, pb::common::MetricType metric_type, const std::vector<pb::common::Vector>& op_left_vectors,
                                    const std::vector<pb::common::Vector>& op_right_vectors, bool is_return_normlize,
                                    std::vector<std::vector<float>>& distances, std::vector<pb::common::Vector>& result_op_left_vectors,
                                    std::vector<pb::common::Vector>& result_op_right_vectors, int device = 0);

 private:
  static butil::Status CalcHammingDistance(int algorithm_type, const std::vector<pb::common::Vector>& op_left_vectors,
                                           const std::vector<pb::common::Vector>& op_right_vectors, bool is_return_normlize,
                                           std::vector<std::vector<float>>& distances, std::vector<pb::common::Vector>& result_op_left_vectors,
                                           std::vector<pb::common::Vector>& result_op_right_vectors, int device);
};

// The inner loop of VectorReader::BruteForceSearch (src/vector/vector_reader.cc:1873-2048): the caller keeps the RocksDB
// iterator, pushes each decoded batch (FLAGS_vector_index_bruteforce_batch_count vectors) and collects the top-k at the end.
class BruteForceScannerB200 {
 public:
  BruteForceScannerB200(pb::common::MetricType metric_type, int32_t dimension, const std::vector<pb::common::VectorWithId>& vector_with_ids,
                        uint32_t topk, int device = 0);
  ~BruteForceScannerB200();
  BruteForceScannerB200(const BruteForceScannerB200&) = delete;
  BruteForceScannerB200& operator=(const BruteForceScannerB200&) = delete;
  butil::Status Push(const std::vector<pb::common::VectorWithId>& vector_with_id_batch);
  butil::Status Finish(std::vector<pb::index::VectorWithDistanceResult>& results);  // ascending by distance, one entry per query

 private:
  b200vs_scan* scan_ = nullptr;
  butil::Status init_status_;
  pb::common::MetricType metric_type_;
  int32_t dimension_;
  size_t nq_;
  uint32_t topk_;
};

}  // namespace dingodb

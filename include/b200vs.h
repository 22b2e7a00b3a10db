/*
 * b200vs.h — C ABI of the B200-native vector-search engine (libb200vs.so).
 *
 * This is the drop-in boundary behind dingo-store's C++ VectorIndex plugin surface
 * (reference: src/vector/vector_index.h:56-279).  A thin C++ subclass of dingodb::VectorIndex
 * (dingo-store_b200/host/vector_index_b200.{h,cc}; binding shown in INTEGRATION.md) marshals protobuf
 * to flat arrays and calls these entry points; everything below the ABI is CUDA for sm_100a.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes only.  No exception or abort crosses the ABI: every entry
 *     point returns a b200vs_status; b200vs_last_error() gives a thread-local message.
 *   - Status codes map 1:1 to the pb::error::Errno classes the reference plugins return
 *     (src/vector/vector_index_flat.cc:209, :193-196; vector_index_ivf_flat.cc:112; vector_index_hnsw.cc:332-336,
 *     :487-493; vector_index_utils.cc:551-561).
 *   - Unless a function name ends in _device, all data pointers are HOST pointers.
 *   - Distances are returned in the reference's API semantics (src/vector/vector_index_utils.cc:611-655):
 *     L2 = squared L2; INNER_PRODUCT and COSINE = 1 - ip.  Results are ascending; rows with fewer than k
 *     hits are padded with id = -1, dist = 0 (labels pre-filled -1, vector_index_flat.cc:218-219).
 *   - Thread-safety: searches may be issued concurrently from many host threads (the reference calls
 *     Search from a 16-thread pool, src/server/server.cc:868-873); writers are serialised against readers
 *     by a reader/writer lock inside the index (reference: RWLock, src/common/synchronization.h:133-156).
 */
#ifndef B200VS_H_
#define B200VS_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct b200vs_index b200vs_index; /* opaque */

/* replaces VectorIndexFactory::New type switch, src/vector/vector_index_factory.cc:40-95.  The binary types
 * (VectorIndexFlat<faiss::IndexBinary>, VectorIndexIvfFlat<faiss::IndexBinary>, factory.cc:73-80) take dim in BITS
 * (a multiple of 8, at most 32768), metric B200VS_HAMMING, and rows of dim / 8 bytes through the *_binary entry points. */
typedef enum {
  B200VS_FLAT = 0, B200VS_IVF_FLAT = 1, B200VS_IVF_PQ = 2, B200VS_HNSW = 3, B200VS_BINARY_FLAT = 4, B200VS_BINARY_IVF_FLAT = 5
} b200vs_type;
/* mirrors pb::common::MetricType L2 / INNER_PRODUCT / COSINE / HAMMING */
typedef enum { B200VS_L2 = 1, B200VS_IP = 2, B200VS_COSINE = 3, B200VS_HAMMING = 4 } b200vs_metric;

typedef enum {
  B200VS_OK = 0,
  B200VS_EILLEGAL_PARAMETERS = 1, /* pb::error::EILLEGAL_PARAMTETERS */
  B200VS_EVECTOR_INVALID = 2,     /* pb::error::EVECTOR_INVALID       */
  B200VS_EVECTOR_NOT_TRAIN = 3,   /* pb::error::EVECTOR_NOT_TRAIN     */
  B200VS_EVECTOR_NOT_SUPPORT = 4, /* pb::error::EVECTOR_NOT_SUPPORT   */
  B200VS_EINTERNAL = 5,           /* pb::error::EINTERNAL             */
  B200VS_EVECTOR_ID_DUPLICATED = 6 /* pb::error::EVECTOR_ID_DUPLICATED */
} b200vs_status;

/* creation parameters: the union of pb::common::Create{Flat,IvfFlat,IvfPq,Hnsw}Param fields read at
 * vector_index_flat.cc:81-82, vector_index_ivf_flat.cc:75-83, vector_index_raw_ivf_pq.cc:60-75,
 * vector_index_hnsw.cc:141-182.  0 = reference default (src/common/constant.h:177-188). */
typedef struct {
  int32_t nlist;        /* ncentroids; default 2048 */
  int32_t pq_m;         /* nsubvector; default 64   */
  int32_t pq_nbits;     /* nbits_per_idx; default 8 (only 8 is implemented) */
  int32_t hnsw_m;       /* nlinks */
  int32_t hnsw_efc;     /* efconstruction */
  int64_t max_elements; /* hnsw max_elements */
  int32_t device;       /* CUDA device ordinal */
  int32_t hnsw_build_threads; /* host threads inserting a batch into the HNSW graph.  0 / 1 = single writer (deterministic
                               * graph, equal to the oracle's); > 1 = concurrent insertion with per-node locks, what the
                               * reference does with its 16-thread pool (vector_index_hnsw.cc:229-243: graph differs run to run) */
} b200vs_params;

/* search-time parameters: pb::common::VectorSearchParameter knobs (ivf_flat().nprobe() ivf_flat.cc:211,
 * ivf_pq().nprobe() raw_ivf_pq.cc:170, hnsw().efsearch() hnsw.cc:332) plus the device form of the
 * reference's FilterFunctors (vector_index.h:67-146): all given filters are ANDed. */
typedef struct {
  int32_t nprobe;   /* <=0 -> 80 (Constant::kSearchIvfFlatParamNprobe); clamped to nlist */
  int32_t efsearch; /* 0 -> keep the sticky ef; outside [0,1024] -> EILLEGAL_PARAMETERS */
  int32_t has_range; /* RangeFilterFunctor: range_min <= id < range_max */
  int32_t negate;    /* SortFilterFunctor / ConcreteFilterFunctor is_negation */
  int64_t range_min, range_max;
  const int64_t* sorted_ids; /* ascending id list (HOST pointer), or NULL */
  int64_t n_ids;
  int32_t exact_only; /* 1 = force the exact FP32 scan (skip the tensor-core candidate pass) */
  int32_t reserved;
} b200vs_search_params;

/* lifecycle — replaces the plugin constructors / destructors */
int b200vs_create(b200vs_type type, b200vs_metric metric, int32_t dim, const b200vs_params* params, b200vs_index** out);
void b200vs_destroy(b200vs_index* idx);

/* VectorIndex::Train(std::vector<float>&) — vector_index_ivf_flat.cc:644-712, raw_ivf_pq.cc:457-500,
 * ivf_pq.cc:327-395.  x row-major [n,dim], RAW values (COSINE is normalised inside).  Flat/HNSW: no-op. */
int b200vs_train(b200vs_index* idx, int64_t n, const float* x);
/* Load / fetch trained state (IVF centroids, PQ codebooks, HNSW graph) as a flat blob — used to search the
 * SAME trained index as the CPU path.  Layouts: see DESIGN.md §Trained-state blobs. */
int b200vs_set_trained_state(b200vs_index* idx, const void* blob, size_t len);
int64_t b200vs_get_trained_state(b200vs_index* idx, void* blob, size_t cap); /* returns bytes needed/written, <0 on error */

/* VectorIndex::Add / Upsert / Delete — flat.cc:121-203, ivf_flat.cc:92-190, hnsw.cc:203-281.
 * ids must be unique within one call (EVECTOR_ID_DUPLICATED); upsert=1 removes pre-existing ids first. */
int b200vs_add_with_ids(b200vs_index* idx, int64_t n, const float* x, const int64_t* ids, int upsert);
int b200vs_remove_ids(b200vs_index* idx, int64_t n, const int64_t* ids, int64_t* n_removed);

/* VectorIndex::Search — flat.cc:205-264, ivf_flat.cc:191-275, raw_ivf_pq.cc:157-210, hnsw.cc:318-485.
 * xq row-major [nq,dim] RAW; out_dist [nq,k], out_ids [nq,k]. */
int b200vs_search(b200vs_index* idx, int64_t nq, const float* xq, int32_t k, const b200vs_search_params* sp,
                  float* out_dist, int64_t* out_ids);
/* b200vs_search coalesces concurrent callers (SURVEY 8b): the unchanged reference slices every batch into one-query tasks
 * on its 16-thread pool (src/vector/vector_index.cc:54, :244-271), so the plugin sees many concurrent nq = 1 calls.  Calls
 * of <= 64 queries without id-list filters queue inside the library; the caller that finds no leader active runs every
 * compatible pending request (same k / nprobe / efsearch / exact_only / id range) as ONE batch and hands the results back.
 * on: 1 / 0 switch it, < 0 only reads; stats (nullable): [0] batches run, [1] requests served through them. */
int b200vs_set_coalescing(b200vs_index* idx, int on, int64_t stats[2]);

/* Same, with xq / out_dist / out_ids DEVICE pointers on the index's device; enqueued on `stream`
 * (a cudaStream_t) and NOT synchronised when it returns.  stream == NULL runs the search on a library-owned stream and
 * returns only when the results are complete (it does not touch the legacy default stream).  The same holds for
 * b200vs_coarse_device and b200vs_search_probes_device. */
int b200vs_search_device(b200vs_index* idx, int64_t nq, const float* xq_dev, int32_t k,
                         const b200vs_search_params* sp, float* out_dist_dev, int64_t* out_ids_dev, void* stream);

/* VectorIndex::RangeSearch — flat.cc:267-323, ivf_flat.cc:278-368 (HNSW: EVECTOR_NOT_SUPPORT, hnsw.cc:487-493).
 * radius in API semantics (mapped 1-r for IP/COSINE, flat.cc:282-285).  At most max_results hits per
 * query are kept (closest first); out_counts[nq] receives the per-query hit count. */
int b200vs_range_search(b200vs_index* idx, int64_t nq, const float* xq, float radius, int32_t max_results,
                        const b200vs_search_params* sp, float* out_dist, int64_t* out_ids, int32_t* out_counts);

/* Stored vectors by id — what VectorIndexHnsw::Search returns per hit when reconstruct = true (hnswlib getDataByLabel,
 * vector_index_hnsw.cc:383-395; cosine indexes never reconstruct, :469-472).  out [n, dim]; found[n] = 1 / 0 (unknown or
 * deleted id: row left untouched).  Implemented for HNSW and FLAT. */
int b200vs_reconstruct(b200vs_index* idx, int64_t n, const int64_t* ids, float* out, uint8_t* found);

/* VectorIndex::VectorIndexSubType (vector_index.h:238; vector_index_ivf_pq.cc:474): for IVF_PQ the index type actually
 * serving searches — B200VS_FLAT while the inner Flat index is in use, B200VS_IVF_PQ once trained on enough data; -1 =
 * untrained.  Other types return their own type. */
int b200vs_sub_type(b200vs_index* idx);

/* GetCount / GetDeletedCount / GetMemorySize / IsTrained / NeedTrain — vector_index.h:150-152,:199-200 */
int b200vs_count(b200vs_index* idx, int64_t* count);
int b200vs_deleted_count(b200vs_index* idx, int64_t* count);
int b200vs_memory_size(b200vs_index* idx, int64_t* bytes);
int b200vs_is_trained(b200vs_index* idx);
int32_t b200vs_dimension(b200vs_index* idx);

/* Save / Load — vector_index.h:168-170 (own container format, see DESIGN.md; faiss/hnswlib file
 * compatibility is SURVEY §8(f)-4, not built). */
int b200vs_save(b200vs_index* idx, const char* path);
int b200vs_load(b200vs_index* idx, const char* path);

/* Export the inverted lists in list-major order (list l owns rows [list_off[l], list_off[l+1])) so a CPU
 * implementation can search the identical index.  Any output pointer may be NULL.  Flat: nlist = 1.  Binary indexes
 * export their rows through `codes` [count, dim / 8] (`vectors` is not written; b200vs_export_list takes vectors = NULL). */
int b200vs_export_lists(b200vs_index* idx, int64_t* list_off /*[nlist+1]*/, float* vectors /*[count,dim]*/,
                        uint8_t* codes /*[count,pq_m]*/, int64_t* ids /*[count]*/);

/* One inverted list (live rows only, stored order): writes up to `cap` rows into vectors [cap, dim] / ids [cap] (either may
 * be NULL) and the list's live row count into *count.  Lets a checker rebuild exactly the lists a query probes without
 * copying a 77 GB shard to the host. */
int b200vs_export_list(b200vs_index* idx, int32_t list, int64_t cap, float* vectors, int64_t* ids, int64_t* count);

/* k-way merge of per-shard top-k, the engine's analogue of VectorIndexWrapper::MergeSearchResults
 * (src/vector/vector_index.cc:1056-1108).  parts_* are DEVICE arrays [nparts, nq, k] (API-semantics
 * distances ascending, id -1 padded) e.g. the output of one ncclAllGather; out_* DEVICE [nq,k]. */
int b200vs_merge_topk_device(int32_t device, int32_t nparts, int64_t nq, int32_t k, const float* parts_dist,
                             const int64_t* parts_ids, float* out_dist, int64_t* out_ids, void* stream);

/* List-sharded multi-GPU building blocks (IVF_FLAT): every rank holds all centroids but owns only some lists.
 * b200vs_coarse_device ranks the centroid rows [list_begin, list_end) only (this rank's share of the coarse work):
 * out_lists = GLOBAL list ids, out_score = the ranking score (L2 distance, or -ip: exact and ascending, so no
 * rounding can reorder ties), both [nq, nprobe] in (score, list id) order, so the per-rank
 * results can be all-gathered and merged with b200vs_merge_topk_device into the global top-nprobe
 * (= faiss quantizer->search(nq, x, nprobe), vector_index_ivf_flat.cc:247-251).  b200vs_search_probes_device then scans
 * the probed lists this rank owns for those (caller-supplied) probes. */
int b200vs_coarse_device(b200vs_index* idx, int64_t nq, const float* xq_dev, int32_t nprobe, int32_t list_begin, int32_t list_end,
                         float* out_score_dev, int64_t* out_lists_dev, void* stream);
int b200vs_search_probes_device(b200vs_index* idx, int64_t nq, const float* xq_dev, int32_t k, const int64_t* probes_dev, int32_t nprobe,
                                const b200vs_search_params* sp, float* out_dist_dev, int64_t* out_ids_dev, void* stream);

/* ---- List-sharded multi-GPU deployment (SURVEY.md 8e; one process per GPU) ----------------------------------------------
 * One LOGICAL IVF_FLAT index over `world` GPUs of one box: the centroid table is replicated, rank r owns the inverted lists
 * [r * ceil(nlist / world), (r + 1) * ceil(nlist / world)) (b200vs_shard_list_range) — equivalently Raft regions mapped to
 * GPUs (src/vector/vector_index.h:54-55).  Every entry point below is COLLECTIVE: all ranks call it with the same
 * arguments (except the rows each rank contributes to add).  Communication is NCCL over NVLink, resolved at run time
 * (dlopen libnccl.so.2; override with B200VS_NCCL_LIB), one communicator per batch in flight.
 *   shard_unique_id : rank 0 creates the rendezvous blob; the host passes it to the other ranks out of band (dingo-store: RPC)
 *   shard_create    : wraps an (untrained or trained, still empty) IVF_FLAT index created with the GLOBAL nlist; `lanes` =
 *                     batches that may be in flight (<= 0: 2)
 *   shard_train     : distributed training — each rank clusters its rows into nlist / world centroids, one all-gather
 *   shard_broadcast_state : or: replicate rank `root`'s trained state (b200vs_train / b200vs_set_trained_state there)
 *   shard_add[_device]    : each rank passes the rows it holds; rows travel to the owner of their nearest centroid's list
 *   shard_plan_add_device / shard_plan_commit : optional first pass of a bulk build (assignment only) that pre-sizes every
 *                     owned list in one allocation — a 77 GB shard cannot afford list relocation or arena re-allocation
 *   shard_search[_device] : all ranks pass the SAME batch.  Coarse quantiser on the rank's slice of the batch + all-gather of
 *                     the probe table; tile scan of the owned probed lists; ONE all-gather of the packed per-shard top-k
 *                     (16-byte (distance, id) records) + k-way merge (VectorIndexWrapper::MergeSearchResults,
 *                     src/vector/vector_index.cc:1056-1108): every rank returns the full merged [nq, k].  The host-pointer
 *                     variant uploads only the rank's slice of the batch and all-gathers the queries over NVLink.
 *                     seq = batch sequence number: 0, 1, 2, ... the same on every rank, each used exactly once.  Batches are
 *                     enqueued in seq order on every rank (concurrent caller threads simply take turns; the GPU work of
 *                     up to `lanes` batches still overlaps), batch seq uses communicator seq % lanes.  seq < 0 = "next in
 *                     call order" for single-threaded callers.  Results equal b200vs_search on the unsharded index. */
#define B200VS_SHARD_ID_BYTES 128
typedef struct b200vs_shard b200vs_shard;
int b200vs_shard_unique_id(uint8_t id[B200VS_SHARD_ID_BYTES]);
int b200vs_shard_create(b200vs_index* idx, int32_t rank, int32_t world, const uint8_t id[B200VS_SHARD_ID_BYTES], int32_t lanes,
                        b200vs_shard** out);
void b200vs_shard_destroy(b200vs_shard* shard);
int b200vs_shard_list_range(b200vs_shard* shard, int32_t rank, int32_t* begin, int32_t* end);
int b200vs_shard_train(b200vs_shard* shard, int64_t n, const float* x);
int b200vs_shard_broadcast_state(b200vs_shard* shard, int32_t root);
int b200vs_shard_add(b200vs_shard* shard, int64_t n, const float* x, const int64_t* ids);
int b200vs_shard_add_device(b200vs_shard* shard, int64_t n, const float* x_dev, const int64_t* ids_dev);
/* collective Delete: every rank passes the same ids; *n_removed = rows removed over all ranks; EVECTOR_INVALID when no rank held
 * any of them (vector_index_ivf_flat.cc:180-184).  shard_add* appends (IndexIVFFlat::add_with_ids); an Upsert is this call (a
 * not-found status ignored) followed by shard_add*. */
int b200vs_shard_remove_ids(b200vs_shard* shard, int64_t n, const int64_t* ids, int64_t* n_removed);
int b200vs_shard_plan_add_device(b200vs_shard* shard, int64_t n, const float* x_dev);
int b200vs_shard_plan_commit(b200vs_shard* shard);
int b200vs_shard_search(b200vs_shard* shard, int64_t seq, int64_t nq, const float* xq, int32_t k, const b200vs_search_params* sp,
                        float* out_dist, int64_t* out_ids);
int b200vs_shard_search_device(b200vs_shard* shard, int64_t seq, int64_t nq, const float* xq_dev, int32_t k,
                               const b200vs_search_params* sp, float* out_dist_dev, int64_t* out_ids_dev, void* stream);

/* Device-pointer write path of a single index (IVF_FLAT): rows and ids already on the index's device.  lists_dev (nullable)
 * = the inverted list of every row when the caller has already assigned them (b200vs_assign_device); returns when done. */
int b200vs_add_with_ids_device(b200vs_index* idx, int64_t n, const float* x_dev, const int64_t* ids_dev, const int64_t* lists_dev,
                               int upsert);
/* faiss quantizer->assign: nearest centroid of every (raw) row, out_lists_dev[n]; synchronous. */
int b200vs_assign_device(b200vs_index* idx, int64_t n, const float* x_dev, int64_t* out_lists_dev);
/* Pre-size every inverted list of an EMPTY trained IVF_FLAT index (rows_per_list[nlist], host) in one arena allocation. */
int b200vs_reserve_lists(b200vs_index* idx, const int64_t* rows_per_list, int32_t nlist);

/* Pairwise distance matrix, the UtilService path UtilServiceImpl::VectorCalcDistance (src/server/util_service.cc:45-92)
 * -> VectorIndexUtils::CalcDistanceEntry / CalcDistanceCore (src/vector/vector_index_utils.cc:48-124).  Host pointers,
 * row-major left [nl, dim], right [nr, dim]; out [nl, nr]: L2 -> squared L2, IP -> 1 - ip, COSINE -> 1 - ip of the
 * normalised copies (algorithm FAISS: NormalizeVectorForFaiss :480-491; HNSWLIB: NormalizeVectorForHnsw :493-500).
 * left_out / right_out (nullable) = what is_return_normlize returns: the normalised copies for COSINE, else the inputs. */
enum { B200VS_ALGORITHM_FAISS = 1, B200VS_ALGORITHM_HNSWLIB = 2 };  /* pb::index::AlgorithmType */
int b200vs_calc_distance(int32_t device, int32_t algorithm, b200vs_metric metric, int32_t dim, int64_t nl, const float* left,
                         int64_t nr, const float* right, float* out, float* left_out, float* right_out);

/* ---- Binary (Hamming) indexes: B200VS_BINARY_FLAT / B200VS_BINARY_IVF_FLAT ------------------------------------------------
 * Rows are packed bits, dim / 8 bytes each, row-major; bit b of a row is bit (b % 8) of byte b / 8 (LSB first).  Distances
 * are popcount(a XOR b) as float (vector_index_utils.cc:640-648), ascending, ties -> smaller id; missing hits are padded
 * with id = -1, dist = 0.  Add / Upsert / Delete / filters / topk <= 0 follow the float Flat and IVF-Flat contracts above.
 * A float entry point (b200vs_train, b200vs_add_with_ids, b200vs_search*, b200vs_range_search) on a binary index, or a
 * binary one on a float index, returns EVECTOR_INVALID.  Binary calls are not coalesced.
 *   train_binary   : IndexBinaryIVF::train — bits expanded to +-1 floats, L2 k-means (niter 10, <= 256 points per centroid,
 *                    seed 1234), centroids thresholded back to bits (> 0 -> 1); fewer rows than nlist -> nlist = 1.  Flat: no-op.
 *                    The sample (min(n, nlist * 256) rows) is expanded to floats on host and device: more than 16 GiB of
 *                    floats (e.g. nlist 2048 at 8192 bits or more) -> EILLEGAL_PARAMETERS.
 *   range_search_binary : hits with distance < (int)radius (faiss binary range_search takes an int radius). */
int b200vs_train_binary(b200vs_index* idx, int64_t n, const uint8_t* x);
int b200vs_add_binary_with_ids(b200vs_index* idx, int64_t n, const uint8_t* x, const int64_t* ids, int upsert);
int b200vs_search_binary(b200vs_index* idx, int64_t nq, const uint8_t* xq, int32_t k, const b200vs_search_params* sp,
                         float* out_dist, int64_t* out_ids);
int b200vs_search_binary_device(b200vs_index* idx, int64_t nq, const uint8_t* xq_dev, int32_t k, const b200vs_search_params* sp,
                                float* out_dist_dev, int64_t* out_ids_dev, void* stream);
int b200vs_range_search_binary(b200vs_index* idx, int64_t nq, const uint8_t* xq, float radius, int32_t max_results,
                               const b200vs_search_params* sp, float* out_dist, int64_t* out_ids, int32_t* out_counts);
/* Pairwise Hamming matrix (VectorCalcDistance, METRIC_TYPE_HAMMING, utils.cc:146-149, :333-356): left [nl, dim_bits / 8],
 * right [nr, dim_bits / 8] host bytes; out [nl, nr]. */
int b200vs_calc_distance_binary(int32_t device, int32_t dim_bits, int64_t nl, const uint8_t* left, int64_t nr, const uint8_t* right,
                                float* out);

/* Streaming brute-force search over vectors that are NOT in an index: VectorReader::BruteForceSearch
 * (src/vector/vector_reader.cc:1873-2048), which scans the region's vector column family, builds a temporary Flat
 * index per FLAGS_vector_index_bruteforce_batch_count vectors, searches it and keeps per-query top-k heaps.
 *   scan_begin : the queries (host, raw; COSINE is normalised inside), k, optional id filters (copied);
 *   scan_push  : one tile of scanned vectors + ids (host; any size, ids unique inside a tile) -> tile top-k on the GPU,
 *                merged into the running top-k with the (distance, id) rule;
 *   scan_finish: running top-k -> out_dist / out_ids [nq, k] (API distances ascending, -1 padded); frees the handle.
 * The result equals one Flat search over the concatenation of all tiles. */
typedef struct b200vs_scan b200vs_scan;
int b200vs_scan_begin(int32_t device, b200vs_metric metric, int32_t dim, int64_t nq, const float* xq, int32_t k,
                      const b200vs_search_params* sp, b200vs_scan** out);
int b200vs_scan_push(b200vs_scan* scan, int64_t n, const float* x, const int64_t* ids);
int b200vs_scan_finish(b200vs_scan* scan, float* out_dist, int64_t* out_ids);
void b200vs_scan_abort(b200vs_scan* scan);

/* Counters of the last search on this index: [0] kernels launched, [1] queries served by the tensor-core
 * candidate pass, [2] queries that failed certification and were re-run on the exact path; with profiling on
 * (b200vs_set_profiling) also [3] device time of the dominant list-scan kernel in ns (CUDA events on the launch
 * stream), [4] rows in the distinct probed lists, [5] distinct probed lists, [6] work items of the tile scan,
 * [7] its tensor-core work (128-row tiles x padded query columns).  Profiling synchronises the stream
 * inside the call: never leave it on in a timed run. */
int b200vs_last_search_stats(b200vs_index* idx, int64_t stats[8]);
/* With profiling on: device milliseconds (CUDA events on the launch stream) the last search spent in each phase of the
 * IVF tile path: [0] coarse prep, [1] coarse scan, [2] coarse select + exact re-score, [3] work planning + query
 * gather, [4] sample pass, [5] thresholds, [6] list scan (capture), [7] final select + exact re-score, [8] exact
 * fallback for uncertified queries, [9] other, [10] collectives of a sharded search (b200vs_shard_search*), [11] pack + merge of
 * the per-shard top-k.  Unused slots are 0. */
int b200vs_last_phase_times(b200vs_index* idx, float ms[16]);
int b200vs_set_profiling(b200vs_index* idx, int on);

const char* b200vs_last_error(void);
const char* b200vs_version(void);

#ifdef __cplusplus
}
#endif
#endif /* B200VS_H_ */

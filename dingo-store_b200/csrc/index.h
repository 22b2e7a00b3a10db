// index.h — host-side index objects of libb200vs (device memory owners + search orchestration).
//
// One object per dingo-store vector index (= per Raft region, src/vector/vector_index.h:54-55).  These are
// the B200 replacements of the faiss / hnswlib objects the reference plugins own
// (index_id_map2_ flat.cc:98, index_ ivf_flat.cc:809-816, raw_ivf_pq.cc:554-564, hnsw_index_ hnsw.cc:181).
#pragma once
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <cstdint>
#include <cstring>
#include <mutex>
#include <shared_mutex>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/b200vs.h"
#include "common.cuh"

namespace b200vs {

extern thread_local std::string g_last_error;
struct StatusError {
  int code;
  std::string msg;
};
[[noreturn]] inline void fail(int code, const std::string& m) { throw StatusError{code, m}; }

template <class T>
struct DevBuf {
  T* p = nullptr;
  size_t cap = 0;  // elements
  DevBuf() = default;
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  ~DevBuf() { if (p) cudaFree(p); }
  void free() { if (p) cudaFree(p); p = nullptr; cap = 0; }
  // grow to >= n elements; keeps the first `keep` elements (copied on `s`)
  void reserve(size_t n, size_t keep, cudaStream_t s) {
    if (n <= cap) return;
    T* np = nullptr;
    B200VS_CUDA(cudaMalloc(&np, n * sizeof(T)));
    if (keep && p) B200VS_CUDA(cudaMemcpyAsync(np, p, keep * sizeof(T), cudaMemcpyDeviceToDevice, s));
    if (p) { B200VS_CUDA(cudaStreamSynchronize(s)); cudaFree(p); }
    p = np; cap = n;
  }
};

// bump allocator for per-search scratch; reset at the start of every search (searches on one index are
// serialised by gpu_mu and stream-ordered, so reuse is safe)
struct Scratch {
  DevBuf<unsigned char> buf;
  size_t used = 0;
  std::vector<std::pair<void*, size_t>> overflow;  // extra cudaMalloc blocks when buf is too small
  size_t peak_overflow = 0;                        // most overflow bytes alive at once since the last reset
  ~Scratch() { release_overflow(); }
  void release_overflow() { for (auto& o : overflow) cudaFree(o.first); overflow.clear(); }
  size_t overflow_bytes() const { size_t b = 0; for (auto& o : overflow) b += o.second + 256; return b; }
  void reset(cudaStream_t s) {
    peak_overflow = std::max(peak_overflow, overflow_bytes());
    if (peak_overflow) {  // grow the main buffer so the next search fits without overflow blocks
      B200VS_CUDA(cudaStreamSynchronize(s));
      release_overflow();
      size_t want = (buf.cap + peak_overflow) * 3 / 2;
      peak_overflow = 0;
      buf.free();
      buf.reserve(want, 0, s);
    }
    used = 0;
  }
  template <class T>
  T* alloc(size_t n) {
    size_t bytes = (n * sizeof(T) + 255) / 256 * 256;
    if (used + bytes <= buf.cap) { T* r = reinterpret_cast<T*>(buf.p + used); used += bytes; return r; }
    void* p = nullptr;
    B200VS_CUDA(cudaMalloc(&p, bytes));
    overflow.emplace_back(p, bytes);
    return reinterpret_cast<T*>(p);
  }
  // scoped reuse inside one operation (chunk loops): everything allocated after mark() is handed back by release().
  // Overflow blocks taken in between are freed (cudaFree waits for the device), so a loop over many chunks holds one
  // chunk's worth of memory, not the sum.
  struct Mark { size_t used, nover; };
  Mark mark() const { return Mark{used, overflow.size()}; }
  void release(const Mark& m) {
    peak_overflow = std::max(peak_overflow, overflow_bytes());
    while (overflow.size() > m.nover) { cudaFree(overflow.back().first); overflow.pop_back(); }
    used = m.used;
  }
};

// A lane = one in-flight search: its own scratch arena, serialised by its own mutex, stream-ordered.  Several lanes let
// concurrent callers (the reference issues searches from a 16-thread pool, src/server/server.cc:868-873) overlap on the
// GPU: the small kernels of one batch run under the HBM-bound list scan of another.  A lane that moves to another
// stream is ordered behind its previous search with an event (device-side wait, the host never blocks).
struct Lane {
  Scratch s;
  std::mutex mu;
  std::atomic<cudaStream_t> last{nullptr};  // stream of the lane's previous search
  cudaStream_t own = nullptr;               // lane-owned stream for host-pointer / NULL-stream calls
  cudaEvent_t done = nullptr;               // recorded behind the lane's latest search
  std::atomic<bool> done_valid{false};
  unsigned long long tick = 0;              // last use (lane_pick_mu), for least-recently-used hand-out
};
constexpr int kLanes = 8;

// Request coalescing for host-pointer searches (SURVEY 8b: "b200vs_search internally coalesces concurrent callers").  The
// unchanged reference caller slices every batch into single-query tasks on a 16-thread pool (src/vector/vector_index.cc:54,
// :244-271), so the plugin sees many concurrent nq = 1 calls.  Callers queue here; the one that finds no leader active
// becomes the leader, takes every compatible pending request (same k / nprobe / efsearch / exact_only, no id filters) and
// runs them as ONE batch — large enough batches reach the tensor-core tile path — then hands the results back.
struct CoalesceReq {
  int64_t nq = 0;
  const float* xq = nullptr;
  int k = 0;
  b200vs_search_params sp{};
  float* out_dist = nullptr;
  int64_t* out_ids = nullptr;
  int rc = 0;
  std::string err;
  bool done = false;
};
struct Coalescer {
  std::mutex mu;
  std::condition_variable cv;
  std::vector<CoalesceReq*> pending;
  bool busy = false;
  std::atomic<int> enabled{1};
  std::atomic<int64_t> batches{0}, requests{0};  // statistics: leader batches run / requests served through them
};

struct SearchCtx {  // resolved per-search parameters, device filter included
  int nprobe = 0;
  int efsearch = 0;
  int exact_only = 0;
  int has_range = 0, negate = 0;
  long long rmin = 0, rmax = 0;
  const long long* sorted_ids_dev = nullptr;
  long long n_ids = 0;
  bool has_filter() const { return has_range || sorted_ids_dev; }
};

struct IndexBase {
  b200vs_type type;
  b200vs_metric metric;
  int dim;
  int device;
  b200vs_params params;
  cudaStream_t stream = nullptr;
  cudaStream_t last_stream = nullptr;
  std::shared_mutex rw;  // readers = searches, writers = add/remove/train (reference RWLock)
  std::mutex gpu_mu;     // writers / maintenance (they also hold rw exclusively)
  Lane lanes[kLanes];
  Coalescer coalescer;
  std::atomic<unsigned> lane_rr{0};
  std::mutex lane_pick_mu;
  unsigned long long lane_tick = 0;
  static thread_local Lane* tl_lane;       // the calling thread's active lane (set by LaneGuard)
  static thread_local IndexBase* tl_owner;
  Lane& cur() { return (tl_owner == this && tl_lane) ? *tl_lane : lanes[0]; }
  // wait for the asynchronous work of every earlier search (device-pointer searches return before the GPU is done);
  // writers call it before touching index memory or the lane-0 scratch
  void quiesce() { for (auto& l : lanes) if (l.done_valid.load()) cudaEventSynchronize(l.done); }
  struct ScratchProxy {  // `ix->scratch.alloc<T>(n)` resolves to the calling thread's lane
    IndexBase* ix;
    template <class T> T* alloc(size_t n) { return ix->cur().s.alloc<T>(n); }
    void reset(cudaStream_t st) { ix->cur().s.reset(st); }
    Scratch::Mark mark() { return ix->cur().s.mark(); }
    void release(const Scratch::Mark& m) { ix->cur().s.release(m); }
  } scratch{this};
  // counters of the LAST search; several lanes may search at once, so they are relaxed atomics (the values of two
  // overlapping searches interleave — they are diagnostics — but there is no data race)
  std::atomic<int64_t> stats[8] = {};
  // profiling only (one caller at a time): CUDA-event marks between the phases of a search, b200vs_last_phase_times
  enum Phase { PH_COARSE_PREP = 0, PH_COARSE_SCAN, PH_COARSE_FINAL, PH_PLAN, PH_SAMPLE, PH_TAU, PH_CAPTURE, PH_FINAL, PH_FALLBACK, PH_OTHER, PH_COMM, PH_MERGE, PH_COUNT };
  float phase_ms[PH_COUNT] = {0};
  std::vector<std::pair<int, cudaEvent_t>> phase_marks;
  void phase(int id, cudaStream_t s) {  // "phase id starts here"
    if (!profiling) return;
    cudaEvent_t e = nullptr;
    if (cudaEventCreate(&e) != cudaSuccess) return;
    cudaEventRecord(e, s);
    phase_marks.emplace_back(id, e);
  }
  void phases_finish(cudaStream_t s) {
    if (phase_marks.empty()) return;
    phase(-1, s);
    cudaEventSynchronize(phase_marks.back().second);
    for (size_t i = 0; i + 1 < phase_marks.size(); ++i) {
      float ms = 0.f;
      if (phase_marks[i].first >= 0 && cudaEventElapsedTime(&ms, phase_marks[i].second, phase_marks[i + 1].second) == cudaSuccess)
        phase_ms[phase_marks[i].first] += ms;
    }
    for (auto& m : phase_marks) cudaEventDestroy(m.second);
    phase_marks.clear();
  }
  void reset_stats() { for (auto& v : stats) v.store(0, std::memory_order_relaxed); if (profiling) for (auto& v : phase_ms) v = 0.f; }
  bool profiling = false;  // b200vs_set_profiling: time the dominant scan kernel with CUDA events
  bool loading = false;    // Load(): rows come back exactly as stored (already normalised for cosine)
  virtual int export_nlist() const { return 1; }

  IndexBase(b200vs_type t, b200vs_metric m, int d, const b200vs_params& p);
  virtual ~IndexBase();
  void set_device() const { B200VS_CUDA(cudaSetDevice(device)); }
  bool ip_like() const { return metric == B200VS_IP || metric == B200VS_COSINE; }

  virtual void train(int64_t n, const float* x) { (void)n; (void)x; }
  virtual bool is_trained() const { return true; }
  virtual void set_state(const void* blob, size_t len) { (void)blob; (void)len; fail(B200VS_EVECTOR_NOT_SUPPORT, "no trained state for this index type"); }
  virtual int64_t get_state(void* blob, size_t cap) { (void)blob; (void)cap; return 0; }
  virtual void add(int64_t n, const float* x, const int64_t* ids, bool upsert) = 0;
  virtual int64_t remove(int64_t n, const int64_t* ids) = 0;
  virtual void clear() { fail(B200VS_EVECTOR_NOT_SUPPORT, "clear is only implemented for FLAT"); }  // drop every row, keep the buffers
  // device-pointer search on stream s; scratch already reset; q is RAW (normalise inside for cosine)
  virtual void search_dev(int64_t nq, const float* xq, int k, const SearchCtx& sc, float* out_dist, long long* out_ids,
                          cudaStream_t s) = 0;
  virtual void range_search_dev(int64_t nq, const float* xq, float radius, int max_results, const SearchCtx& sc,
                                float* out_dist, long long* out_ids, int* out_counts, cudaStream_t s) {
    (void)nq; (void)xq; (void)radius; (void)max_results; (void)sc; (void)out_dist; (void)out_ids; (void)out_counts; (void)s;
    fail(B200VS_EVECTOR_NOT_SUPPORT, "range search not supported");
  }
  // list-sharded multi-GPU building blocks (IVF types): coarse quantiser over centroid rows [c0, c1) only, and the list
  // scan for caller-supplied (merged) probes
  virtual void coarse_range_dev(int64_t nq, const float* xq, int nprobe, int c0, int c1, float* out_score, long long* out_lists, cudaStream_t s) {
    (void)nq; (void)xq; (void)nprobe; (void)c0; (void)c1; (void)out_score; (void)out_lists; (void)s;
    fail(B200VS_EVECTOR_NOT_SUPPORT, "coarse quantiser only exists for IVF_FLAT");
  }
  virtual void search_probes_dev(int64_t nq, const float* xq, int k, const long long* probes, int nprobe, const SearchCtx& sc, float* od,
                                 long long* oi, cudaStream_t s) {
    (void)nq; (void)xq; (void)k; (void)probes; (void)nprobe; (void)sc; (void)od; (void)oi; (void)s;
    fail(B200VS_EVECTOR_NOT_SUPPORT, "probe-driven search only exists for IVF_FLAT");
  }
  // ---- device-pointer write path and the building blocks of a list-sharded deployment (shard.cu); IVF_FLAT only ----
  // rows / ids already on this device.  lists_dev (nullable) = the inverted list of every row, decided by the caller;
  // prepared = store the rows exactly as given (cosine rows are already normalised).
  virtual void add_dev(int64_t n, const float* x_dev, const long long* ids_dev, const long long* lists_dev, bool upsert, bool prepared) {
    (void)n; (void)x_dev; (void)ids_dev; (void)lists_dev; (void)upsert; (void)prepared;
    fail(B200VS_EVECTOR_NOT_SUPPORT, "device-pointer add only exists for IVF_FLAT");
  }
  // nearest-centroid assignment of prepared rows (faiss quantizer->assign): out_lists_dev[n], on stream s (a lane must be held)
  virtual void assign_lists_dev(int64_t n, const float* x_dev, long long* out_lists_dev, cudaStream_t s) {
    (void)n; (void)x_dev; (void)out_lists_dev; (void)s;
    fail(B200VS_EVECTOR_NOT_SUPPORT, "list assignment only exists for IVF_FLAT");
  }
  // pre-size every inverted list (rows_per_list[nlist]) in ONE arena allocation: bulk builds of large shards never
  // relocate a list or re-allocate the arena (a 77 GB shard cannot afford a 2x peak)
  virtual void reserve_lists(const int64_t* rows_per_list, int nlist) {
    (void)rows_per_list; (void)nlist;
    fail(B200VS_EVECTOR_NOT_SUPPORT, "list reservation only exists for IVF_FLAT");
  }
  virtual int nlist_now() const { return 1; }
  // probe table (set semantics, order unspecified) of prepared queries into a caller buffer
  virtual void coarse_probes_dev(int64_t nq, const float* q_prepared, int nprobe, long long* out_lists, cudaStream_t s) {
    (void)nq; (void)q_prepared; (void)nprobe; (void)out_lists; (void)s;
    fail(B200VS_EVECTOR_NOT_SUPPORT, "coarse quantiser only exists for IVF_FLAT");
  }
  // search_probes_dev on queries that are already prepared (normalised for cosine)
  virtual void search_probes_prepared_dev(int64_t nq, const float* q_prepared, int k, const long long* probes, int nprobe, const SearchCtx& sc,
                                          float* od, long long* oi, cudaStream_t s) {
    (void)nq; (void)q_prepared; (void)k; (void)probes; (void)nprobe; (void)sc; (void)od; (void)oi; (void)s;
    fail(B200VS_EVECTOR_NOT_SUPPORT, "probe-driven search only exists for IVF_FLAT");
  }
  virtual int resolve_nprobe_api(const SearchCtx& sc) const { (void)sc; return 1; }

  // ---- binary (Hamming) indexes: rows are dim / 8 bytes.  A float index rejects binary vectors (ExtractVectorValue's
  // value-type check, vector_index_utils.cc:502-530) ----
  bool binary() const { return type == B200VS_BINARY_FLAT || type == B200VS_BINARY_IVF_FLAT; }
  virtual void train_binary(int64_t n, const uint8_t* x) { (void)n; (void)x; fail(B200VS_EVECTOR_INVALID, "binary vectors given to a float index"); }
  virtual void add_binary(int64_t n, const uint8_t* x, const int64_t* ids, bool upsert) {
    (void)n; (void)x; (void)ids; (void)upsert;
    fail(B200VS_EVECTOR_INVALID, "binary vectors given to a float index");
  }
  // xq_dev: [nq, dim / 8] device bytes; scratch already reset
  virtual void search_binary_dev(int64_t nq, const uint8_t* xq_dev, int k, const SearchCtx& sc, float* out_dist, long long* out_ids, cudaStream_t s) {
    (void)nq; (void)xq_dev; (void)k; (void)sc; (void)out_dist; (void)out_ids; (void)s;
    fail(B200VS_EVECTOR_INVALID, "binary vectors given to a float index");
  }
  virtual void range_search_binary_dev(int64_t nq, const uint8_t* xq_dev, float radius, int max_results, const SearchCtx& sc,
                                       float* out_dist, long long* out_ids, int* out_counts, cudaStream_t s) {
    (void)nq; (void)xq_dev; (void)radius; (void)max_results; (void)sc; (void)out_dist; (void)out_ids; (void)out_counts; (void)s;
    fail(B200VS_EVECTOR_INVALID, "binary vectors given to a float index");
  }

  virtual void reconstruct(int64_t n, const int64_t* ids, float* out, uint8_t* found) {
    (void)n; (void)ids; (void)out; (void)found;
    fail(B200VS_EVECTOR_NOT_SUPPORT, "reconstruct is implemented for HNSW and FLAT");
  }
  virtual int sub_type() const { return (int)type; }
  virtual int64_t count() const = 0;
  virtual int64_t deleted_count() const { return 0; }
  virtual int64_t memory_size() const = 0;
  virtual void export_lists(int64_t* list_off, float* vectors, uint8_t* codes, int64_t* ids) = 0;
  virtual int64_t export_list(int list, int64_t cap, float* vectors, int64_t* ids) {
    (void)list; (void)cap; (void)vectors; (void)ids;
    fail(B200VS_EVECTOR_NOT_SUPPORT, "single-list export only exists for IVF_FLAT");
  }
  virtual void save(const std::string& path);
  virtual void load(const std::string& path);

  // helpers shared by the index types
  const float* prepare_queries(int64_t nq, const float* xq_dev, cudaStream_t s);  // cosine -> normalised copy
  void launch_count(int n = 1) { stats[0] += n; }
};

// Shared (reader) hold of an index's rw lock that composes: an operation made of several locked steps (Save = count, then
// trained state, then list export) takes it once at the top, the steps' own guards then see the hold and do not lock again
// (re-acquiring a std::shared_mutex in shared mode can dead-lock behind a queued writer, and releasing it between the steps
// lets an add grow the index past the buffers sized from the earlier count).
struct RwSharedGuard {
  static thread_local const IndexBase* tl_held;
  const IndexBase* prev;
  std::shared_lock<std::shared_mutex> lk;
  explicit RwSharedGuard(IndexBase* ix) : prev(tl_held) {
    if (tl_held != ix) { lk = std::shared_lock<std::shared_mutex>(ix->rw); tl_held = ix; }
  }
  ~RwSharedGuard() { tl_held = prev; }
  RwSharedGuard(const RwSharedGuard&) = delete;
  RwSharedGuard& operator=(const RwSharedGuard&) = delete;
};

// RAII: pick a lane for a search on stream `s` (nullptr = a lane-owned stream), lock it, make it the thread's scratch
struct LaneGuard {
  IndexBase* ix;
  Lane* lane;
  IndexBase* prev_owner;
  Lane* prev_lane;
  cudaStream_t stream;
  LaneGuard(IndexBase* ix_, cudaStream_t s);
  ~LaneGuard();
};

}  // namespace b200vs
struct b200vs_index {  // the opaque handle of include/b200vs.h
  b200vs::IndexBase* impl;
};
namespace b200vs {
inline IndexBase* index_impl(b200vs_index* h) {
  if (!h || !h->impl) fail(B200VS_EILLEGAL_PARAMETERS, "null index handle");
  return h->impl;
}

IndexBase* make_flat(b200vs_metric m, int d, const b200vs_params& p);
IndexBase* make_ivf_flat(b200vs_metric m, int d, const b200vs_params& p);
IndexBase* make_ivf_pq(b200vs_metric m, int d, const b200vs_params& p);
IndexBase* make_hnsw(b200vs_metric m, int d, const b200vs_params& p);
IndexBase* make_binary(b200vs_type t, int d, const b200vs_params& p);  // BINARY_FLAT / BINARY_IVF_FLAT (binary.cu)
// out[i*nr + j] = popcount(a_i ^ b_j) over dim_bits (VectorCalcDistance, METRIC_TYPE_HAMMING); a, b: packed host rows
void binary_pair_distance(int dim_bits, int64_t nl, const uint8_t* a, int64_t nr, const uint8_t* b, float* out, cudaStream_t s);

// ---- generic exact scan + select driver (scan_kernels.cuh) ----
struct ScanJob {
  bool l2 = true;
  const float* vecs = nullptr;
  const long long* ids = nullptr;
  int d = 0;
  int mode = 0;
  long long n = 0;
  const long long* probes = nullptr;
  int nprobe = 0;
  const long long* list_off = nullptr;
  const int* list_len = nullptr;
  double avg_candidates = 0;  // expected candidates per query (sizing of nsplit)
  const SearchCtx* sc = nullptr;
  bool has_thr = false;
  float thr_raw = 0;  // range search: raw metric threshold (L2: dist < thr ; IP: ip > thr)
  bool dominant = false;  // the list scan of an IVF search: timed when profiling is on
};
// profiling helpers: distinct probed lists / rows of a probe table
void profile_probed(IndexBase* ix, const long long* probes, int64_t n_probes, int nlist, const int* list_len, cudaStream_t s);
struct ScopedKernelTimer {  // CUDA events on the launching stream; synchronises in the destructor
  IndexBase* ix; cudaStream_t s; cudaEvent_t e0 = nullptr, e1 = nullptr; bool on;
  ScopedKernelTimer(IndexBase* ix_, cudaStream_t s_, bool on_) : ix(ix_), s(s_), on(on_) {
    if (!on) return;
    B200VS_CUDA(cudaEventCreate(&e0)); B200VS_CUDA(cudaEventCreate(&e1)); B200VS_CUDA(cudaEventRecord(e0, s));
  }
  void stop() {
    if (!on || !e0) return;
    cudaEventRecord(e1, s); cudaEventSynchronize(e1);
    float ms = 0; cudaEventElapsedTime(&ms, e0, e1);
    ix->stats[3] += (int64_t)(ms * 1e6);
    cudaEventDestroy(e0); cudaEventDestroy(e1); e0 = e1 = nullptr;
  }
  ~ScopedKernelTimer() { stop(); }
};
// results: out_dist (API), out_raw (raw metric), out_ids, out_counts — any but out_ids may be null
void run_scan(IndexBase* ix, const ScanJob& job, int64_t nq, const float* queries, int k, float* out_dist,
              float* out_raw, long long* out_ids, int* out_counts, cudaStream_t s);

void launch_normalize_faiss(float* x, int64_t n, int d, cudaStream_t s);
void launch_normalize_hnsw(const float* x, float* out, int64_t n, int d, cudaStream_t s);
void launch_scatter_rows(const float* src, const long long* src_ids, const long long* slots, int64_t n, int d,
                         float* vecs, long long* ids, float* norms, float* row_norms, cudaStream_t s);
void launch_move_rows(const float* svecs, const long long* sids, const float* snorms, const long long* src_rows,
                      const long long* dst_rows, int64_t n, int d, float* dvecs, long long* dids, float* dnorms,
                      cudaStream_t s);
void launch_set_ids(long long* ids, const long long* slots, int64_t n, long long value, cudaStream_t s);
void launch_iota(long long* p, int64_t n, cudaStream_t s);
void launch_negate(float* p, int64_t n, cudaStream_t s);
// out[i*nr + j] = L2 ? ||a_i - b_j||^2 : 1 - <a_i, b_j>, reference summation order (VectorCalcDistance)
void launch_pair_distance(bool l2, const float* a, int64_t nl, const float* b, int64_t nr, int d, float* out, cudaStream_t s);
void launch_merge_api(int nparts, int64_t nq, int k, const float* pd, const long long* pi, float* od, long long* oi,
                      cudaStream_t s);

}  // namespace b200vs

// index.cu — IndexBase, FlatIndex, IvfFlatIndex (device-resident replacements of the faiss objects held by
// VectorIndexFlat / VectorIndexIvfFlat, src/vector/vector_index_flat.cc:73-107, vector_index_ivf_flat.cc:805-837).
#include <algorithm>
#include <cstdio>
#include <random>
#include <unordered_set>

#include "index.h"
#include "ivf_common.h"
#include "flat_small.cuh"
#include "tc_scan.cuh"

namespace b200vs {

thread_local std::string g_last_error;
thread_local Lane* IndexBase::tl_lane = nullptr;
thread_local IndexBase* IndexBase::tl_owner = nullptr;
thread_local const IndexBase* RwSharedGuard::tl_held = nullptr;

LaneGuard::LaneGuard(IndexBase* ix_, cudaStream_t s) : ix(ix_), lane(nullptr), prev_owner(IndexBase::tl_owner), prev_lane(IndexBase::tl_lane), stream(s) {
  const bool own = s == nullptr;  // host-pointer / NULL-stream call: runs on the lane's own stream
  {
    std::lock_guard<std::mutex> pick(ix->lane_pick_mu);
    // 1) the lane this stream used last: its scratch is already ordered behind the caller's earlier work
    if (!own)
      for (auto& l : ix->lanes)
        if (l.last.load() == s && l.mu.try_lock()) { lane = &l; break; }
    // 2) a free lane nobody else's stream is attached to: for host-pointer calls the most recently used such lane
    //    (its scratch arena is already sized and hot), else an unused one; failing that, steal the least recently used
    if (!lane) {
      auto rank = [&](Lane& l) -> unsigned long long {
        const cudaStream_t last = l.last.load();
        if (own && last != nullptr && last == l.own) return (1ull << 60) - l.tick;  // warm host-call lane, MRU first
        if (last == nullptr) return 1ull << 61;                                       // never used
        return (1ull << 62) + l.tick;                                                 // attached to a stream: LRU
      };
      for (auto& l : ix->lanes) {
        if (!l.mu.try_lock()) continue;
        if (!lane) lane = &l;
        else if (rank(l) < rank(*lane)) { lane->mu.unlock(); lane = &l; }
        else l.mu.unlock();
      }
    }
    if (lane) lane->tick = ++ix->lane_tick;
  }
  if (!lane) {  // every lane is busy: queue behind one
    lane = &ix->lanes[ix->lane_rr.fetch_add(1) % kLanes];
    lane->mu.lock();
    std::lock_guard<std::mutex> pick(ix->lane_pick_mu);
    lane->tick = ++ix->lane_tick;
  }
  try {
    if (own) {
      if (!lane->own) B200VS_CUDA(cudaStreamCreateWithFlags(&lane->own, cudaStreamNonBlocking));
      stream = lane->own;
    }
    if (lane->last.load() != stream && lane->done_valid.load()) B200VS_CUDA(cudaStreamWaitEvent(stream, lane->done, 0));
    lane->last.store(stream);
    IndexBase::tl_owner = ix;
    IndexBase::tl_lane = lane;
    if (lane->s.buf.cap == 0) {  // first search on this lane: size its arena like the largest warmed-up lane, so it does
      size_t want = 0;            // not go through overflow blocks + consolidation (cudaFree = device-wide stalls)
      for (auto& l : ix->lanes) want = std::max(want, l.s.buf.cap);
      if (want) lane->s.buf.reserve(want, 0, stream);
    }
    lane->s.reset(stream);
  } catch (...) {
    IndexBase::tl_owner = prev_owner;
    IndexBase::tl_lane = prev_lane;
    lane->mu.unlock();
    throw;
  }
}
LaneGuard::~LaneGuard() {
  IndexBase::tl_owner = prev_owner;
  IndexBase::tl_lane = prev_lane;
  if (!lane->done) cudaEventCreateWithFlags(&lane->done, cudaEventDisableTiming);
  if (lane->done && cudaEventRecord(lane->done, stream) == cudaSuccess) lane->done_valid.store(true);
  lane->mu.unlock();
}

IndexBase::IndexBase(b200vs_type t, b200vs_metric m, int d, const b200vs_params& p)
    : type(t), metric(m), dim(d), device(p.device), params(p) {
  set_device();
  B200VS_CUDA(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
  last_stream = stream;
}
IndexBase::~IndexBase() {
  cudaSetDevice(device);
  if (stream) { cudaStreamSynchronize(stream); cudaStreamDestroy(stream); }
  for (auto& l : lanes) {
    if (l.done) { cudaEventSynchronize(l.done); cudaEventDestroy(l.done); }
    if (l.own) { cudaStreamSynchronize(l.own); cudaStreamDestroy(l.own); }
  }
}

const float* IndexBase::prepare_queries(int64_t nq, const float* xq_dev, cudaStream_t s) {
  if (metric != B200VS_COSINE) return xq_dev;
  float* q = scratch.alloc<float>((size_t)nq * dim);
  if (type == B200VS_HNSW) {  // NormalizeVectorForHnsw, vector_index_hnsw.cc:449-452
    launch_normalize_hnsw(xq_dev, q, nq, dim, s);
  } else {                    // NormalizeVectorForFaiss via ExtractVectorValue(normalize_), flat.cc:243
    B200VS_CUDA(cudaMemcpyAsync(q, xq_dev, (size_t)nq * dim * sizeof(float), cudaMemcpyDeviceToDevice, s));
    launch_normalize_faiss(q, nq, dim, s);
  }
  launch_count(1);
  return q;
}

// Save / Load (VectorIndex::Save/Load, src/vector/vector_index.h:168-170; reference: faiss::write_index / read_index at
// vector_index_flat.cc:354,:379 and hnswlib saveIndex at vector_index_hnsw.cc:290).  Own container, not faiss-compatible
// (SURVEY 8f-4): header, trained-state blob, then the live rows in list-major order exactly as stored.
namespace {
struct FileHdr { char magic[8]; int32_t type, metric, dim, nlist; int64_t state_len, count; };
void wr(FILE* f, const void* p, size_t n) { if (n && fwrite(p, 1, n, f) != n) fail(B200VS_EINTERNAL, "short write"); }
void rd(FILE* f, void* p, size_t n) { if (n && fread(p, 1, n, f) != n) fail(B200VS_EINTERNAL, "short read / truncated index file"); }
}  // namespace

void IndexBase::save(const std::string& path) {
  RwSharedGuard hold(this);  // one reader hold across count / trained state / export: no add can slip in between
  const int64_t st_len = get_state(nullptr, 0);
  std::vector<unsigned char> st((size_t)std::max<int64_t>(st_len, 0));
  if (st_len > 0) get_state(st.data(), st.size());
  const int nl = export_nlist();
  const int64_t n = type == B200VS_HNSW ? 0 : count();  // the HNSW blob already carries rows + labels
  const size_t row_bytes = binary() ? (size_t)dim / 8 : (size_t)dim * 4;  // binary rows are dim / 8 bytes (the `codes` export)
  std::vector<int64_t> off(nl + 1, 0), ids((size_t)n);
  std::vector<unsigned char> vec((size_t)n * row_bytes);
  if (n) export_lists(off.data(), binary() ? nullptr : reinterpret_cast<float*>(vec.data()), binary() ? vec.data() : nullptr, ids.data());
  FILE* f = fopen(path.c_str(), "wb");
  if (!f) fail(B200VS_EINTERNAL, "cannot open " + path);
  try {
    FileHdr h;
    memcpy(h.magic, "B2VSIDX1", 8);
    h.type = type; h.metric = metric; h.dim = dim; h.nlist = nl; h.state_len = st_len > 0 ? st_len : 0; h.count = n;
    wr(f, &h, sizeof(h));
    wr(f, st.data(), st.size());
    wr(f, off.data(), off.size() * 8);
    wr(f, ids.data(), ids.size() * 8);
    wr(f, vec.data(), vec.size());
  } catch (...) { fclose(f); throw; }
  fclose(f);
}

void IndexBase::load(const std::string& path) {
  FILE* f = fopen(path.c_str(), "rb");
  if (!f) fail(B200VS_EINTERNAL, "cannot open " + path);
  try {
    FileHdr h;
    rd(f, &h, sizeof(h));
    const size_t row_bytes = binary() ? (size_t)dim / 8 : (size_t)dim * 4;
    if (memcmp(h.magic, "B2VSIDX1", 8) != 0 || h.type != (int)type || h.metric != (int)metric || h.dim != dim)
      fail(B200VS_EINTERNAL, "index file does not match this index (type / metric / dimension)");
    if (count() != 0) fail(B200VS_EINTERNAL, "load into a non-empty index");
    {  // the header's sizes must fit the file before anything is allocated from them
      const long here = ftell(f);
      fseek(f, 0, SEEK_END);
      const long fsize = ftell(f);
      fseek(f, here, SEEK_SET);
      const double need = (double)h.state_len + ((double)h.nlist + 1) * 8 + (double)h.count * (8 + (double)row_bytes);
      if (h.state_len < 0 || h.count < 0 || h.nlist < 0 || h.nlist > (1 << 24) || need > (double)(fsize - here))
        fail(B200VS_EINTERNAL, "corrupt index file (header sizes exceed the file)");
    }
    std::vector<unsigned char> st((size_t)h.state_len);
    rd(f, st.data(), st.size());
    if (h.state_len > 0) set_state(st.data(), st.size());
    std::vector<int64_t> off((size_t)h.nlist + 1), ids((size_t)h.count);
    std::vector<unsigned char> vec((size_t)h.count * row_bytes);
    rd(f, off.data(), off.size() * 8);
    rd(f, ids.data(), ids.size() * 8);
    rd(f, vec.data(), vec.size());
    loading = true;
    try {
      for (int64_t a = 0; a < h.count; a += 32768) {
        const int64_t m = std::min<int64_t>(32768, h.count - a);
        const unsigned char* rows = vec.data() + (size_t)a * row_bytes;
        if (binary()) add_binary(m, rows, ids.data() + a, false);
        else add(m, reinterpret_cast<const float*>(rows), ids.data() + a, false);
      }
    } catch (...) { loading = false; throw; }
    loading = false;
  } catch (...) { fclose(f); throw; }
  fclose(f);
}

void check_batch_ids_unique(int64_t n, const int64_t* ids) {  // CheckVectorIdDuplicated, vector_index_utils.cc:551-561
  std::unordered_set<int64_t> seen;
  seen.reserve((size_t)n * 2);
  for (int64_t i = 0; i < n; ++i)
    if (!seen.insert(ids[i]).second) fail(B200VS_EVECTOR_ID_DUPLICATED, "vector id duplicated: " + std::to_string(ids[i]));
}

// ============================================================================================
// Flat
// ============================================================================================
struct FlatIndex : IndexBase {
  DevBuf<float> vecs;
  DevBuf<long long> ids;
  DevBuf<float> norms;
  int64_t rows = 0;
  std::vector<int64_t> h_ids;
  std::unordered_map<int64_t, int64_t> id2row;
  int64_t ndeleted = 0;
  DevBuf<long long> d_off1;  // the single "list" of a Flat index, for the tile-scan view
  DevBuf<int> d_len1;
  float max_norm = 0.f;

  FlatIndex(b200vs_metric m, int d, const b200vs_params& p) : IndexBase(B200VS_FLAT, m, d, p) {
    d_off1.reserve(1, 0, stream); d_len1.reserve(1, 0, stream);
    B200VS_CUDA(cudaMemsetAsync(d_off1.p, 0, 8, stream));
    B200VS_CUDA(cudaMemsetAsync(d_len1.p, 0, 4, stream));
    B200VS_CUDA(cudaStreamSynchronize(stream));
  }
  void publish_len() {
    const int len = (int)std::min<int64_t>(rows, 0x7fffffff);
    B200VS_CUDA(cudaMemcpyAsync(d_len1.p, &len, 4, cudaMemcpyHostToDevice, stream));
    B200VS_CUDA(cudaStreamSynchronize(stream));
  }
  TcView view() const {
    TcView v;
    v.vecs = vecs.p; v.ids = ids.p; v.norms = norms.p; v.arena_rows = rows; v.list_off = d_off1.p; v.list_len = d_len1.p;
    v.nlist = 1; v.flat = true; v.total_chunks = (rows + TC_CHUNK - 1) / TC_CHUNK; v.max_chunks_per_list = (int)v.total_chunks; v.max_norm = max_norm;
    return v;
  }

  void reserve_rows(int64_t need) {
    if ((size_t)need * dim <= vecs.cap) return;
    int64_t ncap = std::max<int64_t>(need, std::max<int64_t>(1024, (int64_t)(vecs.cap / dim) * 3 / 2));
    vecs.reserve((size_t)ncap * dim, (size_t)rows * dim, stream);
    ids.reserve((size_t)ncap, (size_t)rows, stream);
    norms.reserve((size_t)ncap, (size_t)rows, stream);
  }

  void tombstone(const std::vector<int64_t>& rws) {
    if (rws.empty()) return;
    long long* d_rows = scratch.alloc<long long>(rws.size());
    B200VS_CUDA(cudaMemcpyAsync(d_rows, rws.data(), rws.size() * 8, cudaMemcpyHostToDevice, stream));
    launch_set_ids(ids.p, d_rows, (int64_t)rws.size(), -1, stream);
    B200VS_CUDA(cudaStreamSynchronize(stream));
    for (int64_t r : rws) h_ids[r] = -1;
    ndeleted += (int64_t)rws.size();
  }

  void compact_if_needed() {
    if (ndeleted == 0 || ndeleted * 2 < rows) return;
    std::vector<long long> src, dst;
    src.reserve(rows - ndeleted);
    for (int64_t r = 0; r < rows; ++r) if (h_ids[r] >= 0) src.push_back(r);
    const int64_t live = (int64_t)src.size();
    dst.resize(live);
    for (int64_t i = 0; i < live; ++i) dst[i] = i;
    DevBuf<float> nv; DevBuf<long long> ni; DevBuf<float> nn;
    const int64_t ncap = std::max<int64_t>(1024, live * 5 / 4);
    nv.reserve((size_t)ncap * dim, 0, stream); ni.reserve(ncap, 0, stream); nn.reserve(ncap, 0, stream);
    long long* d_src = scratch.alloc<long long>(live + 1);
    long long* d_dst = scratch.alloc<long long>(live + 1);
    if (live) {
      B200VS_CUDA(cudaMemcpyAsync(d_src, src.data(), live * 8, cudaMemcpyHostToDevice, stream));
      B200VS_CUDA(cudaMemcpyAsync(d_dst, dst.data(), live * 8, cudaMemcpyHostToDevice, stream));
      launch_move_rows(vecs.p, ids.p, norms.p, d_src, d_dst, live, dim, nv.p, ni.p, nn.p, stream);
    }
    B200VS_CUDA(cudaStreamSynchronize(stream));
    std::swap(vecs.p, nv.p); std::swap(vecs.cap, nv.cap);
    std::swap(ids.p, ni.p); std::swap(ids.cap, ni.cap);
    std::swap(norms.p, nn.p); std::swap(norms.cap, nn.cap);
    std::vector<int64_t> nh(live);
    id2row.clear();
    for (int64_t i = 0; i < live; ++i) { nh[i] = h_ids[src[i]]; id2row[nh[i]] = i; }
    h_ids.swap(nh);
    rows = live; ndeleted = 0;
    publish_len();
  }

  // VectorIndexFlat::AddOrUpsert, vector_index_flat.cc:121-162: duplicate ids inside the batch are rejected,
  // pre-existing ids are ALWAYS removed first (add and upsert behave the same), then add_with_ids.
  void add(int64_t n, const float* x, const int64_t* in_ids, bool) override {
    check_batch_ids_unique(n, in_ids);
    std::unique_lock<std::shared_mutex> wl(rw);
    std::lock_guard<std::mutex> gl(gpu_mu);
    set_device();
    quiesce();
    scratch.reset(stream);
    std::vector<int64_t> dead;
    for (int64_t i = 0; i < n; ++i) {
      auto it = id2row.find(in_ids[i]);
      if (it != id2row.end()) { dead.push_back(it->second); id2row.erase(it); }
    }
    tombstone(dead);
    reserve_rows(rows + n);
    float* st = scratch.alloc<float>((size_t)n * dim);
    long long* st_ids = scratch.alloc<long long>(n);
    long long* st_slots = scratch.alloc<long long>(n);
    std::vector<long long> slots(n);
    for (int64_t i = 0; i < n; ++i) slots[i] = rows + i;
    B200VS_CUDA(cudaMemcpyAsync(st, x, (size_t)n * dim * 4, cudaMemcpyHostToDevice, stream));
    B200VS_CUDA(cudaMemcpyAsync(st_ids, in_ids, (size_t)n * 8, cudaMemcpyHostToDevice, stream));
    B200VS_CUDA(cudaMemcpyAsync(st_slots, slots.data(), (size_t)n * 8, cudaMemcpyHostToDevice, stream));
    if (metric == B200VS_COSINE && !loading) launch_normalize_faiss(st, n, dim, stream);  // flat.cc:155 (normalize_)
    float* st_norms = scratch.alloc<float>(n);
    launch_scatter_rows(st, st_ids, st_slots, n, dim, vecs.p, ids.p, norms.p, st_norms, stream);
    max_norm = std::max(max_norm, device_max_norm(this, st_norms, n, stream));
    B200VS_CUDA(cudaStreamSynchronize(stream));
    h_ids.resize(rows + n);
    for (int64_t i = 0; i < n; ++i) { h_ids[rows + i] = in_ids[i]; id2row[in_ids[i]] = rows + i; }
    rows += n;
    publish_len();
    compact_if_needed();
  }

  // streaming brute-force scan (b200vs_scan_*): the tile index is emptied between tiles, buffers are kept
  void clear() override {
    std::unique_lock<std::shared_mutex> wl(rw);
    std::lock_guard<std::mutex> gl(gpu_mu);
    set_device();
    quiesce();
    rows = 0; ndeleted = 0; max_norm = 0.f;
    h_ids.clear(); id2row.clear();
    publish_len();
  }

  // VectorIndexFlat::Delete, vector_index_flat.cc:171-203: unknown ids are ignored (only ids present in
  // rev_map are handed to remove_ids).
  int64_t remove(int64_t n, const int64_t* del) override {
    std::unique_lock<std::shared_mutex> wl(rw);
    std::lock_guard<std::mutex> gl(gpu_mu);
    set_device();
    quiesce();
    scratch.reset(stream);
    std::vector<int64_t> dead;
    for (int64_t i = 0; i < n; ++i) {
      auto it = id2row.find(del[i]);
      if (it != id2row.end()) { dead.push_back(it->second); id2row.erase(it); }
    }
    tombstone(dead);
    compact_if_needed();
    return (int64_t)dead.size();
  }

  ScanJob job(const SearchCtx& sc) const {
    ScanJob j;
    j.l2 = metric == B200VS_L2;
    j.vecs = vecs.p; j.ids = ids.p; j.d = dim; j.mode = 0; j.n = rows; j.sc = &sc;
    return j;
  }

  void search_dev(int64_t nq, const float* xq, int k, const SearchCtx& sc, float* od, long long* oi, cudaStream_t s) override {
    const float* q = prepare_queries(nq, xq, s);
    const TcView v = view();
    if (rows > 0 && tc_eligible(this, v, nq, k, 1, sc)) {
      long long* probes = scratch.alloc<long long>(nq);
      B200VS_CUDA(cudaMemsetAsync(probes, 0, (size_t)nq * 8, s));
      tc_search(this, v, metric == B200VS_L2, nq, q, k, probes, 1, sc, od, oi, s);
      return;
    }
    if (flat_small_eligible(nq, rows, dim, k, sc)) {  // one query per task is the reference's own shape: single-launch path
      flat_small_search(this, metric == B200VS_L2, vecs.p, ids.p, rows, nq, q, k, sc, od, oi, s);
      return;
    }
    run_scan(this, job(sc), nq, q, k, od, nullptr, oi, nullptr, s);
  }

  // VectorIndexFlat::RangeSearch, vector_index_flat.cc:267-323: radius -> 1 - radius for IP / cosine (:282-285);
  // faiss range_search keeps L2 dis < radius, IP ip > radius.
  void range_search_dev(int64_t nq, const float* xq, float radius, int max_results, const SearchCtx& sc, float* od,
                        long long* oi, int* oc, cudaStream_t s) override {
    const float* q = prepare_queries(nq, xq, s);
    ScanJob j = job(sc);
    j.has_thr = true;
    j.thr_raw = ip_like() ? 1.0F - radius : radius;
    run_scan(this, j, nq, q, max_results, od, nullptr, oi, oc, s);
  }

  void reconstruct(int64_t n, const int64_t* in_ids, float* out, uint8_t* found) override {
    RwSharedGuard rl(this);
    std::lock_guard<std::mutex> gl(gpu_mu);
    set_device();
    for (int64_t i = 0; i < n; ++i) {
      auto it = id2row.find(in_ids[i]);
      if (found) found[i] = it != id2row.end() ? 1 : 0;
      if (it != id2row.end())
        B200VS_CUDA(cudaMemcpyAsync(out + (size_t)i * dim, vecs.p + (size_t)it->second * dim, (size_t)dim * 4, cudaMemcpyDeviceToHost, stream));
    }
    B200VS_CUDA(cudaStreamSynchronize(stream));
  }
  int64_t count() const override { return rows - ndeleted; }
  int64_t deleted_count() const override { return ndeleted; }
  int64_t memory_size() const override { return (int64_t)(vecs.cap * 4 + ids.cap * 8 + norms.cap * 4); }

  void export_lists(int64_t* list_off, float* vectors, uint8_t*, int64_t* out_ids) override {
    RwSharedGuard rl(this);
    std::lock_guard<std::mutex> gl(gpu_mu);
    set_device();
    const int64_t live = rows - ndeleted;
    if (list_off) { list_off[0] = 0; list_off[1] = live; }
    std::vector<float> tmp;
    if (vectors && ndeleted) tmp.resize((size_t)rows * dim);
    if (vectors) {
      float* dst = ndeleted ? tmp.data() : vectors;
      B200VS_CUDA(cudaMemcpy(dst, vecs.p, (size_t)rows * dim * 4, cudaMemcpyDeviceToHost));
    }
    int64_t o = 0;
    for (int64_t r = 0; r < rows; ++r) {
      if (h_ids[r] < 0) continue;
      if (out_ids) out_ids[o] = h_ids[r];
      if (vectors && ndeleted) memcpy(vectors + (size_t)o * dim, tmp.data() + (size_t)r * dim, (size_t)dim * 4);
      ++o;
    }
  }
};

IndexBase* make_flat(b200vs_metric m, int d, const b200vs_params& p) { return new FlatIndex(m, d, p); }

// ============================================================================================
// IVF arena shared by IVF-Flat (and reused by IVF-PQ for ids): see ivf_common.h
// ============================================================================================

struct IvfFlatIndex : IndexBase {
  int nlist;            // may degenerate to 1 at train time (vector_index_ivf_flat.cc:676-680)
  bool trained = false;
  DevBuf<float> centroids;       // [nlist, d]
  DevBuf<long long> cent_ids;    // iota
  DevBuf<float> cent_norms;      // ||c||^2 (tensor-core coarse pass)
  DevBuf<float> vecs;            // arena [arena_cap, d]
  DevBuf<long long> ids;         // arena
  DevBuf<float> norms;           // arena
  IvfLists L;                    // host bookkeeping + device list_off/list_len
  float max_norm = 0.f;
  float cent_max_norm = 0.f;
  DevBuf<float> cent_hi, cent_lo;  // error-compensated split of the centroids (tc_coarse)
  DevBuf<long long> d_coff;  // the centroid table seen as one "list" by the tensor-core coarse pass
  DevBuf<int> d_clen;
  TcView cent_view() const {
    TcView v;
    v.vecs = centroids.p; v.ids = cent_ids.p; v.norms = cent_norms.p; v.arena_rows = nlist; v.list_off = d_coff.p; v.list_len = d_clen.p;
    v.nlist = 1; v.flat = true; v.total_chunks = (nlist + TC_CHUNK - 1) / TC_CHUNK; v.max_chunks_per_list = (int)v.total_chunks;
    v.max_norm = cent_max_norm; v.vecs_hi = cent_hi.p; v.vecs_lo = cent_lo.p;
    return v;
  }
  TcView view() const {
    TcView v;
    v.vecs = vecs.p; v.ids = ids.p; v.norms = norms.p; v.arena_rows = L.arena_used; v.list_off = L.d_off.p; v.list_len = L.d_len.p;
    v.nlist = nlist; v.total_chunks = L.total_chunks; v.max_chunks_per_list = L.max_chunks_per_list; v.max_norm = max_norm;
    v.owned_frac = nlist > 0 ? (float)L.nonempty_lists / (float)nlist : 1.f;
    return v;
  }

  IvfFlatIndex(b200vs_metric m, int d, const b200vs_params& p) : IndexBase(B200VS_IVF_FLAT, m, d, p) {
    nlist = p.nlist > 0 ? p.nlist : 2048;  // Constant::kCreateIvfFlatParamNcentroids
  }
  bool is_trained() const override { return trained; }
  int export_nlist() const override { return nlist; }

  void install_centroids(const float* host_c, int k) {
    quiesce();
    nlist = k;
    centroids.free(); cent_ids.free(); cent_norms.free();
    centroids.reserve((size_t)k * dim, 0, stream);
    cent_ids.reserve(k, 0, stream);
    cent_norms.reserve(k, 0, stream);
    B200VS_CUDA(cudaMemcpyAsync(centroids.p, host_c, (size_t)k * dim * 4, cudaMemcpyHostToDevice, stream));
    launch_iota(cent_ids.p, k, stream);
    launch_row_norms(centroids.p, k, dim, cent_norms.p, stream);
    cent_hi.free(); cent_lo.free();
    cent_hi.reserve((size_t)k * dim, 0, stream); cent_lo.reserve((size_t)k * dim, 0, stream);
    launch_split_rows(centroids.p, k, dim, cent_hi.p, cent_lo.p, stream);
    cent_max_norm = device_max_norm(this, cent_norms.p, k, stream);
    d_coff.reserve(1, 0, stream); d_clen.reserve(1, 0, stream);
    B200VS_CUDA(cudaMemsetAsync(d_coff.p, 0, 8, stream));
    B200VS_CUDA(cudaMemcpyAsync(d_clen.p, &k, 4, cudaMemcpyHostToDevice, stream));
    B200VS_CUDA(cudaStreamSynchronize(stream));
    L.init(k, stream);
    vecs.free(); ids.free(); norms.free();
    trained = true;
  }

  // trained-state blob: int64 hdr[4] = {magic 'IVFC', nlist, dim, metric}; float centroids[nlist*dim]
  void set_state(const void* blob, size_t len) override {
    std::unique_lock<std::shared_mutex> wl(rw);
    std::lock_guard<std::mutex> gl(gpu_mu);
    set_device();
    if (len < 32) fail(B200VS_EILLEGAL_PARAMETERS, "state blob too short");
    const int64_t* hdr = (const int64_t*)blob;
    if (hdr[0] != 0x43465649 || hdr[2] != dim) fail(B200VS_EILLEGAL_PARAMETERS, "bad IVF state blob");
    const int k = (int)hdr[1];
    if (len < 32 + (size_t)k * dim * 4) fail(B200VS_EILLEGAL_PARAMETERS, "state blob truncated");
    install_centroids((const float*)((const char*)blob + 32), k);
  }
  int64_t get_state(void* blob, size_t cap) override {
    RwSharedGuard rl(this);
    if (!trained) return 0;
    const size_t need = 32 + (size_t)nlist * dim * 4;
    if (!blob || cap < need) return (int64_t)need;
    set_device();
    int64_t hdr[4] = {0x43465649, nlist, dim, (int64_t)metric};
    memcpy(blob, hdr, 32);
    B200VS_CUDA(cudaMemcpy((char*)blob + 32, centroids.p, (size_t)nlist * dim * 4, cudaMemcpyDeviceToHost));
    return (int64_t)need;
  }

  // assign rows (device, already normalised) to their nearest centroid: IndexFlat quantiser, k = 1.  Large batches go
  // through the tensor-core coarse pass (certified exact, so the labels equal the exact scan's).
  void assign_dev(const float* x_dev, int64_t n, long long* out_list_dev, cudaStream_t s) {
    const int64_t chunk = std::max<int64_t>(1024, std::min<int64_t>(32768, (1LL << 28) / std::max(1, nlist)));
    for (int64_t a = 0; a < n; a += chunk) {
      const int64_t m = std::min(chunk, n - a);
      const auto mark = scratch.mark();
      coarse(m, x_dev + (size_t)a * dim, 1, s, true, out_list_dev + a);
      scratch.release(mark);  // stream-ordered reuse
    }
  }

  // VectorIndexIvfFlat::Train, vector_index_ivf_flat.cc:644-712 -> faiss IndexIVFFlat::train ->
  // Clustering (niter 10, seed 1234, <= 256 points per centroid); GPU Lloyd iterations here.
  void train(int64_t n, const float* x) override;

  void add(int64_t n, const float* x, const int64_t* in_ids, bool upsert) override;
  void add_dev(int64_t n, const float* x_dev, const long long* ids_dev, const long long* lists_dev, bool upsert, bool prepared) override;
  void add_locked(int64_t n, float* st, const long long* st_ids, const int64_t* h_ids_in, const long long* lists_dev, bool upsert, bool prepared);
  void reserve_lists(const int64_t* rows_per_list, int n_lists) override;
  int nlist_now() const override { return nlist; }
  void assign_lists_dev(int64_t n, const float* x_dev, long long* out_lists_dev, cudaStream_t s) override {
    if (!trained) fail(B200VS_EVECTOR_NOT_TRAIN, "not train");
    assign_dev(x_dev, n, out_lists_dev, s);
  }
  void coarse_probes_dev(int64_t nq, const float* q_prepared, int nprobe, long long* out_lists, cudaStream_t s) override {
    if (!trained) fail(B200VS_EVECTOR_NOT_TRAIN, "not train");
    coarse(nq, q_prepared, nprobe, s, true, out_lists);
  }
  void search_probes_prepared_dev(int64_t nq, const float* q, int k, const long long* probes, int nprobe, const SearchCtx& sc, float* od,
                                  long long* oi, cudaStream_t s) override;
  int resolve_nprobe_api(const SearchCtx& sc) const override { return resolve_nprobe(sc); }
  int64_t remove(int64_t n, const int64_t* del) override;
  int64_t remove_locked(int64_t n, const int64_t* del);
  void maybe_compact();

  int resolve_nprobe(const SearchCtx& sc) const {
    int np = sc.nprobe > 0 ? sc.nprobe : 80;  // Constant::kSearchIvfFlatParamNprobe, ivf_flat.cc:211
    return std::min(np, nlist);               // ivf_flat.cc:234
  }

  void search_dev(int64_t nq, const float* xq, int k, const SearchCtx& sc, float* od, long long* oi, cudaStream_t s) override;
  void range_search_dev(int64_t nq, const float* xq, float radius, int max_results, const SearchCtx& sc, float* od,
                        long long* oi, int* oc, cudaStream_t s) override;
  void coarse_range_dev(int64_t nq, const float* xq, int nprobe, int c0, int c1, float* out_score, long long* out_lists, cudaStream_t s) override;
  void search_probes_dev(int64_t nq, const float* xq, int k, const long long* probes, int nprobe, const SearchCtx& sc, float* od,
                         long long* oi, cudaStream_t s) override;

  long long* coarse(int64_t nq, const float* q, int nprobe, cudaStream_t s, bool allow_tc = true, long long* out = nullptr) {
    long long* probes = out ? out : scratch.alloc<long long>((size_t)nq * nprobe);
    if (allow_tc && tc_coarse_eligible(this, nq, nlist, nprobe)) {  // dense TF32 scores + certified exact re-score
      tc_coarse(this, cent_view(), metric == B200VS_L2, nq, q, nprobe, probes, nullptr, s);
      return probes;
    }
    ScanJob j;
    j.l2 = metric == B200VS_L2;
    j.vecs = centroids.p; j.ids = cent_ids.p; j.d = dim; j.mode = 0; j.n = nlist;
    run_scan(this, j, nq, q, nprobe, nullptr, nullptr, probes, nullptr, s);
    return probes;
  }
  ScanJob list_job(const SearchCtx& sc, const long long* probes, int nprobe) const {
    ScanJob j;
    j.l2 = metric == B200VS_L2;
    j.vecs = vecs.p; j.ids = ids.p; j.d = dim; j.mode = 1; j.probes = probes; j.nprobe = nprobe;
    j.list_off = L.d_off.p; j.list_len = L.d_len.p; j.sc = &sc;
    j.avg_candidates = nlist > 0 ? (double)L.total_len() * nprobe / nlist : 0;
    return j;
  }

  int64_t count() const override { return L.live; }
  int64_t deleted_count() const override { return L.dead; }
  int64_t memory_size() const override {
    return (int64_t)(vecs.cap * 4 + ids.cap * 8 + norms.cap * 4 + centroids.cap * 4);
  }
  void export_lists(int64_t* list_off, float* vectors, uint8_t*, int64_t* out_ids) override;
  int64_t export_list(int list, int64_t cap, float* vectors, int64_t* out_ids) override;
};

void IvfFlatIndex::train(int64_t n, const float* x) {
  if (n <= 0) fail(B200VS_EILLEGAL_PARAMETERS, "data size invalid");
  std::unique_lock<std::shared_mutex> wl(rw);
  std::lock_guard<std::mutex> gl(gpu_mu);
  if (trained) return;  // ivf_flat.cc:670-672
  set_device();
  quiesce();
  scratch.reset(stream);
  int k = nlist;
  if (n < k) k = 1;  // "data size too small, nlist degenerate to 1", ivf_flat.cc:676-680
  std::vector<float> cent;
  kmeans_gpu(this, metric, dim, n, x, k, 10, 256, 1234, cent, [&](const float* xd, int64_t m, const float* cd, int kk, long long* out) {
    // assignment against the CURRENT centroids cd (device): tensor-core coarse pass when the shapes allow (certified
    // exact labels), else the exact scan
    const int64_t chunk = std::max<int64_t>(1024, std::min<int64_t>(32768, (1LL << 28) / std::max(1, kk)));
    const auto mark0 = scratch.mark();
    TcView cv;
    const bool use_tc = tc_coarse_eligible(this, std::min(chunk, m), kk, 1);
    if (use_tc) {
      float* hi = scratch.alloc<float>((size_t)kk * dim);
      float* lo = scratch.alloc<float>((size_t)kk * dim);
      float* nr = scratch.alloc<float>(kk);
      launch_split_rows(cd, kk, dim, hi, lo, stream);
      launch_row_norms(cd, kk, dim, nr, stream);
      cv.vecs = cd; cv.ids = cent_ids.p; cv.norms = nr; cv.arena_rows = kk; cv.list_off = d_coff.p; cv.list_len = nullptr;
      cv.nlist = 1; cv.flat = true; cv.total_chunks = (kk + TC_CHUNK - 1) / TC_CHUNK; cv.max_chunks_per_list = (int)cv.total_chunks;
      cv.max_norm = device_max_norm(this, nr, kk, stream); cv.vecs_hi = hi; cv.vecs_lo = lo;
    }
    ScanJob j;
    j.l2 = metric == B200VS_L2;
    j.vecs = cd; j.ids = cent_ids.p; j.d = dim; j.mode = 0; j.n = kk;
    for (int64_t a = 0; a < m; a += chunk) {
      const int64_t mm = std::min(chunk, m - a);
      const auto mark = scratch.mark();
      if (use_tc && mm >= 16) tc_coarse(this, cv, metric == B200VS_L2, mm, xd + (size_t)a * dim, 1, out + a, nullptr, stream);
      else run_scan(this, j, mm, xd + (size_t)a * dim, 1, nullptr, nullptr, out + a, nullptr, stream);
      scratch.release(mark);
    }
    scratch.release(mark0);
  }, [&](int kk) {
    cent_ids.free(); cent_ids.reserve(kk, 0, stream); launch_iota(cent_ids.p, kk, stream);
    d_coff.reserve(1, 0, stream);
    B200VS_CUDA(cudaMemsetAsync(d_coff.p, 0, 8, stream));
  });
  install_centroids(cent.data(), k);
}

void IvfFlatIndex::add(int64_t n, const float* x, const int64_t* in_ids, bool upsert) {
  std::unique_lock<std::shared_mutex> wl(rw);
  if (!trained) fail(B200VS_EVECTOR_NOT_TRAIN, "not train");  // ivf_flat.cc:111-113 (caller trains and retries, :136-150)
  std::lock_guard<std::mutex> gl(gpu_mu);
  set_device();
  quiesce();
  scratch.reset(stream);
  float* st = scratch.alloc<float>((size_t)n * dim);
  long long* st_ids = scratch.alloc<long long>(n);
  B200VS_CUDA(cudaMemcpyAsync(st, x, (size_t)n * dim * 4, cudaMemcpyHostToDevice, stream));
  B200VS_CUDA(cudaMemcpyAsync(st_ids, in_ids, (size_t)n * 8, cudaMemcpyHostToDevice, stream));
  add_locked(n, st, st_ids, in_ids, nullptr, upsert, loading);
}

void IvfFlatIndex::add_dev(int64_t n, const float* x_dev, const long long* ids_dev, const long long* lists_dev, bool upsert, bool prepared) {
  std::unique_lock<std::shared_mutex> wl(rw);
  if (!trained) fail(B200VS_EVECTOR_NOT_TRAIN, "not train");
  std::lock_guard<std::mutex> gl(gpu_mu);
  set_device();
  quiesce();
  scratch.reset(stream);
  float* st = const_cast<float*>(x_dev);
  if (metric == B200VS_COSINE && !prepared) {  // the normaliser works in place: keep the caller's rows intact
    st = scratch.alloc<float>((size_t)n * dim);
    B200VS_CUDA(cudaMemcpyAsync(st, x_dev, (size_t)n * dim * 4, cudaMemcpyDeviceToDevice, stream));
  }
  add_locked(n, st, ids_dev, nullptr, lists_dev, upsert, prepared);
}

// rw + gpu_mu held, scratch reset.  st / st_ids: device rows and ids (st may be normalised in place); h_ids_in: host copy
// of the ids when the caller has one; lists_dev: precomputed lists or NULL.
void IvfFlatIndex::add_locked(int64_t n, float* st, const long long* st_ids, const int64_t* h_ids_in, const long long* lists_dev, bool upsert,
                              bool prepared) {
  std::vector<int64_t> h_ids_buf;
  if (!h_ids_in) {
    h_ids_buf.resize(n);
    B200VS_CUDA(cudaMemcpyAsync(h_ids_buf.data(), st_ids, (size_t)n * 8, cudaMemcpyDeviceToHost, stream));
    B200VS_CUDA(cudaStreamSynchronize(stream));
    h_ids_in = h_ids_buf.data();
  }
  if (upsert) remove_locked(n, h_ids_in);  // ivf_flat.cc:115-118
  long long* st_slots = scratch.alloc<long long>(n);
  if (metric == B200VS_COSINE && !prepared) launch_normalize_faiss(st, n, dim, stream);
  const long long* st_list = lists_dev;
  if (!st_list) {
    long long* tmp = scratch.alloc<long long>(n);
    assign_dev(st, n, tmp, stream);
    st_list = tmp;
  }
  std::vector<long long> h_list(n), slots(n);
  B200VS_CUDA(cudaMemcpyAsync(h_list.data(), st_list, (size_t)n * 8, cudaMemcpyDeviceToHost, stream));
  B200VS_CUDA(cudaStreamSynchronize(stream));
  // host: reserve slots (may relocate lists / grow the arena)
  std::vector<int> need(nlist, 0);
  for (int64_t i = 0; i < n; ++i) {
    if (h_list[i] < 0 || h_list[i] >= nlist) fail(B200VS_EILLEGAL_PARAMETERS, "list id out of range");
    need[h_list[i]]++;
  }
  L.reserve_for(need, [&](int64_t arena_rows) {
    vecs.reserve((size_t)arena_rows * dim, (size_t)L.arena_used_before * dim, stream);
    ids.reserve((size_t)arena_rows, (size_t)L.arena_used_before, stream);
    norms.reserve((size_t)arena_rows, (size_t)L.arena_used_before, stream);
  }, [&](int64_t src, int64_t dst, int64_t len) {
    B200VS_CUDA(cudaMemcpyAsync(vecs.p + (size_t)dst * dim, vecs.p + (size_t)src * dim, (size_t)len * dim * 4, cudaMemcpyDeviceToDevice, stream));
    B200VS_CUDA(cudaMemcpyAsync(ids.p + dst, ids.p + src, (size_t)len * 8, cudaMemcpyDeviceToDevice, stream));
    B200VS_CUDA(cudaMemcpyAsync(norms.p + dst, norms.p + src, (size_t)len * 4, cudaMemcpyDeviceToDevice, stream));
  });
  for (int64_t i = 0; i < n; ++i) slots[i] = L.append((int)h_list[i], h_ids_in[i]);
  B200VS_CUDA(cudaMemcpyAsync(st_slots, slots.data(), (size_t)n * 8, cudaMemcpyHostToDevice, stream));
  float* st_norms = scratch.alloc<float>(n);
  launch_scatter_rows(st, st_ids, st_slots, n, dim, vecs.p, ids.p, norms.p, st_norms, stream);
  max_norm = std::max(max_norm, device_max_norm(this, st_norms, n, stream));
  L.upload(stream);
  B200VS_CUDA(cudaStreamSynchronize(stream));
}

// one arena allocation holding every list at its final size (+ 1/16 slack): bulk builds of large shards
void IvfFlatIndex::reserve_lists(const int64_t* rows_per_list, int n_lists) {
  std::unique_lock<std::shared_mutex> wl(rw);
  if (!trained) fail(B200VS_EVECTOR_NOT_TRAIN, "not train");
  if (n_lists != nlist) fail(B200VS_EILLEGAL_PARAMETERS, "reserve_lists: list count does not match the trained index");
  std::lock_guard<std::mutex> gl(gpu_mu);
  set_device();
  quiesce();
  if (L.live + L.dead > 0) fail(B200VS_EILLEGAL_PARAMETERS, "reserve_lists needs an empty index");
  int64_t used = 0;
  for (int l = 0; l < nlist; ++l) {
    const int64_t want = rows_per_list[l];
    if (want < 0 || want >= (1LL << 31) - 64) fail(B200VS_EILLEGAL_PARAMETERS, "reserve_lists: bad list size");
    ListMeta& m = L.lists[l];
    m.off = used; m.len = 0; m.dead = 0;
    m.cap = want ? IvfLists::round32(want + want / 16 + 32) : 0;
    used += m.cap;
  }
  const int64_t tail = std::max<int64_t>(used / 64, 4096);  // room for lists that still outgrow their reservation
  L.arena_used = L.arena_used_before = used;
  L.arena_cap = used + tail;
  vecs.free(); ids.free(); norms.free();
  vecs.reserve((size_t)L.arena_cap * dim, 0, stream);
  ids.reserve((size_t)L.arena_cap, 0, stream);
  norms.reserve((size_t)L.arena_cap, 0, stream);
  B200VS_CUDA(cudaMemsetAsync(ids.p, 0xFF, (size_t)L.arena_cap * 8, stream));  // id -1 = unused slot
  L.h_ids.assign(L.arena_cap, -1);
  L.upload(stream);
}

int64_t IvfFlatIndex::remove_locked(int64_t n, const int64_t* del) {
  std::vector<int64_t> rws;
  L.remove_ids(n, del, rws);
  if (!rws.empty()) {
    long long* d_rows = scratch.alloc<long long>(rws.size());
    B200VS_CUDA(cudaMemcpyAsync(d_rows, rws.data(), rws.size() * 8, cudaMemcpyHostToDevice, stream));
    launch_set_ids(ids.p, d_rows, (int64_t)rws.size(), -1, stream);
    B200VS_CUDA(cudaStreamSynchronize(stream));
  }
  return (int64_t)rws.size();
}

void IvfFlatIndex::maybe_compact() {
  if (!L.needs_compaction()) return;
  std::vector<long long> src, dst;
  const int64_t new_rows = L.plan_compaction(src, dst);
  DevBuf<float> nv; DevBuf<long long> ni; DevBuf<float> nn;
  nv.reserve((size_t)std::max<int64_t>(new_rows, 1) * dim, 0, stream);
  ni.reserve(std::max<int64_t>(new_rows, 1), 0, stream);
  nn.reserve(std::max<int64_t>(new_rows, 1), 0, stream);
  const int64_t m = (int64_t)src.size();
  if (m) {
    long long* d_src = scratch.alloc<long long>(m);
    long long* d_dst = scratch.alloc<long long>(m);
    B200VS_CUDA(cudaMemcpyAsync(d_src, src.data(), m * 8, cudaMemcpyHostToDevice, stream));
    B200VS_CUDA(cudaMemcpyAsync(d_dst, dst.data(), m * 8, cudaMemcpyHostToDevice, stream));
    launch_move_rows(vecs.p, ids.p, norms.p, d_src, d_dst, m, dim, nv.p, ni.p, nn.p, stream);
  }
  B200VS_CUDA(cudaStreamSynchronize(stream));
  std::swap(vecs.p, nv.p); std::swap(vecs.cap, nv.cap);
  std::swap(ids.p, ni.p); std::swap(ids.cap, ni.cap);
  std::swap(norms.p, nn.p); std::swap(norms.cap, nn.cap);
  L.commit_compaction();
  L.upload(stream);
  B200VS_CUDA(cudaStreamSynchronize(stream));
}

// VectorIndexIvfFlat::Delete, vector_index_ivf_flat.cc:162-189: untrained -> OK; nothing removed -> EVECTOR_INVALID.
int64_t IvfFlatIndex::remove(int64_t n, const int64_t* del) {
  std::unique_lock<std::shared_mutex> wl(rw);
  if (!trained) return -1;  // signalled as OK by the ABI
  std::lock_guard<std::mutex> gl(gpu_mu);
  set_device();
  quiesce();
  scratch.reset(stream);
  const int64_t r = remove_locked(n, del);
  maybe_compact();
  return r;
}

void fill_empty_results(int64_t nq, int k, float* od, long long* oi, cudaStream_t s) {
  if (od) B200VS_CUDA(cudaMemsetAsync(od, 0, (size_t)nq * k * 4, s));
  B200VS_CUDA(cudaMemsetAsync(oi, 0xFF, (size_t)nq * k * 8, s));  // -1
}

void IvfFlatIndex::search_dev(int64_t nq, const float* xq, int k, const SearchCtx& sc, float* od, long long* oi, cudaStream_t s) {
  if (!trained) { fill_empty_results(nq, k, od, oi, s); return; }  // ivf_flat.cc:224-227
  const float* q = prepare_queries(nq, xq, s);
  const int nprobe = resolve_nprobe(sc);
  long long* probes = coarse(nq, q, nprobe, s, !sc.exact_only);
  if (profiling) profile_probed(this, probes, nq * nprobe, nlist, L.d_len.p, s);
  const TcView v = view();
  if (L.live > 0 && tc_eligible(this, v, nq, k, nprobe, sc)) {
    tc_search(this, v, metric == B200VS_L2, nq, q, k, probes, nprobe, sc, od, oi, s);
    return;
  }
  ScanJob j = list_job(sc, probes, nprobe);
  j.dominant = true;
  run_scan(this, j, nq, q, k, od, nullptr, oi, nullptr, s);
}

void IvfFlatIndex::coarse_range_dev(int64_t nq, const float* xq, int nprobe, int c0, int c1, float* out_score, long long* out_lists, cudaStream_t s) {
  if (!trained) fail(B200VS_EVECTOR_NOT_TRAIN, "not train");
  if (c0 < 0 || c1 > nlist || c0 >= c1 || nprobe <= 0 || nprobe > c1 - c0) fail(B200VS_EILLEGAL_PARAMETERS, "bad centroid range / nprobe");
  const float* q = prepare_queries(nq, xq, s);
  const int rows = c1 - c0;
  if (tc_coarse_eligible(this, nq, rows, nprobe)) {
    TcView v = cent_view();
    v.vecs += (size_t)c0 * dim; v.vecs_hi += (size_t)c0 * dim; v.vecs_lo += (size_t)c0 * dim; v.ids += c0; v.norms += c0;
    v.arena_rows = rows; v.total_chunks = (rows + TC_CHUNK - 1) / TC_CHUNK; v.max_chunks_per_list = (int)v.total_chunks;
    v.id_offset = c0; v.api_scores = true;
    tc_coarse(this, v, metric == B200VS_L2, nq, q, nprobe, out_lists, out_score, s);
    return;
  }
  ScanJob j;
  j.l2 = metric == B200VS_L2;
  j.vecs = centroids.p + (size_t)c0 * dim; j.ids = cent_ids.p + c0; j.d = dim; j.mode = 0; j.n = rows;
  run_scan(this, j, nq, q, nprobe, nullptr, out_score, out_lists, nullptr, s);  // raw metric value
  if (metric != B200VS_L2) launch_negate(out_score, nq * nprobe, s);             // -> ascending ranking score
}

void IvfFlatIndex::search_probes_dev(int64_t nq, const float* xq, int k, const long long* probes, int nprobe, const SearchCtx& sc, float* od,
                                     long long* oi, cudaStream_t s) {
  if (!trained) { fill_empty_results(nq, k, od, oi, s); return; }
  search_probes_prepared_dev(nq, prepare_queries(nq, xq, s), k, probes, nprobe, sc, od, oi, s);
}

void IvfFlatIndex::search_probes_prepared_dev(int64_t nq, const float* q, int k, const long long* probes, int nprobe, const SearchCtx& sc,
                                              float* od, long long* oi, cudaStream_t s) {
  if (!trained) { fill_empty_results(nq, k, od, oi, s); return; }
  if (profiling) profile_probed(this, probes, nq * nprobe, nlist, L.d_len.p, s);
  const TcView v = view();
  if (L.live > 0 && tc_eligible(this, v, nq, k, nprobe, sc)) {
    tc_search(this, v, metric == B200VS_L2, nq, q, k, probes, nprobe, sc, od, oi, s);
    return;
  }
  ScanJob j = list_job(sc, probes, nprobe);
  j.dominant = true;
  run_scan(this, j, nq, q, k, od, nullptr, oi, nullptr, s);
}

void IvfFlatIndex::range_search_dev(int64_t nq, const float* xq, float radius, int max_results, const SearchCtx& sc,
                                    float* od, long long* oi, int* oc, cudaStream_t s) {
  if (!trained) {
    fill_empty_results(nq, max_results, od, oi, s);
    if (oc) B200VS_CUDA(cudaMemsetAsync(oc, 0, (size_t)nq * 4, s));
    return;
  }
  const float* q = prepare_queries(nq, xq, s);
  const int nprobe = resolve_nprobe(sc);
  long long* probes = coarse(nq, q, nprobe, s);
  ScanJob j = list_job(sc, probes, nprobe);
  j.has_thr = true;
  j.thr_raw = ip_like() ? 1.0F - radius : radius;  // ivf_flat.cc:296-299
  run_scan(this, j, nq, q, max_results, od, nullptr, oi, oc, s);
}

void IvfFlatIndex::export_lists(int64_t* list_off, float* vectors, uint8_t*, int64_t* out_ids) {
  RwSharedGuard rl(this);
  std::lock_guard<std::mutex> gl(gpu_mu);
  set_device();
  std::vector<float> rowbuf;
  int64_t o = 0;
  for (int l = 0; l < nlist; ++l) {
    if (list_off) list_off[l] = o;
    const auto& m = L.lists[l];
    if (m.len == 0) continue;
    if (vectors) {
      rowbuf.resize((size_t)m.len * dim);
      B200VS_CUDA(cudaMemcpy(rowbuf.data(), vecs.p + (size_t)m.off * dim, (size_t)m.len * dim * 4, cudaMemcpyDeviceToHost));
    }
    for (int p = 0; p < m.len; ++p) {
      const int64_t id = L.h_ids[m.off + p];
      if (id < 0) continue;
      if (out_ids) out_ids[o] = id;
      if (vectors) memcpy(vectors + (size_t)o * dim, rowbuf.data() + (size_t)p * dim, (size_t)dim * 4);
      ++o;
    }
  }
  if (list_off) list_off[nlist] = o;
}

int64_t IvfFlatIndex::export_list(int list, int64_t cap, float* vectors, int64_t* out_ids) {
  RwSharedGuard rl(this);
  std::lock_guard<std::mutex> gl(gpu_mu);
  if (list < 0 || list >= nlist) fail(B200VS_EILLEGAL_PARAMETERS, "list id out of range");
  set_device();
  quiesce();
  const auto& m = L.lists[list];
  std::vector<float> rowbuf;
  if (vectors && m.len) {
    rowbuf.resize((size_t)m.len * dim);
    B200VS_CUDA(cudaMemcpy(rowbuf.data(), vecs.p + (size_t)m.off * dim, (size_t)m.len * dim * 4, cudaMemcpyDeviceToHost));
  }
  int64_t o = 0;
  for (int p = 0; p < m.len; ++p) {
    const int64_t id = L.h_ids[m.off + p];
    if (id < 0) continue;
    if (o < cap) {
      if (out_ids) out_ids[o] = id;
      if (vectors) memcpy(vectors + (size_t)o * dim, rowbuf.data() + (size_t)p * dim, (size_t)dim * 4);
    }
    ++o;
  }
  return o;
}

IndexBase* make_ivf_flat(b200vs_metric m, int d, const b200vs_params& p) { return new IvfFlatIndex(m, d, p); }

}  // namespace b200vs

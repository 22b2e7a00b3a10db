// api.cu — extern "C" entry points of libb200vs.so (declared in include/b200vs.h).
// No exception leaves this file: every entry point maps failures to a b200vs_status
// (reference convention: butil::Status codes, never exceptions across the plugin virtual;
// src/vector/vector_index_flat.cc:313-315, src/handler/raft_apply_handler.cc:1311-1325).
#include <cstdio>
#include <memory>
#include <new>
#include <string>
#include <vector>

#include "index.h"

using namespace b200vs;

namespace {

template <class F>
int guarded(F&& f) {
  try {
    return f();
  } catch (const StatusError& e) {
    g_last_error = e.msg;
    return e.code;
  } catch (const CudaError& e) {
    g_last_error = e.what();
    return B200VS_EINTERNAL;
  } catch (const std::bad_alloc&) {
    g_last_error = "out of host memory";
    return B200VS_EINTERNAL;
  } catch (const std::exception& e) {
    g_last_error = e.what();
    return B200VS_EINTERNAL;
  } catch (...) {
    g_last_error = "unknown error";
    return B200VS_EINTERNAL;
  }
}

IndexBase* get(b200vs_index* h) { return index_impl(h); }

// resolve search params; uploads the sorted id list into scratch (stream-ordered)
SearchCtx make_ctx(IndexBase* ix, const b200vs_search_params* sp, cudaStream_t s) {
  SearchCtx sc;
  if (!sp) return sc;
  sc.nprobe = sp->nprobe;
  sc.efsearch = sp->efsearch;
  sc.exact_only = sp->exact_only;
  sc.has_range = sp->has_range;
  sc.negate = sp->negate;
  sc.rmin = sp->range_min;
  sc.rmax = sp->range_max;
  if (sp->sorted_ids) {
    long long* d = ix->scratch.alloc<long long>((size_t)std::max<int64_t>(sp->n_ids, 1));
    if (sp->n_ids > 0) B200VS_CUDA(cudaMemcpyAsync(d, sp->sorted_ids, (size_t)sp->n_ids * 8, cudaMemcpyHostToDevice, s));
    sc.sorted_ids_dev = d;
    sc.n_ids = sp->n_ids;
  }
  return sc;
}

// ExtractVectorValue's value-type check (vector_index_utils.cc:502-530): float rows for float indexes, bytes for binary ones
void require_float(IndexBase* ix) {
  if (ix->binary()) fail(B200VS_EVECTOR_INVALID, "float vectors given to a binary index");
}
void require_binary(IndexBase* ix) {
  if (!ix->binary()) fail(B200VS_EVECTOR_INVALID, "binary vectors given to a float index");
}

void check_search_args(IndexBase* ix, int64_t nq, const void* xq, const b200vs_search_params* sp) {
  if (nq <= 0 || !xq) fail(B200VS_EILLEGAL_PARAMETERS, "vector_with_ids is empty");  // flat.cc:208-210
  if (ix->type == B200VS_HNSW && sp && (sp->efsearch < 0 || sp->efsearch > 1024))
    fail(B200VS_EILLEGAL_PARAMETERS, "efsearch is illegal, " + std::to_string(sp->efsearch) + ", must between 0 and 1024");  // hnsw.cc:332-336
}

}  // namespace

extern "C" {

int b200vs_create(b200vs_type type, b200vs_metric metric, int32_t dim, const b200vs_params* params, b200vs_index** out) {
  return guarded([&]() -> int {
    if (!out) fail(B200VS_EILLEGAL_PARAMETERS, "out is null");
    *out = nullptr;
    if (dim <= 0) fail(B200VS_EILLEGAL_PARAMETERS, "dimension must be > 0");
    if (type == B200VS_BINARY_FLAT || type == B200VS_BINARY_IVF_FLAT) {  // vector_index_utils.cc:1085-1099, :1117-1130
      if (metric != B200VS_HAMMING) fail(B200VS_EILLEGAL_PARAMETERS, "binary indexes need metric HAMMING");
      if (dim % 8 != 0 || dim > 32768) fail(B200VS_EILLEGAL_PARAMETERS, "binary dimension must be a multiple of 8 and at most 32768");
    } else if (metric != B200VS_L2 && metric != B200VS_IP && metric != B200VS_COSINE) {
      fail(B200VS_EILLEGAL_PARAMETERS, "unsupported metric type");
    }
    b200vs_params p;
    memset(&p, 0, sizeof(p));
    if (params) p = *params;
    int ndev = 0;
    B200VS_CUDA(cudaGetDeviceCount(&ndev));
    if (p.device < 0 || p.device >= ndev) fail(B200VS_EILLEGAL_PARAMETERS, "bad CUDA device ordinal");
    IndexBase* impl = nullptr;
    switch (type) {
      case B200VS_FLAT: impl = make_flat(metric, dim, p); break;
      case B200VS_IVF_FLAT: impl = make_ivf_flat(metric, dim, p); break;
      case B200VS_IVF_PQ: impl = make_ivf_pq(metric, dim, p); break;
      case B200VS_HNSW: impl = make_hnsw(metric, dim, p); break;
      case B200VS_BINARY_FLAT:
      case B200VS_BINARY_IVF_FLAT: impl = make_binary(type, dim, p); break;
      default: fail(B200VS_EILLEGAL_PARAMETERS, "unknown index type");
    }
    *out = new b200vs_index{impl};
    return B200VS_OK;
  });
}

void b200vs_destroy(b200vs_index* h) {
  if (!h) return;
  try { delete h->impl; } catch (...) {}
  delete h;
}

int b200vs_train(b200vs_index* h, int64_t n, const float* x) {
  return guarded([&]() -> int {
    IndexBase* ix = get(h);
    require_float(ix);
    if (n <= 0 || !x) fail(B200VS_EILLEGAL_PARAMETERS, "data size invalid");  // ivf_flat.cc:646-649
    ix->train(n, x);
    return B200VS_OK;
  });
}

int b200vs_set_trained_state(b200vs_index* h, const void* blob, size_t len) {
  return guarded([&]() -> int {
    IndexBase* ix = get(h);
    if (!blob) fail(B200VS_EILLEGAL_PARAMETERS, "null blob");
    ix->set_state(blob, len);
    return B200VS_OK;
  });
}

int64_t b200vs_get_trained_state(b200vs_index* h, void* blob, size_t cap) {
  int64_t r = 0;
  int rc = guarded([&]() -> int { r = get(h)->get_state(blob, cap); return B200VS_OK; });
  return rc == B200VS_OK ? r : -(int64_t)rc;
}

int b200vs_add_with_ids(b200vs_index* h, int64_t n, const float* x, const int64_t* ids, int upsert) {
  return guarded([&]() -> int {
    IndexBase* ix = get(h);
    require_float(ix);
    if (n <= 0 || !x || !ids) fail(B200VS_EILLEGAL_PARAMETERS, "vector_with_ids is empty");  // flat.cc:123-125
    ix->add(n, x, ids, upsert != 0);
    return B200VS_OK;
  });
}

int b200vs_add_with_ids_device(b200vs_index* h, int64_t n, const float* x_dev, const int64_t* ids_dev, const int64_t* lists_dev, int upsert) {
  return guarded([&]() -> int {
    IndexBase* ix = get(h);
    if (n <= 0 || !x_dev || !ids_dev) fail(B200VS_EILLEGAL_PARAMETERS, "vector_with_ids is empty");
    ix->add_dev(n, x_dev, (const long long*)ids_dev, (const long long*)lists_dev, upsert != 0, false);
    return B200VS_OK;
  });
}

int b200vs_assign_device(b200vs_index* h, int64_t n, const float* x_dev, int64_t* out_lists_dev) {
  return guarded([&]() -> int {
    IndexBase* ix = get(h);
    if (n <= 0 || !x_dev || !out_lists_dev) fail(B200VS_EILLEGAL_PARAMETERS, "bad assign arguments");
    std::shared_lock<std::shared_mutex> rl(ix->rw);
    ix->set_device();
    LaneGuard lane(ix, nullptr);
    const float* q = ix->prepare_queries(n, x_dev, lane.stream);
    ix->assign_lists_dev(n, q, (long long*)out_lists_dev, lane.stream);
    B200VS_CUDA(cudaStreamSynchronize(lane.stream));
    return B200VS_OK;
  });
}

int b200vs_reserve_lists(b200vs_index* h, const int64_t* rows_per_list, int32_t nlist) {
  return guarded([&]() -> int {
    IndexBase* ix = get(h);
    if (!rows_per_list || nlist <= 0) fail(B200VS_EILLEGAL_PARAMETERS, "bad reserve arguments");
    ix->reserve_lists(rows_per_list, nlist);
    return B200VS_OK;
  });
}

int b200vs_remove_ids(b200vs_index* h, int64_t n, const int64_t* ids, int64_t* n_removed) {
  return guarded([&]() -> int {
    IndexBase* ix = get(h);
    if (n_removed) *n_removed = 0;
    if (n <= 0) return B200VS_OK;  // "delete_ids.empty() -> OK", flat.cc:172-174
    if (!ids) fail(B200VS_EILLEGAL_PARAMETERS, "null ids");
    const int64_t r = ix->remove(n, ids);
    if (n_removed) *n_removed = r < 0 ? 0 : r;
    // IVF types: "remove not found vector id" -> EVECTOR_INVALID (ivf_flat.cc:180-184); untrained -> OK (r == -1)
    if (r == 0 && (ix->type == B200VS_IVF_FLAT || ix->type == B200VS_IVF_PQ || ix->type == B200VS_BINARY_IVF_FLAT)) fail(B200VS_EVECTOR_INVALID, "remove not found vector id");
    return B200VS_OK;
  });
}

int b200vs_search_device(b200vs_index* h, int64_t nq, const float* xq_dev, int32_t k, const b200vs_search_params* sp,
                         float* out_dist_dev, int64_t* out_ids_dev, void* stream) {
  return guarded([&]() -> int {
    IndexBase* ix = get(h);
    require_float(ix);
    check_search_args(ix, nq, xq_dev, sp);
    if (k <= 0) return B200VS_OK;  // "topk <= 0 -> OK", flat.cc:212
    if (!out_ids_dev) fail(B200VS_EILLEGAL_PARAMETERS, "null output");
    std::shared_lock<std::shared_mutex> rl(ix->rw);
    ix->set_device();
    LaneGuard lane(ix, (cudaStream_t)stream);
    cudaStream_t s = lane.stream;
    ix->reset_stats();
    SearchCtx sc = make_ctx(ix, sp, s);
    ix->search_dev(nq, xq_dev, k, sc, out_dist_dev, (long long*)out_ids_dev, s);
    ix->phases_finish(s);
    if (!stream) B200VS_CUDA(cudaStreamSynchronize(s));  // NULL stream: library-owned stream, results ready on return
    return B200VS_OK;
  });
}

int b200vs_coarse_device(b200vs_index* h, int64_t nq, const float* xq_dev, int32_t nprobe, int32_t list_begin, int32_t list_end,
                         float* out_score_dev, int64_t* out_lists_dev, void* stream) {
  return guarded([&]() -> int {
    IndexBase* ix = get(h);
    if (nq <= 0 || !xq_dev || !out_score_dev || !out_lists_dev) fail(B200VS_EILLEGAL_PARAMETERS, "bad coarse arguments");
    std::shared_lock<std::shared_mutex> rl(ix->rw);
    ix->set_device();
    LaneGuard lane(ix, (cudaStream_t)stream);
    ix->reset_stats();
    ix->coarse_range_dev(nq, xq_dev, nprobe, list_begin, list_end, out_score_dev, (long long*)out_lists_dev, lane.stream);
    ix->phases_finish(lane.stream);
    if (!stream) B200VS_CUDA(cudaStreamSynchronize(lane.stream));
    return B200VS_OK;
  });
}

int b200vs_search_probes_device(b200vs_index* h, int64_t nq, const float* xq_dev, int32_t k, const int64_t* probes_dev, int32_t nprobe,
                                const b200vs_search_params* sp, float* out_dist_dev, int64_t* out_ids_dev, void* stream) {
  return guarded([&]() -> int {
    IndexBase* ix = get(h);
    check_search_args(ix, nq, xq_dev, sp);
    if (k <= 0) return B200VS_OK;
    if (!probes_dev || nprobe <= 0 || !out_ids_dev) fail(B200VS_EILLEGAL_PARAMETERS, "bad probe arguments");
    std::shared_lock<std::shared_mutex> rl(ix->rw);
    ix->set_device();
    LaneGuard lane(ix, (cudaStream_t)stream);
    ix->reset_stats();
    SearchCtx sc = make_ctx(ix, sp, lane.stream);
    ix->search_probes_dev(nq, xq_dev, k, (const long long*)probes_dev, nprobe, sc, out_dist_dev, (long long*)out_ids_dev, lane.stream);
    ix->phases_finish(lane.stream);
    if (!stream) B200VS_CUDA(cudaStreamSynchronize(lane.stream));
    return B200VS_OK;
  });
}

}  // extern "C"

namespace {

// one host-pointer search: H2D, search, D2H, wait.  xq / outputs may be pinned staging (coalesced batches) or caller memory.
void host_search_once(IndexBase* ix, int64_t nq, const float* xq, int k, const b200vs_search_params* sp, float* out_dist, int64_t* out_ids) {
  std::shared_lock<std::shared_mutex> rl(ix->rw);
  ix->set_device();
  LaneGuard lane(ix, nullptr);  // a free lane on its own stream, so concurrent callers overlap
  cudaStream_t s = lane.stream;
  ix->reset_stats();
  float* dq = ix->scratch.alloc<float>((size_t)nq * ix->dim);
  float* dd = ix->scratch.alloc<float>((size_t)nq * k);
  long long* di = ix->scratch.alloc<long long>((size_t)nq * k);
  B200VS_CUDA(cudaMemcpyAsync(dq, xq, (size_t)nq * ix->dim * 4, cudaMemcpyHostToDevice, s));
  SearchCtx sc = make_ctx(ix, sp, s);
  ix->search_dev(nq, dq, k, sc, dd, di, s);
  ix->phases_finish(s);
  B200VS_CUDA(cudaMemcpyAsync(out_dist, dd, (size_t)nq * k * 4, cudaMemcpyDeviceToHost, s));
  B200VS_CUDA(cudaMemcpyAsync(out_ids, di, (size_t)nq * k * 8, cudaMemcpyDeviceToHost, s));
  B200VS_CUDA(cudaStreamSynchronize(s));
}

bool coalesce_compatible(const CoalesceReq& a, const CoalesceReq& b) {
  return a.k == b.k && a.sp.nprobe == b.sp.nprobe && a.sp.efsearch == b.sp.efsearch && a.sp.exact_only == b.sp.exact_only &&
         a.sp.has_range == b.sp.has_range && (!a.sp.has_range || (a.sp.range_min == b.sp.range_min && a.sp.range_max == b.sp.range_max));
}

constexpr int64_t kCoalesceMaxReq = 64;     // requests at most this large join a shared batch
constexpr int64_t kCoalesceMaxBatch = 4096; // queries per shared batch (the service limit, index_service.cc:50)

// the leader's work: one batch for all requests in `batch` (>= 2 of them, compatible)
void run_coalesced(IndexBase* ix, std::vector<CoalesceReq*>& batch) {
  int64_t total = 0;
  for (auto* r : batch) total += r->nq;
  const int k = batch[0]->k, d = ix->dim;
  // pinned staging owned by the calling (leader) thread: queries in, results out (one H2D, one D2H of each kind)
  const size_t qbytes = (size_t)total * d * 4, dbytes = (size_t)total * k * 4, ibytes = (size_t)total * k * 8;
  const size_t need = qbytes + dbytes + ibytes + 64;
  static thread_local void* pin = nullptr;
  static thread_local size_t pin_cap = 0;
  if (pin_cap < need) {
    ix->set_device();
    if (pin) cudaFreeHost(pin);
    pin = nullptr; pin_cap = 0;
    B200VS_CUDA(cudaHostAlloc(&pin, need * 2, cudaHostAllocPortable));  // portable: the calling thread may serve indexes on several devices
    pin_cap = need * 2;
  }
  float* hq = reinterpret_cast<float*>(pin);
  float* hd = reinterpret_cast<float*>(reinterpret_cast<char*>(pin) + ((qbytes + 15) & ~(size_t)15));
  int64_t* hi = reinterpret_cast<int64_t*>(reinterpret_cast<char*>(hd) + ((dbytes + 15) & ~(size_t)15));
  int64_t off = 0;
  for (auto* r : batch) { memcpy(hq + (size_t)off * d, r->xq, (size_t)r->nq * d * 4); off += r->nq; }
  host_search_once(ix, total, hq, k, &batch[0]->sp, hd, hi);
  off = 0;
  for (auto* r : batch) {
    memcpy(r->out_dist, hd + (size_t)off * k, (size_t)r->nq * k * 4);
    memcpy(r->out_ids, hi + (size_t)off * k, (size_t)r->nq * k * 8);
    off += r->nq;
  }
}

int coalesced_search(IndexBase* ix, int64_t nq, const float* xq, int k, const b200vs_search_params* sp, float* out_dist, int64_t* out_ids) {
  Coalescer& C = ix->coalescer;
  CoalesceReq me;
  me.nq = nq; me.xq = xq; me.k = k; me.out_dist = out_dist; me.out_ids = out_ids;
  if (sp) me.sp = *sp;
  std::unique_lock<std::mutex> lk(C.mu);
  C.pending.push_back(&me);
  while (!me.done) {
    if (C.busy) { C.cv.wait(lk); continue; }
    // become the leader: everything compatible with the oldest pending request, in arrival order
    C.busy = true;
    std::vector<CoalesceReq*> batch, rest;
    int64_t total = 0;
    for (auto* r : C.pending) {
      if ((batch.empty() || coalesce_compatible(*batch[0], *r)) && total + r->nq <= kCoalesceMaxBatch) { batch.push_back(r); total += r->nq; }
      else rest.push_back(r);
    }
    C.pending.swap(rest);
    lk.unlock();
    int rc = B200VS_OK;
    std::string err;
    try {
      if (batch.size() == 1) host_search_once(ix, batch[0]->nq, batch[0]->xq, batch[0]->k, &batch[0]->sp, batch[0]->out_dist, batch[0]->out_ids);
      else run_coalesced(ix, batch);
    } catch (const StatusError& e) { rc = e.code; err = e.msg; }
    catch (const std::exception& e) { rc = B200VS_EINTERNAL; err = e.what(); }
    catch (...) { rc = B200VS_EINTERNAL; err = "unknown error"; }
    C.batches.fetch_add(1);
    C.requests.fetch_add((int64_t)batch.size());
    lk.lock();
    for (auto* r : batch) { r->rc = rc; r->err = err; r->done = true; }
    C.busy = false;
    C.cv.notify_all();
  }
  lk.unlock();
  if (me.rc != B200VS_OK) g_last_error = me.err;
  return me.rc;
}

}  // namespace

extern "C" {

int b200vs_search(b200vs_index* h, int64_t nq, const float* xq, int32_t k, const b200vs_search_params* sp, float* out_dist,
                  int64_t* out_ids) {
  return guarded([&]() -> int {
    IndexBase* ix = get(h);
    require_float(ix);
    check_search_args(ix, nq, xq, sp);
    if (k <= 0) return B200VS_OK;
    if (!out_ids || !out_dist) fail(B200VS_EILLEGAL_PARAMETERS, "null output");
    // small filter-free requests share batches with concurrent callers (the reference issues one query per pool task)
    if (nq <= kCoalesceMaxReq && ix->coalescer.enabled.load() && !(sp && sp->sorted_ids) && !ix->profiling)
      return coalesced_search(ix, nq, xq, k, sp, out_dist, out_ids);
    host_search_once(ix, nq, xq, k, sp, out_dist, out_ids);
    return B200VS_OK;
  });
}

/* Request coalescing of b200vs_search (on by default): concurrent host-pointer calls of <= 64 queries without id-list filters
 * are merged into shared batches.  stats (nullable): [0] batches run, [1] requests served through them. */
int b200vs_set_coalescing(b200vs_index* h, int on, int64_t stats[2]) {
  return guarded([&]() -> int {
    IndexBase* ix = get(h);
    if (on >= 0) ix->coalescer.enabled.store(on ? 1 : 0);
    if (stats) { stats[0] = ix->coalescer.batches.load(); stats[1] = ix->coalescer.requests.load(); }
    return B200VS_OK;
  });
}

int b200vs_range_search(b200vs_index* h, int64_t nq, const float* xq, float radius, int32_t max_results,
                        const b200vs_search_params* sp, float* out_dist, int64_t* out_ids, int32_t* out_counts) {
  return guarded([&]() -> int {
    IndexBase* ix = get(h);
    require_float(ix);
    check_search_args(ix, nq, xq, sp);
    if (ix->type == B200VS_HNSW) fail(B200VS_EVECTOR_NOT_SUPPORT, "RangeSearch not support in Hnsw!!!");  // hnsw.cc:487-493
    if (max_results <= 0 || !out_ids || !out_dist || !out_counts) fail(B200VS_EILLEGAL_PARAMETERS, "bad range-search outputs");
    std::shared_lock<std::shared_mutex> rl(ix->rw);
    ix->set_device();
    LaneGuard lane(ix, nullptr);
    cudaStream_t s = lane.stream;
    float* dq = ix->scratch.alloc<float>((size_t)nq * ix->dim);
    float* dd = ix->scratch.alloc<float>((size_t)nq * max_results);
    long long* di = ix->scratch.alloc<long long>((size_t)nq * max_results);
    int* dc = ix->scratch.alloc<int>((size_t)nq);
    B200VS_CUDA(cudaMemcpyAsync(dq, xq, (size_t)nq * ix->dim * 4, cudaMemcpyHostToDevice, s));
    SearchCtx sc = make_ctx(ix, sp, s);
    ix->range_search_dev(nq, dq, radius, max_results, sc, dd, di, dc, s);
    ix->phases_finish(s);
    B200VS_CUDA(cudaMemcpyAsync(out_dist, dd, (size_t)nq * max_results * 4, cudaMemcpyDeviceToHost, s));
    B200VS_CUDA(cudaMemcpyAsync(out_ids, di, (size_t)nq * max_results * 8, cudaMemcpyDeviceToHost, s));
    B200VS_CUDA(cudaMemcpyAsync(out_counts, dc, (size_t)nq * 4, cudaMemcpyDeviceToHost, s));
    B200VS_CUDA(cudaStreamSynchronize(s));
    return B200VS_OK;
  });
}

int b200vs_reconstruct(b200vs_index* h, int64_t n, const int64_t* ids, float* out, uint8_t* found) {
  return guarded([&]() -> int {
    IndexBase* ix = get(h);
    if (n <= 0) return B200VS_OK;
    if (!ids || !out) fail(B200VS_EILLEGAL_PARAMETERS, "null ids / output");
    ix->reconstruct(n, ids, out, found);
    return B200VS_OK;
  });
}
int b200vs_sub_type(b200vs_index* h) {
  int r = -1;
  guarded([&]() -> int { IndexBase* ix = get(h); std::shared_lock<std::shared_mutex> rl(ix->rw); r = ix->sub_type(); return B200VS_OK; });
  return r;
}

int b200vs_count(b200vs_index* h, int64_t* count) {
  return guarded([&]() -> int { IndexBase* ix = get(h); std::shared_lock<std::shared_mutex> rl(ix->rw); if (count) *count = ix->count(); return B200VS_OK; });
}
int b200vs_deleted_count(b200vs_index* h, int64_t* count) {
  return guarded([&]() -> int { IndexBase* ix = get(h); std::shared_lock<std::shared_mutex> rl(ix->rw); if (count) *count = ix->deleted_count(); return B200VS_OK; });
}
int b200vs_memory_size(b200vs_index* h, int64_t* bytes) {
  return guarded([&]() -> int { IndexBase* ix = get(h); std::shared_lock<std::shared_mutex> rl(ix->rw); if (bytes) *bytes = ix->memory_size(); return B200VS_OK; });
}
int b200vs_is_trained(b200vs_index* h) {
  int r = 0;
  guarded([&]() -> int { IndexBase* ix = get(h); std::shared_lock<std::shared_mutex> rl(ix->rw); r = ix->is_trained() ? 1 : 0; return B200VS_OK; });
  return r;
}
int32_t b200vs_dimension(b200vs_index* h) { return h && h->impl ? h->impl->dim : -1; }

int b200vs_save(b200vs_index* h, const char* path) {
  return guarded([&]() -> int { if (!path) fail(B200VS_EILLEGAL_PARAMETERS, "null path"); get(h)->save(path); return B200VS_OK; });
}
int b200vs_load(b200vs_index* h, const char* path) {
  return guarded([&]() -> int { if (!path) fail(B200VS_EILLEGAL_PARAMETERS, "null path"); get(h)->load(path); return B200VS_OK; });
}

int b200vs_export_lists(b200vs_index* h, int64_t* list_off, float* vectors, uint8_t* codes, int64_t* ids) {
  return guarded([&]() -> int { get(h)->export_lists(list_off, vectors, codes, ids); return B200VS_OK; });
}

int b200vs_export_list(b200vs_index* h, int32_t list, int64_t cap, float* vectors, int64_t* ids, int64_t* count) {
  return guarded([&]() -> int {
    if (cap < 0) fail(B200VS_EILLEGAL_PARAMETERS, "bad capacity");
    const int64_t n = get(h)->export_list(list, cap, vectors, ids);
    if (count) *count = n;
    return B200VS_OK;
  });
}

int b200vs_merge_topk_device(int32_t device, int32_t nparts, int64_t nq, int32_t k, const float* parts_dist,
                             const int64_t* parts_ids, float* out_dist, int64_t* out_ids, void* stream) {
  return guarded([&]() -> int {
    if (nparts <= 0 || nq <= 0 || k <= 0 || !parts_dist || !parts_ids || !out_dist || !out_ids) fail(B200VS_EILLEGAL_PARAMETERS, "bad merge arguments");
    B200VS_CUDA(cudaSetDevice(device));
    launch_merge_api(nparts, nq, k, parts_dist, (const long long*)parts_ids, out_dist, (long long*)out_ids, (cudaStream_t)stream);
    return B200VS_OK;
  });
}

// ---- VectorCalcDistance: pairwise distance matrix (src/vector/vector_index_utils.cc:48-124, :193-419) ----
int b200vs_calc_distance(int32_t device, int32_t algorithm, b200vs_metric metric, int32_t dim, int64_t nl, const float* left,
                         int64_t nr, const float* right, float* out, float* left_out, float* right_out) {
  return guarded([&]() -> int {
    if (algorithm != B200VS_ALGORITHM_FAISS && algorithm != B200VS_ALGORITHM_HNSWLIB)
      fail(B200VS_EILLEGAL_PARAMETERS, "invalid algorithm type : ALGORITHM_NONE");      // utils.cc:70-76
    if (metric != B200VS_L2 && metric != B200VS_IP && metric != B200VS_COSINE)
      fail(B200VS_EILLEGAL_PARAMETERS, "invalid metric_type type : METRIC_TYPE_NONE");   // utils.cc:151-157
    if (dim <= 0 || nl < 0 || nr < 0) fail(B200VS_EILLEGAL_PARAMETERS, "bad distance-matrix shape");
    if (nl == 0 || nr == 0) return B200VS_OK;  // CalcDistanceCore over empty operands: empty result
    if (!left || !right || !out) fail(B200VS_EILLEGAL_PARAMETERS, "null operand");
    B200VS_CUDA(cudaSetDevice(device));
    cudaStream_t s = nullptr;
    B200VS_CUDA(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
    DevBuf<float> dl, dr, dn, dout;
    try {
      dl.reserve((size_t)nl * dim, 0, s); dr.reserve((size_t)nr * dim, 0, s); dout.reserve((size_t)nl * nr, 0, s);
      B200VS_CUDA(cudaMemcpyAsync(dl.p, left, (size_t)nl * dim * 4, cudaMemcpyHostToDevice, s));
      B200VS_CUDA(cudaMemcpyAsync(dr.p, right, (size_t)nr * dim * 4, cudaMemcpyHostToDevice, s));
      if (metric == B200VS_COSINE) {
        if (algorithm == B200VS_ALGORITHM_FAISS) {  // NormalizeVectorForFaiss on copies, utils.cc:283-284
          launch_normalize_faiss(dl.p, nl, dim, s);
          launch_normalize_faiss(dr.p, nr, dim, s);
        } else {                                    // NormalizeVectorForHnsw, utils.cc:407-413 (out of place)
          dn.reserve((size_t)std::max(nl, nr) * dim, 0, s);
          launch_normalize_hnsw(dl.p, dn.p, nl, dim, s);
          B200VS_CUDA(cudaMemcpyAsync(dl.p, dn.p, (size_t)nl * dim * 4, cudaMemcpyDeviceToDevice, s));
          launch_normalize_hnsw(dr.p, dn.p, nr, dim, s);
          B200VS_CUDA(cudaMemcpyAsync(dr.p, dn.p, (size_t)nr * dim * 4, cudaMemcpyDeviceToDevice, s));
        }
      }
      launch_pair_distance(metric == B200VS_L2, dl.p, nl, dr.p, nr, dim, dout.p, s);
      B200VS_CUDA(cudaMemcpyAsync(out, dout.p, (size_t)nl * nr * 4, cudaMemcpyDeviceToHost, s));
      if (left_out) B200VS_CUDA(cudaMemcpyAsync(left_out, dl.p, (size_t)nl * dim * 4, cudaMemcpyDeviceToHost, s));
      if (right_out) B200VS_CUDA(cudaMemcpyAsync(right_out, dr.p, (size_t)nr * dim * 4, cudaMemcpyDeviceToHost, s));
      B200VS_CUDA(cudaStreamSynchronize(s));
    } catch (...) {
      cudaStreamSynchronize(s); dl.free(); dr.free(); dn.free(); dout.free(); cudaStreamDestroy(s);
      throw;
    }
    dl.free(); dr.free(); dn.free(); dout.free();
    cudaStreamDestroy(s);
    return B200VS_OK;
  });
}

// ---- binary (Hamming) indexes ----
int b200vs_train_binary(b200vs_index* h, int64_t n, const uint8_t* x) {
  return guarded([&]() -> int {
    IndexBase* ix = get(h);
    require_binary(ix);
    if (n <= 0 || !x) fail(B200VS_EILLEGAL_PARAMETERS, "data size invalid");
    ix->train_binary(n, x);
    return B200VS_OK;
  });
}

int b200vs_add_binary_with_ids(b200vs_index* h, int64_t n, const uint8_t* x, const int64_t* ids, int upsert) {
  return guarded([&]() -> int {
    IndexBase* ix = get(h);
    require_binary(ix);
    if (n <= 0 || !x || !ids) fail(B200VS_EILLEGAL_PARAMETERS, "vector_with_ids is empty");
    ix->add_binary(n, x, ids, upsert != 0);
    return B200VS_OK;
  });
}

int b200vs_search_binary_device(b200vs_index* h, int64_t nq, const uint8_t* xq_dev, int32_t k, const b200vs_search_params* sp,
                                float* out_dist_dev, int64_t* out_ids_dev, void* stream) {
  return guarded([&]() -> int {
    IndexBase* ix = get(h);
    require_binary(ix);
    check_search_args(ix, nq, xq_dev, sp);
    if (k <= 0) return B200VS_OK;
    if (!out_ids_dev) fail(B200VS_EILLEGAL_PARAMETERS, "null output");
    std::shared_lock<std::shared_mutex> rl(ix->rw);
    ix->set_device();
    LaneGuard lane(ix, (cudaStream_t)stream);
    ix->reset_stats();
    SearchCtx sc = make_ctx(ix, sp, lane.stream);
    ix->search_binary_dev(nq, xq_dev, k, sc, out_dist_dev, (long long*)out_ids_dev, lane.stream);
    ix->phases_finish(lane.stream);
    if (!stream) B200VS_CUDA(cudaStreamSynchronize(lane.stream));
    return B200VS_OK;
  });
}

int b200vs_search_binary(b200vs_index* h, int64_t nq, const uint8_t* xq, int32_t k, const b200vs_search_params* sp, float* out_dist,
                         int64_t* out_ids) {
  return guarded([&]() -> int {
    IndexBase* ix = get(h);
    require_binary(ix);
    check_search_args(ix, nq, xq, sp);
    if (k <= 0) return B200VS_OK;
    if (!out_ids || !out_dist) fail(B200VS_EILLEGAL_PARAMETERS, "null output");
    std::shared_lock<std::shared_mutex> rl(ix->rw);
    ix->set_device();
    LaneGuard lane(ix, nullptr);
    cudaStream_t s = lane.stream;
    ix->reset_stats();
    const size_t qbytes = (size_t)nq * (ix->dim / 8);
    uint8_t* dq = ix->scratch.alloc<uint8_t>(qbytes);
    float* dd = ix->scratch.alloc<float>((size_t)nq * k);
    long long* di = ix->scratch.alloc<long long>((size_t)nq * k);
    B200VS_CUDA(cudaMemcpyAsync(dq, xq, qbytes, cudaMemcpyHostToDevice, s));
    SearchCtx sc = make_ctx(ix, sp, s);
    ix->search_binary_dev(nq, dq, k, sc, dd, di, s);
    ix->phases_finish(s);
    B200VS_CUDA(cudaMemcpyAsync(out_dist, dd, (size_t)nq * k * 4, cudaMemcpyDeviceToHost, s));
    B200VS_CUDA(cudaMemcpyAsync(out_ids, di, (size_t)nq * k * 8, cudaMemcpyDeviceToHost, s));
    B200VS_CUDA(cudaStreamSynchronize(s));
    return B200VS_OK;
  });
}

int b200vs_range_search_binary(b200vs_index* h, int64_t nq, const uint8_t* xq, float radius, int32_t max_results,
                               const b200vs_search_params* sp, float* out_dist, int64_t* out_ids, int32_t* out_counts) {
  return guarded([&]() -> int {
    IndexBase* ix = get(h);
    require_binary(ix);
    check_search_args(ix, nq, xq, sp);
    if (max_results <= 0 || !out_ids || !out_dist || !out_counts) fail(B200VS_EILLEGAL_PARAMETERS, "bad range-search outputs");
    std::shared_lock<std::shared_mutex> rl(ix->rw);
    ix->set_device();
    LaneGuard lane(ix, nullptr);
    cudaStream_t s = lane.stream;
    const size_t qbytes = (size_t)nq * (ix->dim / 8);
    uint8_t* dq = ix->scratch.alloc<uint8_t>(qbytes);
    float* dd = ix->scratch.alloc<float>((size_t)nq * max_results);
    long long* di = ix->scratch.alloc<long long>((size_t)nq * max_results);
    int* dc = ix->scratch.alloc<int>((size_t)nq);
    B200VS_CUDA(cudaMemcpyAsync(dq, xq, qbytes, cudaMemcpyHostToDevice, s));
    SearchCtx sc = make_ctx(ix, sp, s);
    ix->range_search_binary_dev(nq, dq, radius, max_results, sc, dd, di, dc, s);
    B200VS_CUDA(cudaMemcpyAsync(out_dist, dd, (size_t)nq * max_results * 4, cudaMemcpyDeviceToHost, s));
    B200VS_CUDA(cudaMemcpyAsync(out_ids, di, (size_t)nq * max_results * 8, cudaMemcpyDeviceToHost, s));
    B200VS_CUDA(cudaMemcpyAsync(out_counts, dc, (size_t)nq * 4, cudaMemcpyDeviceToHost, s));
    B200VS_CUDA(cudaStreamSynchronize(s));
    return B200VS_OK;
  });
}

// VectorCalcDistance, METRIC_TYPE_HAMMING (vector_index_utils.cc:146-149, :333-356)
int b200vs_calc_distance_binary(int32_t device, int32_t dim_bits, int64_t nl, const uint8_t* left, int64_t nr, const uint8_t* right,
                                float* out) {
  return guarded([&]() -> int {
    if (dim_bits <= 0 || dim_bits % 8 != 0 || dim_bits > 32768 || nl < 0 || nr < 0) fail(B200VS_EILLEGAL_PARAMETERS, "bad distance-matrix shape");
    if (nl == 0 || nr == 0) return B200VS_OK;
    if (!left || !right || !out) fail(B200VS_EILLEGAL_PARAMETERS, "null operand");
    B200VS_CUDA(cudaSetDevice(device));
    cudaStream_t s = nullptr;
    B200VS_CUDA(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
    try {
      binary_pair_distance(dim_bits, nl, left, nr, right, out, s);
    } catch (...) {
      cudaStreamSynchronize(s); cudaStreamDestroy(s);
      throw;
    }
    cudaStreamDestroy(s);
    return B200VS_OK;
  });
}

// ---- streaming brute-force scan: VectorReader::BruteForceSearch (src/vector/vector_reader.cc:1873-2048) ----
struct b200vs_scan {
  IndexBase* flat = nullptr;  // one tile at a time
  int64_t nq = 0;
  int k = 0;
  bool has_sp = false;
  b200vs_search_params sp{};
  std::vector<int64_t> allow;  // private copy of sp.sorted_ids (the caller's array need not outlive scan_begin)
  cudaStream_t s = nullptr;
  DevBuf<float> q, parts_d, out_d;      // parts = [2, nq, k]: running result, tile result
  DevBuf<long long> parts_i, out_i;
  int64_t pushed = 0;
  ~b200vs_scan() {
    if (flat) { cudaSetDevice(flat->device); }
    if (s) cudaStreamSynchronize(s);
    q.free(); parts_d.free(); out_d.free(); parts_i.free(); out_i.free();
    delete flat;
    if (s) cudaStreamDestroy(s);
  }
};

int b200vs_scan_begin(int32_t device, b200vs_metric metric, int32_t dim, int64_t nq, const float* xq, int32_t k,
                      const b200vs_search_params* sp, b200vs_scan** out) {
  return guarded([&]() -> int {
    if (!out) fail(B200VS_EILLEGAL_PARAMETERS, "out is null");
    *out = nullptr;
    if (dim <= 0) fail(B200VS_EVECTOR_INVALID, "vector index dimension is invalid");  // vector_reader.cc:1889-1894
    if (metric != B200VS_L2 && metric != B200VS_IP && metric != B200VS_COSINE) fail(B200VS_EILLEGAL_PARAMETERS, "unsupported metric type");
    if (nq <= 0 || !xq) fail(B200VS_EILLEGAL_PARAMETERS, "vector_with_ids is empty");
    if (k <= 0) fail(B200VS_EILLEGAL_PARAMETERS, "topk must be > 0");
    b200vs_params p{};
    p.device = device;
    std::unique_ptr<b200vs_scan> st(new b200vs_scan());
    st->flat = make_flat(metric, dim, p);
    st->nq = nq; st->k = k;
    if (sp) {
      st->has_sp = true; st->sp = *sp;
      if (sp->sorted_ids && sp->n_ids > 0) st->allow.assign(sp->sorted_ids, sp->sorted_ids + sp->n_ids);
      st->sp.sorted_ids = sp->sorted_ids ? st->allow.data() : nullptr;
    }
    B200VS_CUDA(cudaSetDevice(device));
    B200VS_CUDA(cudaStreamCreateWithFlags(&st->s, cudaStreamNonBlocking));
    const size_t nk = (size_t)nq * k;
    st->q.reserve((size_t)nq * dim, 0, st->s);
    st->parts_d.reserve(2 * nk, 0, st->s); st->parts_i.reserve(2 * nk, 0, st->s);
    st->out_d.reserve(nk, 0, st->s); st->out_i.reserve(nk, 0, st->s);
    B200VS_CUDA(cudaMemcpyAsync(st->q.p, xq, (size_t)nq * dim * 4, cudaMemcpyHostToDevice, st->s));
    B200VS_CUDA(cudaMemsetAsync(st->parts_d.p, 0, 2 * nk * 4, st->s));
    B200VS_CUDA(cudaMemsetAsync(st->parts_i.p, 0xFF, 2 * nk * 8, st->s));  // id -1 = empty slot
    B200VS_CUDA(cudaStreamSynchronize(st->s));
    *out = st.release();
    return B200VS_OK;
  });
}

int b200vs_scan_push(b200vs_scan* st, int64_t n, const float* x, const int64_t* ids) {
  return guarded([&]() -> int {
    if (!st || !st->flat) fail(B200VS_EILLEGAL_PARAMETERS, "null scan handle");
    if (n <= 0) return B200VS_OK;
    if (!x || !ids) fail(B200VS_EILLEGAL_PARAMETERS, "null tile");
    IndexBase* ix = st->flat;
    const size_t nk = (size_t)st->nq * st->k;
    if (st->pushed > 0) ix->clear();
    ix->add(n, x, ids, false);  // one temporary Flat index per tile, as the reference builds (vector_reader.cc:1937-1946)
    {
      std::shared_lock<std::shared_mutex> rl(ix->rw);
      ix->set_device();
      LaneGuard lane(ix, st->s);
      ix->reset_stats();
      SearchCtx sc = make_ctx(ix, st->has_sp ? &st->sp : nullptr, st->s);
      ix->search_dev(st->nq, st->q.p, st->k, sc, st->parts_d.p + nk, st->parts_i.p + nk, st->s);
    }
    // running top-k <- merge(running, tile): the reference's per-query priority queues (:1956-1971)
    launch_merge_api(2, st->nq, st->k, st->parts_d.p, st->parts_i.p, st->out_d.p, st->out_i.p, st->s);
    B200VS_CUDA(cudaMemcpyAsync(st->parts_d.p, st->out_d.p, nk * 4, cudaMemcpyDeviceToDevice, st->s));
    B200VS_CUDA(cudaMemcpyAsync(st->parts_i.p, st->out_i.p, nk * 8, cudaMemcpyDeviceToDevice, st->s));
    B200VS_CUDA(cudaStreamSynchronize(st->s));  // the next push rewrites the tile index
    st->pushed += n;
    return B200VS_OK;
  });
}

int b200vs_scan_finish(b200vs_scan* st, float* out_dist, int64_t* out_ids) {
  const int rc = guarded([&]() -> int {
    if (!st || !st->flat) fail(B200VS_EILLEGAL_PARAMETERS, "null scan handle");
    if (!out_dist || !out_ids) fail(B200VS_EILLEGAL_PARAMETERS, "null output");
    B200VS_CUDA(cudaSetDevice(st->flat->device));
    const size_t nk = (size_t)st->nq * st->k;
    B200VS_CUDA(cudaMemcpyAsync(out_dist, st->parts_d.p, nk * 4, cudaMemcpyDeviceToHost, st->s));
    B200VS_CUDA(cudaMemcpyAsync(out_ids, st->parts_i.p, nk * 8, cudaMemcpyDeviceToHost, st->s));
    B200VS_CUDA(cudaStreamSynchronize(st->s));
    return B200VS_OK;
  });
  delete st;
  return rc;
}

void b200vs_scan_abort(b200vs_scan* st) { delete st; }

int b200vs_last_phase_times(b200vs_index* h, float ms[16]) {
  return guarded([&]() -> int {
    IndexBase* ix = get(h);
    for (int i = 0; i < 16; ++i) ms[i] = i < IndexBase::PH_COUNT ? ix->phase_ms[i] : 0.f;
    return B200VS_OK;
  });
}

int b200vs_last_search_stats(b200vs_index* h, int64_t stats[8]) {
  return guarded([&]() -> int { IndexBase* ix = get(h); for (int i = 0; i < 8; ++i) stats[i] = ix->stats[i]; return B200VS_OK; });
}

int b200vs_set_profiling(b200vs_index* h, int on) {
  return guarded([&]() -> int { get(h)->profiling = on != 0; return B200VS_OK; });
}

const char* b200vs_last_error(void) { return g_last_error.c_str(); }
const char* b200vs_version(void) { return "b200vs 0.1 (sm_100a)"; }

}  // extern "C"

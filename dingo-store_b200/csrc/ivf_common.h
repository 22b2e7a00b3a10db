// ivf_common.h — inverted-list bookkeeping and GPU k-means shared by IVF-Flat and IVF-PQ.
//
// Inverted lists live in ONE device arena (rows of the payload array), list l owning rows
// [off, off+len) with capacity cap >= len.  Appends go in place; a full list is relocated to the arena
// tail with 1.5x capacity; removals tombstone the row (id = -1) and a compaction pass rebuilds the arena when
// garbage + tombstones outweigh live rows.  Lists stay contiguous so the scan kernels stream them with
// 128-B coalesced loads / TMA tiles.  Replaces faiss::ArrayInvertedLists behind IndexIVFFlat/IndexIVFPQ
// (constructed at src/vector/vector_index_ivf_flat.cc:809-816, vector_index_raw_ivf_pq.cc:554-564).
#pragma once
#include <algorithm>
#include <random>
#include <unordered_map>
#include <vector>

#include "index.h"

namespace b200vs {

struct ListMeta {
  int64_t off = 0;
  int32_t len = 0;  // rows in use (live + tombstones)
  int32_t cap = 0;
  int32_t dead = 0;
};

struct IvfLists {
  std::vector<ListMeta> lists;
  std::vector<int64_t> h_ids;  // arena mirror of ids (-1 = tombstone / unused)
  std::unordered_multimap<int64_t, uint64_t> where;  // id -> (list << 32 | pos)
  int64_t arena_used = 0, arena_used_before = 0, arena_cap = 0;
  int64_t live = 0, dead = 0, garbage = 0;
  int64_t total_chunks = 0;      // sum of ceil(len / 512) — tensor-core work-item bound (tc_scan.cuh TC_CHUNK = 512)
  int max_chunks_per_list = 0;
  int nonempty_lists = 0;        // lists that hold rows here (a list-sharded rank owns only some)
  DevBuf<long long> d_off;
  DevBuf<int> d_len;
  // compaction plan
  std::vector<ListMeta> plan_lists;
  std::vector<int64_t> plan_ids;
  int64_t plan_rows = 0;

  void init(int nlist, cudaStream_t s) {
    lists.assign(nlist, ListMeta());
    h_ids.clear(); where.clear();
    arena_used = arena_used_before = arena_cap = 0;
    live = dead = garbage = 0;
    d_off.free(); d_len.free();
    d_off.reserve(nlist, 0, s);
    d_len.reserve(nlist, 0, s);
    upload(s);
  }
  int64_t total_len() const { return live + dead; }

  void upload(cudaStream_t s) {
    const size_t n = lists.size();
    std::vector<long long> off(n);
    std::vector<int> len(n);
    total_chunks = 0; max_chunks_per_list = 0; nonempty_lists = 0;
    for (size_t i = 0; i < n; ++i) {
      off[i] = lists[i].off; len[i] = lists[i].len;
      const int c = (lists[i].len + 511) / 512;
      total_chunks += c; max_chunks_per_list = std::max(max_chunks_per_list, c);
      if (lists[i].len > 0) ++nonempty_lists;
    }
    B200VS_CUDA(cudaMemcpyAsync(d_off.p, off.data(), n * 8, cudaMemcpyHostToDevice, s));
    B200VS_CUDA(cudaMemcpyAsync(d_len.p, len.data(), n * 4, cudaMemcpyHostToDevice, s));
    B200VS_CUDA(cudaStreamSynchronize(s));  // host vectors die here
  }

  static int32_t round32(int64_t v) { return (int32_t)((v + 31) / 32 * 32); }

  // make room for need[l] more rows in every list. grow(rows): enlarge payload arrays to `rows` keeping
  // arena_used_before rows; move(src,dst,len): device copy of a relocated list.
  template <class Grow, class Move>
  void reserve_for(const std::vector<int>& need, Grow grow, Move move) {
    struct Rel { int l; int64_t src, dst; int32_t len; };
    std::vector<Rel> rels;
    arena_used_before = arena_used;
    for (size_t l = 0; l < lists.size(); ++l) {
      if (need[l] == 0) continue;
      ListMeta& m = lists[l];
      if (m.len + need[l] <= m.cap) continue;
      const int32_t ncap = round32(std::max<int64_t>(64, ((int64_t)m.len + need[l]) * 3 / 2));
      rels.push_back({(int)l, m.off, arena_used, m.len});
      garbage += m.cap;
      m.off = arena_used; m.cap = ncap;
      arena_used += ncap;
    }
    if (arena_used > arena_cap) {
      const int64_t ncap = std::max<int64_t>(arena_used, arena_cap * 3 / 2);
      grow(ncap);
      arena_cap = ncap;
    }
    h_ids.resize(arena_cap, -1);
    for (const Rel& r : rels) {
      if (r.len == 0) continue;
      move(r.src, r.dst, (int64_t)r.len);
      std::copy(h_ids.begin() + r.src, h_ids.begin() + r.src + r.len, h_ids.begin() + r.dst);
    }
  }

  int64_t append(int l, int64_t id) {
    ListMeta& m = lists[l];
    const int64_t row = m.off + m.len;
    where.emplace(id, ((uint64_t)l << 32) | (uint32_t)m.len);
    h_ids[row] = id;
    m.len++;
    live++;
    return row;
  }

  // faiss remove_ids(IDSelectorBatch): every entry whose id matches is removed
  void remove_ids(int64_t n, const int64_t* del, std::vector<int64_t>& rows) {
    for (int64_t i = 0; i < n; ++i) {
      auto range = where.equal_range(del[i]);
      for (auto it = range.first; it != range.second; ++it) {
        const int l = (int)(it->second >> 32);
        const uint32_t pos = (uint32_t)(it->second & 0xffffffffu);
        const int64_t row = lists[l].off + pos;
        if (h_ids[row] < 0) continue;
        h_ids[row] = -1;
        lists[l].dead++;
        rows.push_back(row);
        live--; dead++;
      }
      where.erase(range.first, range.second);
    }
  }

  bool needs_compaction() const { return garbage + dead > std::max<int64_t>(live, 4096); }

  int64_t plan_compaction(std::vector<long long>& src, std::vector<long long>& dst) {
    plan_lists.assign(lists.size(), ListMeta());
    int64_t used = 0;
    src.clear(); dst.clear();
    for (size_t l = 0; l < lists.size(); ++l) {
      const ListMeta& m = lists[l];
      const int32_t nlive = m.len - m.dead;
      ListMeta& pm = plan_lists[l];
      pm.off = used; pm.len = 0; pm.dead = 0;
      pm.cap = nlive ? round32((int64_t)nlive * 5 / 4 + 32) : 0;
      for (int p = 0; p < m.len; ++p) {
        if (h_ids[m.off + p] < 0) continue;
        src.push_back(m.off + p);
        dst.push_back(pm.off + pm.len);
        pm.len++;
      }
      used += pm.cap;
    }
    plan_rows = used;
    plan_ids.assign(std::max<int64_t>(used, 1), -1);
    for (size_t i = 0; i < src.size(); ++i) plan_ids[dst[i]] = h_ids[src[i]];
    return used;
  }
  void commit_compaction() {
    lists.swap(plan_lists);
    h_ids.swap(plan_ids);
    arena_used = arena_used_before = plan_rows;
    arena_cap = std::max<int64_t>(plan_rows, 1);
    garbage = 0; dead = 0;
    where.clear();
    for (size_t l = 0; l < lists.size(); ++l)
      for (int p = 0; p < lists[l].len; ++p) where.emplace(h_ids[lists[l].off + p], ((uint64_t)l << 32) | (uint32_t)p);
    plan_lists.clear(); plan_ids.clear();
  }
};

void launch_kmeans_accumulate(const float* x, const long long* assign, int64_t n, int d, float* sums, int* counts,
                              cudaStream_t s);

// faiss rand_perm (public algorithm): the training subsample and the initial centroids of kmeans_gpu
inline void kmeans_rand_perm(std::vector<int64_t>& perm, int64_t m, int64_t sd) {
  perm.resize(m);
  for (int64_t i = 0; i < m; ++i) perm[i] = i;
  std::mt19937 mt((unsigned)sd);
  for (int64_t i = 0; i + 1 < m; ++i) { int64_t i2 = i + (int64_t)(mt() % (unsigned long)(m - i)); std::swap(perm[i], perm[i2]); }
}

// faiss::Clustering-shaped Lloyd k-means with the assignment step on the GPU (public algorithm; the
// reference reaches it through index_->train at vector_index_ivf_flat.cc:695 / raw_ivf_pq.cc:485).
// x_host RAW rows; cosine rows are normalised on the device first.  `assign(xd, m, cd, k, out)` labels m device
// rows against the k device centroids cd; `prepare_ids(k)` lets the caller size its centroid-id array.
template <class AssignFn, class PrepFn>
void kmeans_gpu(IndexBase* ix, b200vs_metric metric, int d, int64_t n, const float* x_host, int k, int niter,
                int max_pts, int64_t seed, std::vector<float>& cent, AssignFn assign, PrepFn prepare_ids) {
  cudaStream_t s = ix->stream;
  auto rand_perm = kmeans_rand_perm;
  std::vector<float> sub;
  const float* xs = x_host;
  int64_t m = n;
  if (n > (int64_t)k * max_pts) {
    std::vector<int64_t> perm;
    rand_perm(perm, n, seed);
    m = (int64_t)k * max_pts;
    sub.resize((size_t)m * d);
    for (int64_t i = 0; i < m; ++i) memcpy(&sub[(size_t)i * d], x_host + (size_t)perm[i] * d, (size_t)d * 4);
    xs = sub.data();
  }
  DevBuf<float> xd, cd, sums;
  DevBuf<int> counts;
  DevBuf<long long> asg;
  xd.reserve((size_t)m * d, 0, s);
  B200VS_CUDA(cudaMemcpyAsync(xd.p, xs, (size_t)m * d * 4, cudaMemcpyHostToDevice, s));
  if (metric == B200VS_COSINE) launch_normalize_faiss(xd.p, m, d, s);
  B200VS_CUDA(cudaStreamSynchronize(s));
  cent.assign((size_t)k * d, 0.f);
  std::vector<float> hx;  // normalised copy for initialisation when cosine
  const float* init_src = xs;
  if (metric == B200VS_COSINE) {
    hx.resize((size_t)m * d);
    B200VS_CUDA(cudaMemcpy(hx.data(), xd.p, (size_t)m * d * 4, cudaMemcpyDeviceToHost));
    init_src = hx.data();
  }
  if (m == k) { memcpy(cent.data(), init_src, (size_t)m * d * 4); return; }
  {
    std::vector<int64_t> perm;
    rand_perm(perm, m, seed + 1);
    for (int i = 0; i < k; ++i) memcpy(&cent[(size_t)i * d], init_src + (size_t)perm[i] * d, (size_t)d * 4);
  }
  prepare_ids(k);
  cd.reserve((size_t)k * d, 0, s);
  sums.reserve((size_t)k * d, 0, s);
  counts.reserve(k, 0, s);
  asg.reserve(m, 0, s);
  std::vector<float> hs((size_t)k * d);
  std::vector<int> hc(k);
  for (int it = 0; it < niter; ++it) {
    B200VS_CUDA(cudaMemcpyAsync(cd.p, cent.data(), (size_t)k * d * 4, cudaMemcpyHostToDevice, s));
    assign(xd.p, m, cd.p, k, asg.p);
    B200VS_CUDA(cudaMemsetAsync(sums.p, 0, (size_t)k * d * 4, s));
    B200VS_CUDA(cudaMemsetAsync(counts.p, 0, (size_t)k * 4, s));
    launch_kmeans_accumulate(xd.p, asg.p, m, d, sums.p, counts.p, s);
    B200VS_CUDA(cudaMemcpyAsync(hs.data(), sums.p, (size_t)k * d * 4, cudaMemcpyDeviceToHost, s));
    B200VS_CUDA(cudaMemcpyAsync(hc.data(), counts.p, (size_t)k * 4, cudaMemcpyDeviceToHost, s));
    B200VS_CUDA(cudaStreamSynchronize(s));
    std::vector<float> hassign(k);
    for (int c = 0; c < k; ++c) {
      hassign[c] = (float)hc[c];
      if (hc[c] == 0) continue;
      const float inv = 1.0f / (float)hc[c];
      for (int j = 0; j < d; ++j) cent[(size_t)c * d + j] = hs[(size_t)c * d + j] * inv;
    }
    // split_clusters (faiss public algorithm): refill empty clusters from big ones with a +-1/1024 perturbation
    const float EPS = 1 / 1024.;
    std::mt19937 mt(1234);
    for (int ci = 0; ci < k; ++ci) {
      if (hassign[ci] != 0) continue;
      int cj;
      for (cj = 0;; cj = (cj + 1) % k) {
        const float p = (hassign[cj] - 1.0f) / (float)(m - k);
        const float r = mt() / float(mt.max());
        if (r < p) break;
      }
      memcpy(&cent[(size_t)ci * d], &cent[(size_t)cj * d], (size_t)d * 4);
      for (int j = 0; j < d; ++j) {
        if (j % 2 == 0) { cent[(size_t)ci * d + j] *= 1 + EPS; cent[(size_t)cj * d + j] *= 1 - EPS; }
        else            { cent[(size_t)ci * d + j] *= 1 - EPS; cent[(size_t)cj * d + j] *= 1 + EPS; }
      }
      hassign[ci] = hassign[cj] / 2;
      hassign[cj] -= hassign[ci];
    }
  }
  ix->launch_count(2 * niter);
}

void check_batch_ids_unique(int64_t n, const int64_t* ids);
void fill_empty_results(int64_t nq, int k, float* od, long long* oi, cudaStream_t s);

}  // namespace b200vs

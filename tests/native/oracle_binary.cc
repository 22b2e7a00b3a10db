// oracle_binary.cc — CPU oracle of the binary (Hamming) indexes (TEST INFRASTRUCTURE, see oracle_binary.h).
#include "oracle_binary.h"

#include "../../oracle/oracle_common.h"

using oracle::filter_pass;
using oracle::parallel_blocks;
using oracle::parallel_for;
using oracle::TopK;

namespace {

// the radius faiss binary range_search receives: static_cast<int>(radius) (flat.cc:282-311, ivf_flat.cc:342-345)
int int_radius(float radius) { return static_cast<int>(radius); }

// top-k (or range hits) of one query over rows [r0, r1) of xb
void scan_rows(int32_t dim, const uint8_t* xb, const int64_t* ids, int64_t r0, int64_t r1, const uint8_t* q, const oracle_filter* filt,
               bool range, int radius, TopK& top) {
  const size_t code = (size_t)dim / 8;
  for (int64_t r = r0; r < r1; ++r) {
    const int64_t id = ids[r];
    if (id < 0 || !filter_pass(filt, id)) continue;
    const int32_t d = oracle_hamming(q, xb + (size_t)r * code, dim);
    if (range && !(d < radius)) continue;
    top.push((float)d, id);
  }
}

// the nprobe nearest centroids by (distance, list id): the IndexBinaryFlat quantiser with the engine's tie rule
void probes_of(int32_t dim, int32_t nlist, const uint8_t* centroids, const uint8_t* q, int32_t nprobe, std::vector<int64_t>& out) {
  TopK top(nprobe, false);
  for (int32_t c = 0; c < nlist; ++c) top.push((float)oracle_hamming(q, centroids + (size_t)c * (dim / 8), dim), c);
  std::vector<float> d(nprobe);
  out.assign(nprobe, -1);
  top.finish(d.data(), out.data());
}

}  // namespace

extern "C" {

int32_t oracle_hamming(const uint8_t* a, const uint8_t* b, int32_t dim) {
  const int32_t nb = dim / 8;
  int32_t d = 0, i = 0;
  for (; i + 8 <= nb; i += 8) {
    uint64_t x, y;
    memcpy(&x, a + i, 8);
    memcpy(&y, b + i, 8);
    d += __builtin_popcountll(x ^ y);
  }
  for (; i < nb; ++i) d += __builtin_popcount((unsigned)(a[i] ^ b[i]));
  return d;
}

int oracle_binary_flat_search(int32_t dim, int64_t n, const uint8_t* xb, const int64_t* ids, int64_t nq, const uint8_t* xq,
                              int32_t k, const oracle_filter* filt, int nthreads, float* out_dist, int64_t* out_ids) {
  if (dim <= 0 || dim % 8 || k <= 0) return -1;
  parallel_for(nq, nthreads, [&](int64_t qi) {
    TopK top(k, false);
    scan_rows(dim, xb, ids, 0, n, xq + (size_t)qi * (dim / 8), filt, false, 0, top);
    top.finish(out_dist + qi * k, out_ids + qi * k);
  });
  return 0;
}

int oracle_binary_flat_range_search(int32_t dim, int64_t n, const uint8_t* xb, const int64_t* ids, int64_t nq, const uint8_t* xq,
                                    float radius, int32_t max_results, const oracle_filter* filt, int nthreads, float* out_dist,
                                    int64_t* out_ids, int32_t* out_counts) {
  if (dim <= 0 || dim % 8 || max_results <= 0) return -1;
  const int r = int_radius(radius);
  parallel_for(nq, nthreads, [&](int64_t qi) {
    TopK top(max_results, false);
    scan_rows(dim, xb, ids, 0, n, xq + (size_t)qi * (dim / 8), filt, true, r, top);
    out_counts[qi] = top.n;
    top.finish(out_dist + qi * max_results, out_ids + qi * max_results);
  });
  return 0;
}

void oracle_binary_to_real(int64_t n, int32_t dim, const uint8_t* x, float* out) {
  for (int64_t i = 0; i < n; ++i)
    for (int32_t b = 0; b < dim; ++b)
      out[(size_t)i * dim + b] = (x[(size_t)i * (dim / 8) + b / 8] >> (b % 8)) & 1 ? 1.0f : -1.0f;
}

void oracle_real_to_binary(int64_t n, int32_t dim, const float* x, uint8_t* out) {
  for (int64_t i = 0; i < n; ++i)
    for (int32_t j = 0; j < dim / 8; ++j) {
      uint8_t v = 0;
      for (int b = 0; b < 8; ++b) v |= (x[(size_t)i * dim + j * 8 + b] > 0 ? 1 : 0) << b;
      out[(size_t)i * (dim / 8) + j] = v;
    }
}

int oracle_binary_kmeans(int32_t dim, int64_t n, const uint8_t* x, int32_t k, int32_t niter, int32_t max_points_per_centroid,
                         int64_t seed, int nthreads, uint8_t* centroids) {
  if (dim <= 0 || dim % 8 || n < k) return -1;
  std::vector<float> real((size_t)n * dim), cent((size_t)k * dim);
  oracle_binary_to_real(n, dim, x, real.data());
  const int rc = oracle_kmeans(ORACLE_L2, dim, n, real.data(), k, niter, max_points_per_centroid, seed, nthreads, cent.data());
  if (rc != 0) return rc;
  oracle_real_to_binary(k, dim, cent.data(), centroids);
  return 0;
}

int oracle_binary_assign(int32_t dim, int64_t n, const uint8_t* x, int32_t nlist, const uint8_t* centroids, int nthreads,
                         int32_t* out_assign) {
  if (dim <= 0 || dim % 8 || nlist <= 0) return -1;
  parallel_blocks(n, nthreads, 256, [&](int64_t a, int64_t b) {
    for (int64_t i = a; i < b; ++i) {
      const uint8_t* xi = x + (size_t)i * (dim / 8);
      int32_t best = 0, bd = oracle_hamming(xi, centroids, dim);
      for (int32_t c = 1; c < nlist; ++c) {
        const int32_t d = oracle_hamming(xi, centroids + (size_t)c * (dim / 8), dim);
        if (d < bd) { bd = d; best = c; }
      }
      out_assign[i] = best;
    }
  });
  return 0;
}

static int ivf_search(int32_t dim, int32_t nlist, const uint8_t* centroids, const int64_t* list_off, const uint8_t* xb, const int64_t* ids,
                      int64_t nq, const uint8_t* xq, int32_t k, int32_t nprobe, const oracle_filter* filt, int nthreads, bool range,
                      float radius, float* out_dist, int64_t* out_ids, int32_t* out_counts) {
  if (dim <= 0 || dim % 8 || k <= 0 || nlist <= 0) return -1;
  nprobe = std::max(1, std::min(nprobe, nlist));
  const int r = int_radius(radius);
  parallel_for(nq, nthreads, [&](int64_t qi) {
    const uint8_t* q = xq + (size_t)qi * (dim / 8);
    std::vector<int64_t> probes;
    probes_of(dim, nlist, centroids, q, nprobe, probes);
    TopK top(k, false);
    for (int64_t l : probes)
      if (l >= 0) scan_rows(dim, xb, ids, list_off[l], list_off[l + 1], q, filt, range, r, top);
    if (out_counts) out_counts[qi] = top.n;
    top.finish(out_dist + qi * k, out_ids + qi * k);
  });
  return 0;
}

int oracle_binary_ivf_search(int32_t dim, int32_t nlist, const uint8_t* centroids, const int64_t* list_off, const uint8_t* xb,
                             const int64_t* ids, int64_t nq, const uint8_t* xq, int32_t k, int32_t nprobe, const oracle_filter* filt,
                             int nthreads, float* out_dist, int64_t* out_ids) {
  return ivf_search(dim, nlist, centroids, list_off, xb, ids, nq, xq, k, nprobe, filt, nthreads, false, 0.f, out_dist, out_ids, nullptr);
}

int oracle_binary_ivf_range_search(int32_t dim, int32_t nlist, const uint8_t* centroids, const int64_t* list_off, const uint8_t* xb,
                                   const int64_t* ids, int64_t nq, const uint8_t* xq, float radius, int32_t max_results,
                                   int32_t nprobe, const oracle_filter* filt, int nthreads, float* out_dist, int64_t* out_ids,
                                   int32_t* out_counts) {
  return ivf_search(dim, nlist, centroids, list_off, xb, ids, nq, xq, max_results, nprobe, filt, nthreads, true, radius, out_dist,
                    out_ids, out_counts);
}

int oracle_calc_distance_hamming(int32_t dim, int64_t nl, const uint8_t* left, int64_t nr, const uint8_t* right, float* out) {
  if (dim <= 0 || dim % 8) return -1;
  for (int64_t i = 0; i < nl; ++i)
    for (int64_t j = 0; j < nr; ++j)
      out[(size_t)i * nr + j] = (float)oracle_hamming(left + (size_t)i * (dim / 8), right + (size_t)j * (dim / 8), dim);
  return 0;
}

}  // extern "C"

// binary.cu — Hamming-space indexes: BINARY_FLAT and BINARY_IVF_FLAT (device-resident replacements of the
// faiss::IndexBinaryIDMap2 / faiss::IndexBinaryIVF objects held by VectorIndexFlat / VectorIndexIvfFlat<faiss::IndexBinary>,
// src/vector/vector_index_factory.cc:73-80, vector_index_flat.cc:63-71, vector_index_ivf_flat.cc:62, :75-80).
//
// Rows are stored zero-padded to a 16-byte stride, so every kernel reads them with 16-byte loads; queries are padded the
// same way on upload and the padding XORs to zero.  Distances are exact integers, carried through the shared top-k
// machinery (BlockSelect, merge_select_kernel) as the order-preserving key of float(distance), so the (distance, id) rule
// and the API output (float distance) come for free.  One scan kernel serves the Flat scan, the IVF list scan and the IVF
// coarse quantiser (a Flat search over the nlist centroids with ids 0..nlist-1 and k = nprobe).
#include <algorithm>
#include <cstring>

#include "index.h"
#include "ivf_common.h"
#include "scan_kernels.cuh"

namespace b200vs {

namespace {

constexpr int BIN_THREADS = 256;
constexpr int kMaxBinaryDim = 32768;  // bits; Constant::kVectorMaxDimension (constant.h:165)
constexpr double kMaxTrainFloatBytes = 16.0 * (1 << 30);  // the +-1 float copy of the training sample (train_binary)

inline int bin_words(int dim_bits) { return (dim_bits / 8 + 15) / 16; }  // 16-byte words per stored row

struct BinScanArgs {
  const uint4* rows;        // [rows, W]
  const long long* ids;     // [rows], < 0 = removed slot
  const uint4* queries;     // [nq, W]
  int W;
  int mode;                 // 0: one segment [0, n)   1: IVF probes (one query per CTA)
  long long n;
  const long long* probes;  // mode 1: [nq, nprobe] list ids (may contain -1)
  int nprobe;
  const long long* list_off;
  const int* list_len;
  long long nq;
  int k, nsplit, pool_cap;
  uint32_t* ws_kd;          // [nq, nsplit, k]
  long long* ws_kid;
  FilterDev filt;
  int has_thr;              // range search: keep distance < thr
  uint32_t thr_key;
};

__device__ __forceinline__ uint32_t popc4(const uint4 a, const uint4 b) {
  return __popc(a.x ^ b.x) + __popc(a.y ^ b.y) + __popc(a.z ^ b.z) + __popc(a.w ^ b.w);
}

// Grid (nsplit, ceil(nq / QT)).  A CTA keeps QT queries in shared memory and streams its share of the candidate rows once:
// one row per thread, Σ popc(q ^ r) over the row's 16-byte words for each resident query, candidates pushed into that
// query's BlockSelect pool.  Partial top-k lists go to ws [query, split, k] for merge_select_kernel.
template <int QT>
__global__ void __launch_bounds__(BIN_THREADS) hamming_scan_kernel(const BinScanArgs a) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int W = a.W;
  const long long q0 = (long long)blockIdx.y * QT;
  const int nqt = (int)min((long long)QT, a.nq - q0);
  const int split = blockIdx.x;
  uint4* qs = reinterpret_cast<uint4*>(smem);
  for (int i = threadIdx.x; i < QT * W; i += blockDim.x) {
    const int q = i / W;
    qs[i] = q < nqt ? a.queries[(size_t)(q0 + q) * W + (i - q * W)] : make_uint4(0u, 0u, 0u, 0u);
  }
  size_t off = (size_t)QT * W * 16;
  int* prefix = reinterpret_cast<int*>(smem + off);
  const int nseg = a.mode == 0 ? 1 : a.nprobe;
  off += ((size_t)(nseg + 1) * 4 + 15) / 16 * 16;
  const long long* myprobes = a.mode == 1 ? a.probes + (size_t)q0 * a.nprobe : nullptr;
  long long total = a.n;
  if (a.mode == 1) {
    if (threadIdx.x < 32) {  // warp-chunked exclusive scan of the probed list lengths
      int carry = 0;
      for (int base = 0; base < nseg; base += 32) {
        const int p = base + threadIdx.x;
        int len = 0;
        if (p < nseg) { const long long l = myprobes[p]; len = l >= 0 ? a.list_len[l] : 0; }
        int incl = len;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { int v = __shfl_up_sync(0xffffffffu, incl, o); if ((int)threadIdx.x >= o) incl += v; }
        if (p < nseg) prefix[p] = carry + incl - len;
        carry += __shfl_sync(0xffffffffu, incl, 31);
      }
      if (threadIdx.x == 0) prefix[nseg] = carry;
    }
    __syncthreads();
    total = prefix[nseg];
  }
  unsigned char* pools = smem + off;
  const size_t pool_bytes = BlockSelect::smem_bytes(a.pool_cap);
  auto sel = [&](int q) { BlockSelect s; s.attach(pools + q * pool_bytes, a.pool_cap, a.k); return s; };
  for (int q = 0; q < QT; ++q) sel(q).init(pools + q * pool_bytes, a.pool_cap, a.k);
  if (a.has_thr && threadIdx.x == 0)
    for (int q = 0; q < QT; ++q) { BlockSelect s = sel(q); *s.thr_d = a.thr_key; *s.thr_id = (long long)0x8000000000000000LL; }
  __syncthreads();

  auto map_row = [&](long long i) -> long long {
    if (a.mode == 0) return i;
    int lo = 0, hi = nseg - 1;  // last p with prefix[p] <= i
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if (prefix[mid] <= i) lo = mid; else hi = mid - 1;
    }
    return a.list_off[myprobes[lo]] + (i - prefix[lo]);
  };

  const long long r0 = total * split / a.nsplit, r1 = total * (split + 1) / a.nsplit;
  for (long long base = r0; base < r1; base += BIN_THREADS) {
    // room for one push per thread in every pool (the decision is block-uniform: all threads read the same counts)
    __syncthreads();
    unsigned full = 0;
    for (int q = 0; q < nqt; ++q) if (*sel(q).count + BIN_THREADS > a.pool_cap) full |= 1u << q;
    __syncthreads();
    for (int q = 0; q < nqt; ++q) if (full >> q & 1u) sel(q).prune();
    const long long i = base + threadIdx.x;
    if (i >= r1) continue;
    const long long row = map_row(i);
    const long long id = a.ids[row];
    if (id < 0 || !filter_pass(a.filt, id)) continue;
    uint32_t dist[QT];
#pragma unroll
    for (int q = 0; q < QT; ++q) dist[q] = 0;
    const uint4* rp = a.rows + (size_t)row * W;
#pragma unroll 4
    for (int w = 0; w < W; ++w) {
      const uint4 r = __ldg(rp + w);
#pragma unroll
      for (int q = 0; q < QT; ++q) dist[q] += popc4(r, qs[q * W + w]);
    }
#pragma unroll
    for (int q = 0; q < QT; ++q) {
      if (q >= nqt) break;
      const uint32_t key = f2ord((float)dist[q]);
      BlockSelect s = sel(q);
      if (s.passes(key, id)) s.push(key, id);
    }
  }
  for (int q = 0; q < nqt; ++q) sel(q).prune();
  for (int q = 0; q < nqt; ++q) {
    BlockSelect s = sel(q);
    const int have = *s.count;
    uint32_t* okd = a.ws_kd + ((size_t)(q0 + q) * a.nsplit + split) * a.k;
    long long* oki = a.ws_kid + ((size_t)(q0 + q) * a.nsplit + split) * a.k;
    for (int j = threadIdx.x; j < a.k; j += blockDim.x) {
      okd[j] = j < have ? s.kd[j] : KEY_SENTINEL_D;
      oki[j] = j < have ? s.kid[j] : KEY_SENTINEL_ID;
    }
  }
}

// out[i * nr + j] = Hamming distance of left row i and right row j (padded rows)
__global__ void hamming_pair_kernel(const uint4* __restrict__ a, long long nl, const uint4* __restrict__ b, long long nr, int W,
                                    float* __restrict__ out) {
  const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= nl * nr) return;
  const uint4* x = a + (size_t)(p / nr) * W;
  const uint4* y = b + (size_t)(p % nr) * W;
  uint32_t d = 0;
  for (int w = 0; w < W; ++w) d += popc4(__ldg(x + w), __ldg(y + w));
  out[p] = (float)d;
}

// faiss binary_to_real: bit b of a row -> +1.f / -1.f, LSB first within each byte
__global__ void binary_to_real_kernel(const uint8_t* __restrict__ x, long long n, int dim, int stride, float* __restrict__ out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n * dim) return;
  const long long r = i / dim;
  const int b = (int)(i - r * dim);
  out[i] = (x[(size_t)r * stride + (b >> 3)] >> (b & 7)) & 1 ? 1.0f : -1.0f;
}

// faiss real_to_binary: component > 0 -> bit 1; one thread per output byte of a padded row (padding bytes -> 0)
__global__ void real_to_binary_kernel(const float* __restrict__ x, long long n, int dim, int stride, uint8_t* __restrict__ out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n * stride) return;
  const long long r = i / stride;
  const int byte = (int)(i - r * stride);
  uint8_t v = 0;
  if (byte < dim / 8)
    for (int j = 0; j < 8; ++j) v |= (x[(size_t)r * dim + byte * 8 + j] > 0.f ? 1 : 0) << j;
  out[i] = v;
}

// rows[slots[i]] = src[i], ids[slots[i]] = src_ids[i]
__global__ void scatter_bin_rows_kernel(const uint4* __restrict__ src, const long long* __restrict__ src_ids,
                                        const long long* __restrict__ slots, long long n, int W, uint4* rows, long long* ids) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n * W) return;
  const long long i = t / W;
  const int w = (int)(t - i * W);
  const long long s = slots[i];
  rows[(size_t)s * W + w] = src[t];
  if (w == 0) ids[s] = src_ids[i];
}

// dst[dst_rows[i]] = src[src_rows[i]] for rows and ids (list relocation / compaction)
__global__ void move_bin_rows_kernel(const uint4* __restrict__ srows, const long long* __restrict__ sids, const long long* __restrict__ src_rows,
                                     const long long* __restrict__ dst_rows, long long n, int W, uint4* drows, long long* dids) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n * W) return;
  const long long i = t / W;
  const int w = (int)(t - i * W);
  const long long sr = src_rows[i], dr = dst_rows[i];
  drows[(size_t)dr * W + w] = srows[(size_t)sr * W + w];
  if (w == 0) dids[dr] = sids[sr];
}

struct BinJob {
  const uint4* rows = nullptr;
  const long long* ids = nullptr;
  int W = 0;
  int mode = 0;
  long long n = 0;
  const long long* probes = nullptr;
  int nprobe = 0;
  const long long* list_off = nullptr;
  const int* list_len = nullptr;
  double avg_candidates = 0;  // mode 1: expected candidates per query (sizing of nsplit)
  const SearchCtx* sc = nullptr;
  bool has_thr = false;
  int radius = 0;             // range search: distance < radius
};

constexpr size_t kMaxDynSmem = 227 * 1024;
constexpr size_t kTileSmemBudget = 100 * 1024;  // larger query tiles only while a few CTAs still fit on one SM

size_t bin_smem_bytes(int qt, int W, int nseg, int cap) {
  return (size_t)qt * W * 16 + ((size_t)(nseg + 1) * 4 + 15) / 16 * 16 + (size_t)qt * BlockSelect::smem_bytes(cap);
}

template <int QT>
void launch_hamming_scan(const BinScanArgs& a, dim3 grid, size_t smem, cudaStream_t s) {
  if (smem > kMaxDynSmem) fail(B200VS_EILLEGAL_PARAMETERS, "request needs more shared memory than one SM has (topk/nprobe/dimension too large)");
  B200VS_CUDA(cudaFuncSetAttribute(hamming_scan_kernel<QT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxDynSmem));
  hamming_scan_kernel<QT><<<grid, BIN_THREADS, smem, s>>>(a);
}

// scan + select + merge: out_dist [nq, k] (float distances, 0 padded), out_ids [nq, k] (-1 padded), out_counts [nq] (nullable)
void hamming_search(IndexBase* ix, const BinJob& job, int64_t nq, const uint4* q, int k, float* out_dist, long long* out_ids,
                    int* out_counts, cudaStream_t s) {
  if (nq <= 0 || k <= 0) return;
  const int cap = select_pool_cap(k, BIN_THREADS);
  const int nseg = job.mode == 0 ? 1 : job.nprobe;
  int qt = 1;  // query tile: the IVF list scan serves one query per CTA (each query probes its own lists)
  if (job.mode == 0)
    for (int t : {8, 4, 2})
      if (t / 2 < nq && bin_smem_bytes(t, job.W, nseg, cap) <= kTileSmemBudget) { qt = t; break; }
  const int64_t tiles = cdiv(nq, qt);
  if (tiles > 65535) fail(B200VS_EILLEGAL_PARAMETERS, "batch too large for one call");
  // split each query tile's candidates over several CTAs while the batch alone cannot fill the 148 SMs (batch 1 included)
  const double cand = job.mode == 0 ? (double)job.n : job.avg_candidates;
  int64_t nsplit = std::max<int64_t>(1, cdiv(148 * 4, tiles));
  nsplit = std::min<int64_t>(nsplit, std::max<int64_t>(1, (int64_t)(cand / 1024.0)));
  nsplit = std::min<int64_t>(nsplit, std::max<int64_t>(1, 65536 / k));  // merge work per query
  BinScanArgs a;
  a.rows = job.rows; a.ids = job.ids; a.queries = q; a.W = job.W; a.mode = job.mode; a.n = job.n;
  a.probes = job.probes; a.nprobe = job.nprobe; a.list_off = job.list_off; a.list_len = job.list_len;
  a.nq = nq; a.k = k; a.nsplit = (int)nsplit; a.pool_cap = cap;
  a.ws_kd = ix->scratch.alloc<uint32_t>((size_t)nq * nsplit * k);
  a.ws_kid = ix->scratch.alloc<long long>((size_t)nq * nsplit * k);
  const SearchCtx* sc = job.sc;
  a.filt.has_range = sc ? sc->has_range : 0;
  a.filt.negate = sc ? sc->negate : 0;
  a.filt.rmin = sc ? sc->rmin : 0;
  a.filt.rmax = sc ? sc->rmax : 0;
  a.filt.sorted_ids = sc ? sc->sorted_ids_dev : nullptr;
  a.filt.n_ids = sc ? sc->n_ids : 0;
  a.has_thr = job.has_thr ? 1 : 0;
  a.thr_key = job.has_thr ? f2ord((float)job.radius) : 0;
  const dim3 grid((unsigned)nsplit, (unsigned)tiles);
  const size_t smem = bin_smem_bytes(qt, job.W, nseg, cap);
  switch (qt) {
    case 8: launch_hamming_scan<8>(a, grid, smem, s); break;
    case 4: launch_hamming_scan<4>(a, grid, smem, s); break;
    case 2: launch_hamming_scan<2>(a, grid, smem, s); break;
    default: launch_hamming_scan<1>(a, grid, smem, s); break;
  }
  const size_t smem2 = BlockSelect::smem_bytes(cap);
  if (smem2 > kMaxDynSmem) fail(B200VS_EILLEGAL_PARAMETERS, "topk too large");
  B200VS_CUDA(cudaFuncSetAttribute(merge_select_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxDynSmem));
  merge_select_kernel<true><<<(unsigned)nq, SCAN_THREADS, smem2, s>>>(a.ws_kd, a.ws_kid, (int)nsplit, k, cap, out_dist, nullptr,
                                                                       out_ids, out_counts, nullptr, nullptr);
  B200VS_CUDA(cudaGetLastError());
  ix->launch_count(2);
}

}  // namespace

// ============================================================================================
// BinaryIndex: BINARY_FLAT is the one-list case of BINARY_IVF_FLAT (no centroids, always trained)
// ============================================================================================
struct BinaryIndex : IndexBase {
  const bool ivf;
  const int W;     // 16-byte words per stored row
  const int code;  // dim / 8 bytes per row as given
  int nlist;       // may degenerate to 1 at train time (vector_index_ivf_flat.cc:610-615)
  bool trained;
  DevBuf<uint4> cents;          // [nlist, W]
  DevBuf<long long> cent_ids;   // iota
  DevBuf<uint4> rows;           // arena [arena_cap, W]
  DevBuf<long long> ids;        // arena
  IvfLists L;

  BinaryIndex(b200vs_type t, int d, const b200vs_params& p)
      : IndexBase(t, B200VS_HAMMING, d, p), ivf(t == B200VS_BINARY_IVF_FLAT), W(bin_words(d)), code(d / 8) {
    nlist = ivf ? (p.nlist > 0 ? p.nlist : 2048) : 1;  // Constant::kCreateBinaryIvfFlatParamNcentroids (constant.h:180)
    trained = !ivf;
    if (!ivf) L.init(1, stream);
  }
  bool is_trained() const override { return trained; }
  int export_nlist() const override { return nlist; }

  // ---- the float entry points do not apply (the ABI rejects them before they get here) ----
  void train(int64_t, const float*) override { fail(B200VS_EVECTOR_INVALID, "float vectors given to a binary index"); }
  void add(int64_t, const float*, const int64_t*, bool) override { fail(B200VS_EVECTOR_INVALID, "float vectors given to a binary index"); }
  void search_dev(int64_t, const float*, int, const SearchCtx&, float*, long long*, cudaStream_t) override {
    fail(B200VS_EVECTOR_INVALID, "float vectors given to a binary index");
  }
  void range_search_dev(int64_t, const float*, float, int, const SearchCtx&, float*, long long*, int*, cudaStream_t) override {
    fail(B200VS_EVECTOR_INVALID, "float vectors given to a binary index");
  }

  // packed rows [n, code] (host or device) -> zero-padded [n, W] words in scratch
  uint4* stage_rows(int64_t n, const uint8_t* x, cudaMemcpyKind kind, cudaStream_t s) {
    uint4* d = scratch.alloc<uint4>((size_t)n * W);
    if ((size_t)W * 16 != (size_t)code) B200VS_CUDA(cudaMemsetAsync(d, 0, (size_t)n * W * 16, s));
    B200VS_CUDA(cudaMemcpy2DAsync(d, (size_t)W * 16, x, (size_t)code, (size_t)code, (size_t)n, kind, s));
    return d;
  }

  void install_centroids(const uint4* dev_c, int k) {  // dev_c: padded rows on the device (copied)
    nlist = k;
    cents.free(); cent_ids.free();
    cents.reserve((size_t)k * W, 0, stream);
    cent_ids.reserve(k, 0, stream);
    B200VS_CUDA(cudaMemcpyAsync(cents.p, dev_c, (size_t)k * W * 16, cudaMemcpyDeviceToDevice, stream));
    launch_iota(cent_ids.p, k, stream);
    B200VS_CUDA(cudaStreamSynchronize(stream));
    L.init(k, stream);
    rows.free(); ids.free();
    trained = true;
  }

  // trained-state blob: int64 hdr[4] = {magic 'BIVF', nlist, dim, metric}; uint8 centroids[nlist * dim / 8]
  static constexpr int64_t kMagic = 0x46564942;
  void set_state(const void* blob, size_t len) override {
    if (!ivf) fail(B200VS_EVECTOR_NOT_SUPPORT, "no trained state for this index type");
    std::unique_lock<std::shared_mutex> wl(rw);
    std::lock_guard<std::mutex> gl(gpu_mu);
    set_device();
    quiesce();
    if (len < 32) fail(B200VS_EILLEGAL_PARAMETERS, "state blob too short");
    const int64_t* hdr = (const int64_t*)blob;
    if (hdr[0] != kMagic || hdr[2] != dim || hdr[3] != B200VS_HAMMING) fail(B200VS_EILLEGAL_PARAMETERS, "bad binary IVF state blob");
    const int64_t k = hdr[1];
    if (k <= 0 || k > (1 << 24) || len < 32 + (size_t)k * code) fail(B200VS_EILLEGAL_PARAMETERS, "state blob truncated");
    scratch.reset(stream);
    install_centroids(stage_rows(k, (const uint8_t*)blob + 32, cudaMemcpyHostToDevice, stream), (int)k);
  }
  int64_t get_state(void* blob, size_t cap) override {
    RwSharedGuard rl(this);
    if (!ivf || !trained) return 0;
    const size_t need = 32 + (size_t)nlist * code;
    if (!blob || cap < need) return (int64_t)need;
    set_device();
    const int64_t hdr[4] = {kMagic, nlist, dim, (int64_t)metric};
    memcpy(blob, hdr, 32);
    B200VS_CUDA(cudaMemcpy2D((char*)blob + 32, code, cents.p, (size_t)W * 16, code, nlist, cudaMemcpyDeviceToHost));
    return (int64_t)need;
  }

  // faiss IndexBinaryIVF::train: binary_to_real -> float L2 k-means (the float IVF settings: niter 10, <= 256 points per
  // centroid, seed 1234, index.cu IvfFlatIndex::train) -> real_to_binary
  void train_binary(int64_t n, const uint8_t* x) override {
    if (n <= 0) fail(B200VS_EILLEGAL_PARAMETERS, "data size invalid");
    if (!ivf) return;
    std::unique_lock<std::shared_mutex> wl(rw);
    std::lock_guard<std::mutex> gl(gpu_mu);
    if (trained) return;  // ivf_flat.cc:578-640
    set_device();
    quiesce();
    scratch.reset(stream);
    const int k = n < nlist ? 1 : nlist;  // "data size too small, nlist degenerate to 1", ivf_flat.cc:610-615
    // kmeans_gpu's training subsample, taken on the packed rows so only the sample is expanded to floats
    std::vector<uint8_t> sub;
    const uint8_t* xs = x;
    int64_t m = n;
    if (n > (int64_t)k * 256) {
      std::vector<int64_t> perm;
      kmeans_rand_perm(perm, n, 1234);
      m = (int64_t)k * 256;
      sub.resize((size_t)m * code);
      for (int64_t i = 0; i < m; ++i) memcpy(&sub[(size_t)i * code], x + (size_t)perm[i] * code, code);
      xs = sub.data();
    }
    // the expanded sample lives as floats on the host and the device (up to nlist * 256 rows * dim * 4 bytes)
    const double real_bytes = (double)m * dim * 4;
    if (real_bytes > kMaxTrainFloatBytes)
      fail(B200VS_EILLEGAL_PARAMETERS, "binary IVF training sample of " + std::to_string(m) + " rows x " + std::to_string(dim) +
                                           " bits needs " + std::to_string((int64_t)(real_bytes / (1 << 30))) +
                                           " GiB as floats (limit 16 GiB): use fewer centroids or a smaller dimension");
    std::vector<float> real((size_t)m * dim);
    {
      const auto mark = scratch.mark();
      uint4* d8 = stage_rows(m, xs, cudaMemcpyHostToDevice, stream);
      float* df = scratch.alloc<float>((size_t)m * dim);
      binary_to_real_kernel<<<(unsigned)cdiv(m * dim, 256), 256, 0, stream>>>((const uint8_t*)d8, m, dim, W * 16, df);
      B200VS_CUDA(cudaGetLastError());
      B200VS_CUDA(cudaMemcpyAsync(real.data(), df, real.size() * 4, cudaMemcpyDeviceToHost, stream));
      B200VS_CUDA(cudaStreamSynchronize(stream));
      scratch.release(mark);
    }
    std::vector<float> cent;
    kmeans_gpu(this, B200VS_L2, dim, m, real.data(), k, 10, 256, 1234, cent, [&](const float* xd, int64_t mm, const float* cd, int kk, long long* out) {
      ScanJob j;  // exact FP32 L2 assignment, the float IVF's reference-order scan
      j.l2 = true; j.vecs = cd; j.ids = cent_ids.p; j.d = dim; j.mode = 0; j.n = kk;
      const int64_t chunk = std::max<int64_t>(1024, std::min<int64_t>(32768, (1LL << 28) / std::max(1, kk)));
      for (int64_t a = 0; a < mm; a += chunk) {
        const auto mark = scratch.mark();
        run_scan(this, j, std::min(chunk, mm - a), xd + (size_t)a * dim, 1, nullptr, nullptr, out + a, nullptr, stream);
        scratch.release(mark);
      }
    }, [&](int kk) { cent_ids.free(); cent_ids.reserve(kk, 0, stream); launch_iota(cent_ids.p, kk, stream); });
    float* dc = scratch.alloc<float>((size_t)k * dim);
    uint8_t* db = scratch.alloc<uint8_t>((size_t)k * W * 16);
    B200VS_CUDA(cudaMemcpyAsync(dc, cent.data(), (size_t)k * dim * 4, cudaMemcpyHostToDevice, stream));
    real_to_binary_kernel<<<(unsigned)cdiv((int64_t)k * W * 16, 256), 256, 0, stream>>>(dc, k, dim, W * 16, db);
    B200VS_CUDA(cudaGetLastError());
    install_centroids((const uint4*)db, k);
  }

  BinJob centroid_job() const {
    BinJob j;
    j.rows = cents.p; j.ids = cent_ids.p; j.W = W; j.mode = 0; j.n = nlist;
    return j;
  }
  BinJob flat_job(const SearchCtx* sc) const {  // the single list of a Flat index
    BinJob j;
    const ListMeta& m = L.lists[0];
    j.rows = rows.p + (size_t)m.off * W; j.ids = ids.p + m.off; j.W = W; j.mode = 0; j.n = m.len; j.sc = sc;
    return j;
  }
  BinJob list_job(const SearchCtx* sc, const long long* probes, int nprobe) const {
    BinJob j;
    j.rows = rows.p; j.ids = ids.p; j.W = W; j.mode = 1; j.probes = probes; j.nprobe = nprobe;
    j.list_off = L.d_off.p; j.list_len = L.d_len.p; j.sc = sc;
    j.avg_candidates = nlist > 0 ? (double)L.total_len() * nprobe / nlist : 0;
    return j;
  }
  int resolve_nprobe(const SearchCtx& sc) const {
    const int np = sc.nprobe > 0 ? sc.nprobe : 80;  // Constant::kSearchBinaryIvfFlatParamNprobe (constant.h:181)
    return std::min(np, nlist);
  }
  // coarse quantiser: Flat search over the centroids, k = nprobe -> (distance, list id) order
  long long* coarse(int64_t nq, const uint4* q, int nprobe, cudaStream_t s, long long* out = nullptr) {
    long long* probes = out ? out : scratch.alloc<long long>((size_t)nq * nprobe);
    hamming_search(this, centroid_job(), nq, q, nprobe, nullptr, probes, nullptr, s);
    return probes;
  }

  // Flat (flat.cc:121-162): duplicate ids in a batch are rejected and pre-existing ids are always replaced.
  // IVF (ivf_flat.cc:92-160): untrained -> EVECTOR_NOT_TRAIN; only upsert removes pre-existing ids.
  void add_binary(int64_t n, const uint8_t* x, const int64_t* in_ids, bool upsert) override {
    if (!ivf) check_batch_ids_unique(n, in_ids);
    std::unique_lock<std::shared_mutex> wl(rw);
    if (!trained) fail(B200VS_EVECTOR_NOT_TRAIN, "not train");
    std::lock_guard<std::mutex> gl(gpu_mu);
    set_device();
    quiesce();
    scratch.reset(stream);
    if (!ivf || upsert) remove_locked(n, in_ids);
    uint4* st = stage_rows(n, x, cudaMemcpyHostToDevice, stream);
    long long* st_ids = scratch.alloc<long long>(n);
    long long* st_slots = scratch.alloc<long long>(n);
    B200VS_CUDA(cudaMemcpyAsync(st_ids, in_ids, (size_t)n * 8, cudaMemcpyHostToDevice, stream));
    std::vector<long long> h_list(n, 0), slots(n);
    if (ivf) {  // nearest list by (distance, list id)
      long long* dl = scratch.alloc<long long>(n);
      for (int64_t a = 0; a < n; a += 32768) {
        const int64_t m = std::min<int64_t>(32768, n - a);
        const auto mark = scratch.mark();
        coarse(m, st + (size_t)a * W, 1, stream, dl + a);
        scratch.release(mark);
      }
      B200VS_CUDA(cudaMemcpyAsync(h_list.data(), dl, (size_t)n * 8, cudaMemcpyDeviceToHost, stream));
      B200VS_CUDA(cudaStreamSynchronize(stream));
    }
    std::vector<int> need(nlist, 0);
    for (int64_t i = 0; i < n; ++i) {
      if (h_list[i] < 0 || h_list[i] >= nlist) fail(B200VS_EINTERNAL, "list id out of range");
      need[h_list[i]]++;
    }
    L.reserve_for(need, [&](int64_t arena_rows) {
      rows.reserve((size_t)arena_rows * W, (size_t)L.arena_used_before * W, stream);
      ids.reserve((size_t)arena_rows, (size_t)L.arena_used_before, stream);
    }, [&](int64_t src, int64_t dst, int64_t len) {
      B200VS_CUDA(cudaMemcpyAsync(rows.p + (size_t)dst * W, rows.p + (size_t)src * W, (size_t)len * W * 16, cudaMemcpyDeviceToDevice, stream));
      B200VS_CUDA(cudaMemcpyAsync(ids.p + dst, ids.p + src, (size_t)len * 8, cudaMemcpyDeviceToDevice, stream));
    });
    for (int64_t i = 0; i < n; ++i) slots[i] = L.append((int)h_list[i], in_ids[i]);
    B200VS_CUDA(cudaMemcpyAsync(st_slots, slots.data(), (size_t)n * 8, cudaMemcpyHostToDevice, stream));
    scatter_bin_rows_kernel<<<(unsigned)cdiv(n * W, 256), 256, 0, stream>>>(st, st_ids, st_slots, n, W, rows.p, ids.p);
    B200VS_CUDA(cudaGetLastError());
    L.upload(stream);
    maybe_compact();
  }

  int64_t remove_locked(int64_t n, const int64_t* del) {
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

  void maybe_compact() {
    if (!L.needs_compaction()) return;
    std::vector<long long> src, dst;
    const int64_t new_rows = std::max<int64_t>(L.plan_compaction(src, dst), 1);
    DevBuf<uint4> nr; DevBuf<long long> ni;
    nr.reserve((size_t)new_rows * W, 0, stream);
    ni.reserve(new_rows, 0, stream);
    const int64_t m = (int64_t)src.size();
    if (m) {
      long long* d_src = scratch.alloc<long long>(m);
      long long* d_dst = scratch.alloc<long long>(m);
      B200VS_CUDA(cudaMemcpyAsync(d_src, src.data(), m * 8, cudaMemcpyHostToDevice, stream));
      B200VS_CUDA(cudaMemcpyAsync(d_dst, dst.data(), m * 8, cudaMemcpyHostToDevice, stream));
      move_bin_rows_kernel<<<(unsigned)cdiv(m * W, 256), 256, 0, stream>>>(rows.p, ids.p, d_src, d_dst, m, W, nr.p, ni.p);
      B200VS_CUDA(cudaGetLastError());
    }
    B200VS_CUDA(cudaStreamSynchronize(stream));
    std::swap(rows.p, nr.p); std::swap(rows.cap, nr.cap);
    std::swap(ids.p, ni.p); std::swap(ids.cap, ni.cap);
    L.commit_compaction();
    L.upload(stream);
  }

  // Flat: unknown ids are ignored (flat.cc:171-203).  IVF: untrained -> OK (-1), nothing removed -> EVECTOR_INVALID (ABI).
  int64_t remove(int64_t n, const int64_t* del) override {
    std::unique_lock<std::shared_mutex> wl(rw);
    if (!trained) return -1;
    std::lock_guard<std::mutex> gl(gpu_mu);
    set_device();
    quiesce();
    scratch.reset(stream);
    const int64_t r = remove_locked(n, del);
    maybe_compact();
    return r;
  }

  void search_binary_dev(int64_t nq, const uint8_t* xq, int k, const SearchCtx& sc, float* od, long long* oi, cudaStream_t s) override {
    if (!trained) { fill_empty_results(nq, k, od, oi, s); return; }  // ivf_flat.cc:224-227
    const uint4* q = stage_rows(nq, xq, cudaMemcpyDeviceToDevice, s);
    if (!ivf) { hamming_search(this, flat_job(&sc), nq, q, k, od, oi, nullptr, s); return; }
    const int nprobe = resolve_nprobe(sc);
    long long* probes = coarse(nq, q, nprobe, s);
    if (profiling) profile_probed(this, probes, nq * nprobe, nlist, L.d_len.p, s);
    hamming_search(this, list_job(&sc, probes, nprobe), nq, q, k, od, oi, nullptr, s);
  }

  // faiss binary range_search takes an int radius: the API's float radius is truncated, hits are distance < radius
  // (flat.cc:282-311, ivf_flat.cc:342-345)
  void range_search_binary_dev(int64_t nq, const uint8_t* xq, float radius, int max_results, const SearchCtx& sc, float* od,
                               long long* oi, int* oc, cudaStream_t s) override {
    if (!trained) {
      fill_empty_results(nq, max_results, od, oi, s);
      if (oc) B200VS_CUDA(cudaMemsetAsync(oc, 0, (size_t)nq * 4, s));
      return;
    }
    const uint4* q = stage_rows(nq, xq, cudaMemcpyDeviceToDevice, s);
    BinJob j;
    if (!ivf) {
      j = flat_job(&sc);
    } else {
      const int nprobe = resolve_nprobe(sc);
      j = list_job(&sc, coarse(nq, q, nprobe, s), nprobe);
    }
    j.has_thr = true;
    j.radius = (int)std::max(-1.0f, std::min(radius, (float)(kMaxBinaryDim + 1)));
    hamming_search(this, j, nq, q, max_results, od, oi, oc, s);
  }

  int64_t count() const override { return L.live; }
  int64_t deleted_count() const override { return L.dead; }
  int64_t memory_size() const override { return (int64_t)(rows.cap * 16 + ids.cap * 8 + cents.cap * 16); }

  // rows go out through `codes` [count, dim / 8]; `vectors` does not apply
  void export_lists(int64_t* list_off, float*, uint8_t* codes, int64_t* out_ids) override {
    RwSharedGuard rl(this);
    std::lock_guard<std::mutex> gl(gpu_mu);
    set_device();
    quiesce();
    std::vector<uint8_t> buf;
    int64_t o = 0;
    for (int l = 0; l < nlist; ++l) {
      if (list_off) list_off[l] = o;
      if (!trained) continue;
      const ListMeta& m = L.lists[l];
      if (m.len == 0) continue;
      if (codes) {
        buf.resize((size_t)m.len * code);
        B200VS_CUDA(cudaMemcpy2D(buf.data(), code, rows.p + (size_t)m.off * W, (size_t)W * 16, code, m.len, cudaMemcpyDeviceToHost));
      }
      for (int p = 0; p < m.len; ++p) {
        const int64_t id = L.h_ids[m.off + p];
        if (id < 0) continue;
        if (out_ids) out_ids[o] = id;
        if (codes) memcpy(codes + (size_t)o * code, buf.data() + (size_t)p * code, code);
        ++o;
      }
    }
    if (list_off) list_off[nlist] = o;
  }
  int64_t export_list(int list, int64_t cap, float* vectors, int64_t* out_ids) override {
    if (vectors) fail(B200VS_EILLEGAL_PARAMETERS, "binary rows are exported through b200vs_export_lists (codes)");
    RwSharedGuard rl(this);
    if (list < 0 || list >= nlist) fail(B200VS_EILLEGAL_PARAMETERS, "list id out of range");
    if (!trained) return 0;
    const ListMeta& m = L.lists[list];
    int64_t o = 0;
    for (int p = 0; p < m.len; ++p) {
      const int64_t id = L.h_ids[m.off + p];
      if (id < 0) continue;
      if (o < cap && out_ids) out_ids[o] = id;
      ++o;
    }
    return o;
  }
};

IndexBase* make_binary(b200vs_type t, int d, const b200vs_params& p) { return new BinaryIndex(t, d, p); }

void binary_pair_distance(int dim_bits, int64_t nl, const uint8_t* a, int64_t nr, const uint8_t* b, float* out, cudaStream_t s) {
  const int W = bin_words(dim_bits), code = dim_bits / 8;
  DevBuf<uint4> da, db;
  DevBuf<float> dout;
  da.reserve((size_t)nl * W, 0, s); db.reserve((size_t)nr * W, 0, s); dout.reserve((size_t)nl * nr, 0, s);
  if ((size_t)W * 16 != (size_t)code) {
    B200VS_CUDA(cudaMemsetAsync(da.p, 0, (size_t)nl * W * 16, s));
    B200VS_CUDA(cudaMemsetAsync(db.p, 0, (size_t)nr * W * 16, s));
  }
  B200VS_CUDA(cudaMemcpy2DAsync(da.p, (size_t)W * 16, a, code, code, nl, cudaMemcpyHostToDevice, s));
  B200VS_CUDA(cudaMemcpy2DAsync(db.p, (size_t)W * 16, b, code, code, nr, cudaMemcpyHostToDevice, s));
  hamming_pair_kernel<<<(unsigned)cdiv(nl * nr, 256), 256, 0, s>>>(da.p, nl, db.p, nr, W, dout.p);
  B200VS_CUDA(cudaGetLastError());
  B200VS_CUDA(cudaMemcpyAsync(out, dout.p, (size_t)nl * nr * 4, cudaMemcpyDeviceToHost, s));
  B200VS_CUDA(cudaStreamSynchronize(s));  // the device buffers die here
}

}  // namespace b200vs

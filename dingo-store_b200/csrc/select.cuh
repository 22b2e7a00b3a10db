// select.cuh — block-level streaming top-k over (key, id) pairs, smaller = better.
//
// Replaces the CPU heaps on the reference path (faiss HeapBlockResultHandler behind
// IndexFlat/IndexIVF::search, called at src/vector/vector_index_flat.cc:249-252 and
// vector_index_ivf_flat.cc:247-251; std::priority_queue at vector_index_hnsw.cc:433) and the 2-way
// merge of VectorIndexWrapper::MergeSearchResults (src/vector/vector_index.cc:1056-1108).
//
// Scheme: a shared-memory pool of `cap` (power of two) entries.  Producers append candidates that beat
// the current threshold (the k-th best seen so far); when the pool may overflow the block sorts it with an
// in-place bitonic network, keeps the best k and tightens the threshold.  Total order = (key, id), which
// is the engine's documented tie rule (DESIGN.md §Ties).  Works for any k <= 4096 (the RPC limit,
// src/server/index_service.cc:197-211).
#pragma once
#include "common.cuh"

namespace b200vs {

struct BlockSelect {
  uint32_t* kd;    // [cap]
  long long* kid;  // [cap]
  int* count;      // shared counter
  uint32_t* thr_d;
  long long* thr_id;
  int cap, k;

  // smem bytes needed for a pool of `cap` entries (+ header)
  __host__ __device__ static size_t smem_bytes(int cap) { return (size_t)cap * 12 + 32; }

  // view of a pool laid out at `smem` (no initialisation): lets a block keep several pools without holding their pointers
  __device__ __forceinline__ void attach(unsigned char* smem, int cap_, int k_) {
    cap = cap_; k = k_;
    kid = reinterpret_cast<long long*>(smem);
    kd = reinterpret_cast<uint32_t*>(smem + (size_t)cap * 8);
    unsigned char* hdr = smem + (size_t)cap * 12;
    thr_id = reinterpret_cast<long long*>(hdr);
    thr_d = reinterpret_cast<uint32_t*>(hdr + 8);
    count = reinterpret_cast<int*>(hdr + 12);
  }

  // carve from a 16-byte aligned shared buffer; all threads call
  __device__ void init(unsigned char* smem, int cap_, int k_) {
    attach(smem, cap_, k_);
    if (threadIdx.x == 0) { *count = 0; *thr_d = KEY_SENTINEL_D; *thr_id = KEY_SENTINEL_ID; }
    __syncthreads();
  }

  __device__ __forceinline__ bool passes(uint32_t d, long long id) const { return key_less(d, id, *thr_d, *thr_id); }

  // append without capacity check (caller guarantees room via maybe_prune)
  __device__ __forceinline__ void push(uint32_t d, long long id) {
    int p = atomicAdd(count, 1);
    kd[p] = d; kid[p] = id;
  }

  // in-place bitonic sort of the whole pool (ascending); all threads call
  __device__ void sort_pool() {
    const int n = *count;
    // only sort the smallest power of two covering n (the rest of the pool is never read)
    int m = 2;
    while (m < n) m <<= 1;
    __syncthreads();
    for (int i = n + threadIdx.x; i < m; i += blockDim.x) { kd[i] = KEY_SENTINEL_D; kid[i] = KEY_SENTINEL_ID; }
    __syncthreads();
    for (int size = 2; size <= m; size <<= 1) {
      for (int stride = size >> 1; stride > 0; stride >>= 1) {
        for (int i = threadIdx.x; i < (m >> 1); i += blockDim.x) {
          const int pos = 2 * i - (i & (stride - 1));
          const int j = pos + stride;
          const bool up = ((pos & size) == 0);
          const uint32_t ad = kd[pos], bd = kd[j];
          const long long ai = kid[pos], bi = kid[j];
          const bool lt = key_less(bd, bi, ad, ai);  // b < a
          const bool gt = key_less(ad, ai, bd, bi);  // a < b
          if (up ? lt : gt) { kd[pos] = bd; kd[j] = ad; kid[pos] = bi; kid[j] = ai; }
        }
        __syncthreads();
      }
    }
  }

  // sort, keep best k, tighten threshold; all threads call
  __device__ void prune() {
    __syncthreads();
    const int n = *count;
    sort_pool();
    if (threadIdx.x == 0) {
      *count = n < k ? n : k;
      if (n >= k) { *thr_d = kd[k - 1]; *thr_id = kid[k - 1]; }
    }
    __syncthreads();
  }

  // call at an iteration boundary (all threads): ensures room for `incoming` more pushes
  __device__ __forceinline__ void maybe_prune(int incoming) {
    __syncthreads();
    const int c = *count;
    __syncthreads();  // nobody pushes before every thread has read the same count
    if (c + incoming > cap) prune();
  }
};

inline int select_pool_cap(int k, int pushes_per_iter) {
  int need = k + pushes_per_iter;
  int c = next_pow2(need);
  if (c < 2 * k) c = next_pow2(2 * k);
  if (c < 512) c = 512;
  return c;
}

}  // namespace b200vs

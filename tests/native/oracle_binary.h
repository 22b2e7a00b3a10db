/*
 * oracle_binary.h — C ABI of the CPU oracle for the binary (Hamming) indexes (TEST INFRASTRUCTURE, NOT product code).
 *
 * Companion of oracle/oracle.h, built as its own library (liboracle_binary.so, linked against liboracle.so for the
 * float k-means) so the float oracle stays unchanged.  Restated from the reference's binary plugins:
 * VectorIndexFlat<faiss::IndexBinary> / VectorIndexIvfFlat<faiss::IndexBinary> (vector_index_factory.cc:73-80,
 * vector_index_flat.cc:63-71, :99-102, vector_index_ivf_flat.cc:62, :75-80) and VectorCalcDistance's HAMMING branch
 * (vector_index_utils.cc:146-149, :333-356, :640-648).
 *
 * Parity status: the faiss binary algorithms (IndexBinaryFlat / IndexBinaryIVF search, hamming_range_search,
 * IndexBinaryIVF::train) are NOT vendored; they are restated from the published algorithms — "parity unpinned".
 *
 * Rows are packed bits, dim / 8 bytes, bit b = bit (b % 8) of byte b / 8.  Results: ascending (distance, id); distances
 * are popcount(a ^ b) as float; missing hits padded with id -1, distance 0.  ids[i] < 0 marks a removed slot.
 */
#ifndef B200VS_ORACLE_BINARY_H_
#define B200VS_ORACLE_BINARY_H_

#include <stddef.h>
#include <stdint.h>

#include "../../oracle/oracle.h"

#ifdef __cplusplus
extern "C" {
#endif

/* popcount(a XOR b) over dim bits (vector_index_utils.cc:640-648) */
int32_t oracle_hamming(const uint8_t* a, const uint8_t* b, int32_t dim);

/* IndexBinaryIDMap2 search (flat.cc:205-264) */
int oracle_binary_flat_search(int32_t dim, int64_t n, const uint8_t* xb, const int64_t* ids, int64_t nq, const uint8_t* xq,
                              int32_t k, const oracle_filter* filt, int nthreads, float* out_dist, int64_t* out_ids);
/* faiss hamming_range_search: the API's float radius truncated to int, hits distance < radius (flat.cc:282-311); the closest
 * max_results hits per query are kept, out_counts[q] = how many */
int oracle_binary_flat_range_search(int32_t dim, int64_t n, const uint8_t* xb, const int64_t* ids, int64_t nq, const uint8_t* xq,
                                    float radius, int32_t max_results, const oracle_filter* filt, int nthreads, float* out_dist,
                                    int64_t* out_ids, int32_t* out_counts);

/* faiss binary_to_real (+1 / -1 per bit, LSB first) and real_to_binary (> 0 -> 1) */
void oracle_binary_to_real(int64_t n, int32_t dim, const uint8_t* x, float* out);
void oracle_real_to_binary(int64_t n, int32_t dim, const float* x, uint8_t* out);

/* IndexBinaryIVF::train: binary_to_real -> oracle_kmeans (L2) -> real_to_binary; centroids [k, dim / 8] */
int oracle_binary_kmeans(int32_t dim, int64_t n, const uint8_t* x, int32_t k, int32_t niter, int32_t max_points_per_centroid,
                         int64_t seed, int nthreads, uint8_t* centroids);
/* nearest centroid by (Hamming distance, list id) */
int oracle_binary_assign(int32_t dim, int64_t n, const uint8_t* x, int32_t nlist, const uint8_t* centroids, int nthreads,
                         int32_t* out_assign);

/* IndexBinaryIVF search (ivf_flat.cc:191-275): probes = the nprobe smallest (Hamming distance, list id) centroids; lists
 * given list-major, list l owns rows [list_off[l], list_off[l+1]) */
int oracle_binary_ivf_search(int32_t dim, int32_t nlist, const uint8_t* centroids, const int64_t* list_off, const uint8_t* xb,
                             const int64_t* ids, int64_t nq, const uint8_t* xq, int32_t k, int32_t nprobe, const oracle_filter* filt,
                             int nthreads, float* out_dist, int64_t* out_ids);
int oracle_binary_ivf_range_search(int32_t dim, int32_t nlist, const uint8_t* centroids, const int64_t* list_off, const uint8_t* xb,
                                   const int64_t* ids, int64_t nq, const uint8_t* xq, float radius, int32_t max_results,
                                   int32_t nprobe, const oracle_filter* filt, int nthreads, float* out_dist, int64_t* out_ids,
                                   int32_t* out_counts);

/* VectorCalcDistance, METRIC_TYPE_HAMMING: out[i * nr + j] = Hamming(left i, right j) */
int oracle_calc_distance_hamming(int32_t dim, int64_t nl, const uint8_t* left, int64_t nr, const uint8_t* right, float* out);

#ifdef __cplusplus
}
#endif
#endif

// Internal layout of the affine handle shared by the SIMT (tdnn.cu) and tcgen05 (tdnn_tc.cu) engines.
#pragma once

#include "common.cuh"

struct ktf_affine {
  ktf_affine_cfg cfg;
  float* d_w = nullptr;       // (U, K*D) fp32, Kaldi layout
  float* d_bias = nullptr;    // (U)
  float* d_scale = nullptr;   // (U) BatchNorm scale, or null
  float* d_offset = nullptr;  // (U) BatchNorm offset, or null
  void* tc = nullptr;         // engine-private state of the tcgen05 path
};

namespace ktf {
int affine_tc_prepare(ktf_affine* a, const float* weights_host, const float* bn_scale_host, const float* bn_offset_host);
void affine_tc_release(ktf_affine* a);
int affine_tc_forward(const ktf_affine* a, const float* x_dev, const int64_t* in_offsets_dev,
                      const int64_t* out_offsets_dev, int64_t batch, int64_t total_in_rows,
                      int64_t total_out_rows, float* y_dev, float* stats_dev, cudaStream_t st);
// per-utterance column sums / sums of squares of an fp32 (rows, dim) matrix -> (batch, 2, dim)
int stats_sums_f32(const float* y_dev, const int64_t* offsets_dev, int64_t batch, int dim, float* sums_dev,
                   cudaStream_t st);
// tcgen05 engine as a plain "NT" GEMM: C[i, j] = sum_k A[i, k] * B[j, k] + row_add[i] + col_add[j];
// A (m, K), B (n, K) row-major 16-bit (bf16, or fp16 when fp16 != 0), C fp32 or (c_bf16 != 0) bf16, row stride ldc
// elements.  With `row_best` (m zero-initialised 64-bit keys) nothing is stored (C may be null): every row keeps its best
// entry as a key -- order-preserving float bits << 32 | (0xffffffff - column), maximised atomically; the lowest column
// wins a tie.
int tc_gemm_nt(const void* A, long long m, long long lda, const void* B, long long n, long long ldb, long long K,
               int fp16, const float* row_add, const float* col_add, void* C, long long ldc, int c_bf16,
               cudaStream_t st, unsigned long long* row_best = nullptr);
// The same GEMM reduced to the k (1..32) largest entries of every row, nothing else stored: partial lists
// (num_lists, m, k) of fp32 values and columns, unordered, (-inf, -1) where a list has fewer than k entries; every column
// is in exactly one list.  num_lists = tc_topk_lists(m, n, K) (0 when m or n is 0).
int tc_topk_lists(long long m, long long n, long long K);
int tc_gemm_topk(const void* A, long long m, long long lda, const void* B, long long n, long long ldb, long long K,
                 int fp16, const float* row_add, const float* col_add, int k, float* part_score, long long* part_index,
                 cudaStream_t st);
}  // namespace ktf

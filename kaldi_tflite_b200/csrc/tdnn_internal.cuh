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
// One score GEMM on the tcgen05 engine: C[i, j] = sum_k A[i, k] * B[j, k] + row_add[i] + col_add[j] (the score s),
// A (m, K) and B (n, K) row-major 16-bit (bf16, or fp16 when fp16 != 0), K and both leading dimensions multiples of 8.
struct TcScore {
  const void* A;
  long long m, lda;
  const void* B;
  long long n, ldb;
  long long K;
  int fp16;
  const float* row_add;
  const float* col_add;
  // Optional AS-norm part (PLDA): with s = (acc + col_add[j]) + A_i, the value is
  // (s - col_mean[j]) * col_half_inv[j] + (s - mu_t) * h_t, where row_add then holds one float4 (A_i, h_t, mu_t, unused)
  // per row and the h are 0.5 / sigma.  Absent when col_half_inv is null.
  const float* col_half_inv;
  const float* col_mean;
  // Exactly one output:
  // - rows: C fp32 or (c_bf16 != 0) the fp32 value rounded once to bf16, row stride ldc elements;
  // - row_best (raw value only; m zero-initialised 64-bit keys, C may be null): every row keeps its best entry as a key
  //   -- order-preserving float bits << 32 | (0xffffffff - column), maximised atomically; the lowest column wins a tie;
  // - top-k (part_score non-null, 1 <= k <= 32): the k largest values of every row as partial lists (num_lists, m, k)
  //   of fp32 values and columns, unordered, (-inf, -1) where a list has fewer than k entries; every column is in
  //   exactly one list, num_lists = tc_topk_lists(m, n, K) (0 when m or n is 0).  AS-norm NaN and -inf values are
  //   never listed.
  // Every value is bit-equal whichever output carries it.
  void* C;
  long long ldc;
  int c_bf16;
  unsigned long long* row_best;
  int k;
  float* part_score;
  long long* part_index;
  // - within-group rows (raw value, value (acc + row_add[i]) + col_add[j]; non-null `within`, m == n, C fp32): only the
  //   tiles of TcWithin::tiles are computed, and entry (i, j) is stored, at C[rows[i].dst + j], only when
  //   rows[i].lo <= j < rows[i].hi.
  const struct TcWithin* within;
};
// Row i of a within-group score: its group is columns [lo, hi), and its entries go to dst + column.
struct WithinRow {
  long long dst;
  int lo, hi;
};
struct TcWithin {
  const int2* tiles;         // (row block of 256 rows, n-tile of 256 columns), from tc_within_tiles
  long long num_tiles;
  const WithinRow* rows;     // (m)
};
int tc_gemm_score(const TcScore& s, cudaStream_t st);
int tc_topk_lists(long long m, long long n, long long K);
// The tiles a within-group score computes for groups [offsets[g], offsets[g + 1]) of the rows (relative to offsets[0]):
// every 256-row block with the n-tiles that cover the groups its rows belong to.  Returns their number and writes them
// to `tiles` when it is not null.
long long tc_within_tiles(const int64_t* offsets, int num_groups, int2* tiles);
}  // namespace ktf

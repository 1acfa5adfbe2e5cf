// PLDA transform + all-pairs log-likelihood-ratio scoring.
//
// Replaces layers/plda/plda.py:163-263 (under /root/reference/kaldi_tflite/lib/).
// The reference materialises a (B, dim, B) broadcast tensor; here the score is evaluated in
// its algebraically identical GEMM form (SURVEY.md 8a row a13):
//     score[i, j] = A_i + B_j + sum_d u_i[d] * c[d] * u_j[d]
//     r = psi/(psi+1), v1 = 1 + r, v0 = 1 + psi, c = r / v1
//     A_i = sum_d u_i[d]^2 * (0.5/v0 - 0.5/v1) - 0.5 * (sum log v1 - sum log v0)
//     B_j = -0.5 * sum_d (r u_j[d])^2 / v1
// Arithmetic is fp32 or fp64 (the reference's default parameter dtype) per handle.
//
// fp32 handles run the cross term on the tcgen05 engine (tdnn_tc.cu) at fp32-equivalent precision:
// both operands are split into fp16 hi + lo parts (22 significant bits) and the three significant
// partial products are evaluated as ONE GEMM over a tripled K:
//     [a_hi | a_lo | a_hi] . [b_hi | b_hi | b_lo]^T = a_hi b_hi + a_lo b_hi + a_hi b_lo      (fp32 accumulate)
// with A_i / B_j added in the epilogue.  At dim 128 the kernel is bound by the fp32 score writes
// (64 FLOP per output byte), not by the tensor pipe (SURVEY.md 8d cfg5).  fp64 handles and
// configurations whose operands could leave the fp16 range use exact SIMT tiles.
#include <cuda_fp16.h>
#include <math.h>

#include <algorithm>
#include <vector>

#include "common.cuh"
#include "gemm_simt.cuh"
#include "tdnn_internal.cuh"

struct ktf_plda {
  int dim = 0;
  int normalize_length = 1;
  int simple_length_norm = 0;
  int dtype_bytes = 4;
  double num_examples = 1.0; // utterances averaged into an enrolled vector (plda.py:163-182, 215-231)
  void* d_T = nullptr;       // (dim, dim)
  void* d_offset = nullptr;  // (dim)  -T m
  void* d_psi = nullptr;     // (dim)
  void* d_c = nullptr;       // (dim)  r / v1
  void* d_wa = nullptr;      // (dim)  0.5/v0 - 0.5/v1
  void* d_wb = nullptr;      // (dim)  -0.5 r^2 / v1
  double logdet_term = 0.0;  // -0.5 (sum log v1 - sum log v0)
  int use_tc = 0;            // fp32 handle on an sm_100 device with fp16-safe operand range
  mutable ktf::Workspace ws; // split operands + A_i / B_j of the tensor-core path (grow-only)
};

namespace {

template <typename T>
struct CastLoad {  // float input rows promoted to the PLDA dtype
  const float* p;
  long long ld;
  __device__ __forceinline__ T operator()(long long r, int k) const { return (T)p[r * ld + k]; }
};

template <typename T>
struct OffsetEpi {
  T* u;
  const T* offset;
  int dim;
  __device__ __forceinline__ void operator()(long long row, long long col, T acc) const {
    u[row * dim + col] = acc + offset[col];
  }
};

template <typename T>
struct ScaledLoad {
  const T* p;
  const T* c;
  long long ld;
  __device__ __forceinline__ T operator()(long long r, int k) const { return p[r * ld + k] * c[k]; }
};

template <typename T>
struct ScoreEpi {
  T* s;
  const T* A;
  const T* B;
  long long ld;
  __device__ __forceinline__ void operator()(long long row, long long col, T acc) const {
    s[row * ld + col] = acc + A[row] + B[col];
  }
};

template <typename T>
__device__ __forceinline__ T warp_sum(T v) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// One warp per vector: length normalisation (plda.py:163-196).
template <typename T>
__global__ void plda_norm_kernel(T* __restrict__ u, long long n, int dim, const T* __restrict__ psi,
                                 int simple, T inv_examples) {
  const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= n) return;
  const int lane = threadIdx.x & 31;
  T* p = u + row * dim;
  T acc = T(0);
  for (int d = lane; d < dim; d += 32) {
    const T v = p[d];
    acc += simple ? v * v : v * v / (psi[d] + inv_examples);
  }
  acc = warp_sum(acc);
  const T nf = simple ? sqrt((T)dim) / sqrt(acc) : sqrt((T)dim / acc);
  for (int d = lane; d < dim; d += 32) p[d] *= nf;
}

// One warp per vector: out[row] = sum_d w[d] * u[d]^2 + add
template <typename T>
__global__ void plda_quad_kernel(const T* __restrict__ u, long long n, int dim, const T* __restrict__ w,
                                 T add, T* __restrict__ out) {
  const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= n) return;
  const int lane = threadIdx.x & 31;
  const T* p = u + row * dim;
  T acc = T(0);
  for (int d = lane; d < dim; d += 32) acc += w[d] * p[d] * p[d];
  acc = warp_sum(acc);
  if (lane == 0) out[row] = acc + add;
}

// fp32 rows (optionally scaled per column) -> fp16 hi/lo split rows of 3*dim columns:
//   layout 0 (test side):   [hi | lo | hi]      layout 1 (enrolled side): [hi | hi | lo]
__global__ void plda_split_kernel(const float* __restrict__ u, long long n, int dim, const float* __restrict__ c,
                                  int layout, __half* __restrict__ out) {
  const long long total = n * dim;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / dim;
    const int d = (int)(i - r * dim);
    float v = u[i];
    if (c) v *= c[d];
    const __half hi = __float2half_rn(v);
    const __half lo = __float2half_rn(v - __half2float(hi));
    __half* o = out + r * (3LL * dim);
    o[d] = hi;
    o[dim + d] = layout == 0 ? lo : hi;
    o[2 * dim + d] = layout == 0 ? hi : lo;
  }
}

// Decodes the best-entry keys of tc_gemm_nt(row_best): score and column of every test row (-1: no enrolled vector).
__global__ void plda_top1_decode_kernel(const unsigned long long* __restrict__ keys, long long n,
                                        float* __restrict__ score, long long* __restrict__ index) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= n) return;
  const unsigned long long key = keys[i];
  const unsigned u = (unsigned)(key >> 32);
  const unsigned bits = (u & 0x80000000u) ? (u & 0x7fffffffu) : ~u;
  score[i] = key ? __uint_as_float(bits) : -INFINITY;
  index[i] = key ? (long long)(0xffffffffu - (unsigned)(key & 0xffffffffull)) : -1;
}

// Candidate of a top-k merge: larger score first (top1_key's order-preserving bits), then the lower index, then the
// lower position in the input (c < 0: none).
struct MergeCand {
  unsigned u;
  long long idx;
  int c;
};
__device__ __forceinline__ bool merge_before(const MergeCand& a, const MergeCand& b) {
  if (a.c < 0) return false;
  if (b.c < 0) return true;
  if (a.u != b.u) return a.u > b.u;
  if (a.idx != b.idx) return a.idx < b.idx;
  return a.c < b.c;
}

// One warp per row: the k best of the row's num_lists x k_in (score, index) candidates (index < 0: none), best first,
// ties to the lower index, padded with (-inf, -1).  A lane holds the best of its candidates (positions lane, lane + 32,
// ...); each round the warp takes the best of the lanes' and only the lane that gave it looks for its next one.
__global__ void topk_merge_kernel(const float* __restrict__ s_in, const long long* __restrict__ i_in, int num_lists,
                                  long long n_rows, int k_in, int k, float* __restrict__ s_out,
                                  long long* __restrict__ i_out) {
  const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= n_rows) return;
  const int lane = threadIdx.x & 31;
  const int n_cand = num_lists * k_in;
  auto next_after = [&](const MergeCand& prev) {   // my best candidate that comes after prev (prev.c < 0: no bound)
    MergeCand b{0u, 0, -1};
    for (int c = lane; c < n_cand; c += 32) {
      const long long off = ((long long)(c / k_in) * n_rows + row) * k_in + c % k_in;
      const long long idx = i_in[off];
      if (idx < 0) continue;
      const unsigned bits = __float_as_uint(s_in[off]);
      const MergeCand x{(bits & 0x80000000u) ? ~bits : (bits | 0x80000000u), idx, c};
      if ((prev.c < 0 || merge_before(prev, x)) && merge_before(x, b)) b = x;
    }
    return b;
  };
  MergeCand mine = next_after(MergeCand{0u, 0, -1});
  float out_s = -INFINITY;
  long long out_i = -1;
  for (int i = 0; i < k; ++i) {
    MergeCand w = mine;
    for (int o = 16; o > 0; o >>= 1) {
      const MergeCand x{__shfl_xor_sync(0xffffffffu, w.u, o), __shfl_xor_sync(0xffffffffu, w.idx, o),
                        __shfl_xor_sync(0xffffffffu, w.c, o)};
      if (merge_before(x, w)) w = x;
    }
    if (w.c < 0) break;                            // warp-uniform: fewer than k candidates
    if (lane == i) {
      out_s = __uint_as_float((w.u & 0x80000000u) ? (w.u & 0x7fffffffu) : ~w.u);
      out_i = w.idx;
    }
    if (mine.c == w.c) mine = next_after(w);
  }
  if (lane < k) {
    s_out[row * k + lane] = out_s;
    i_out[row * k + lane] = out_i;
  }
}

int topk_merge(const float* s_in, const long long* i_in, int num_lists, long long n_rows, int k_in, int k, float* s_out,
               long long* i_out, cudaStream_t st) {
  if (n_rows <= 0) return KTF_OK;
  topk_merge_kernel<<<(unsigned)((n_rows + 7) / 8), 256, 0, st>>>(s_in, i_in, num_lists, n_rows, k_in, k, s_out, i_out);
  KTF_LAUNCH_OK();
  return KTF_OK;
}

// Operands of the tensor-core score GEMM, in the handle's workspace: the fp16 hi/lo splits of both sides (K = 3 dim) and
// A_i / B_j, followed by `extra` bytes of the caller's.
struct TcOperands {
  const __half* A;
  const __half* B;
  const float* Ai;
  const float* Bj;
  char* extra;
};

int tc_operands(const ktf_plda* p, const float* ut, int64_t nt, const float* ue, int64_t ne, size_t extra,
                cudaStream_t st, TcOperands* o) {
  const int dim = p->dim;
  const long long K = 3LL * dim;
  ktf::Carver cv;
  const size_t o_a = cv.take((size_t)nt * K * sizeof(__half));
  const size_t o_b = cv.take((size_t)ne * K * sizeof(__half));
  const size_t o_ai = cv.take((size_t)nt * sizeof(float));
  const size_t o_bj = cv.take((size_t)ne * sizeof(float));
  const size_t o_extra = cv.take(extra);
  int rc = p->ws.ensure(cv.off);
  if (rc != KTF_OK) return rc;
  char* base = static_cast<char*>(p->ws.ptr);
  __half* As = reinterpret_cast<__half*>(base + o_a);
  __half* Bs = reinterpret_cast<__half*>(base + o_b);
  float* Ai = reinterpret_cast<float*>(base + o_ai);
  float* Bj = reinterpret_cast<float*>(base + o_bj);
  plda_quad_kernel<float><<<(unsigned)((nt + 7) / 8), 256, 0, st>>>(ut, nt, dim, (const float*)p->d_wa,
                                                                    (float)p->logdet_term, Ai);
  KTF_LAUNCH_OK();
  plda_quad_kernel<float><<<(unsigned)((ne + 7) / 8), 256, 0, st>>>(ue, ne, dim, (const float*)p->d_wb, 0.0f, Bj);
  KTF_LAUNCH_OK();
  auto blocks = [](long long items) {
    return (unsigned)std::min<long long>((items + 255) / 256, (long long)ktf::num_sms() * 16);
  };
  plda_split_kernel<<<blocks(nt * dim), 256, 0, st>>>(ut, nt, dim, (const float*)p->d_c, 0, As);
  KTF_LAUNCH_OK();
  plda_split_kernel<<<blocks(ne * dim), 256, 0, st>>>(ue, ne, dim, nullptr, 1, Bs);
  KTF_LAUNCH_OK();
  *o = TcOperands{As, Bs, Ai, Bj, base + o_extra};
  return KTF_OK;
}

// top1_score / top1_index non-null: no score matrix, the best enrolled column of every test row instead.
int score_tc(const ktf_plda* p, const float* ut, int64_t nt, const float* ue, int64_t ne, void* scores, int64_t ld,
             int scores_bf16, cudaStream_t st, float* top1_score = nullptr, long long* top1_index = nullptr) {
  const long long K = 3LL * p->dim;
  TcOperands o;
  int rc = tc_operands(p, ut, nt, ue, ne, top1_score ? (size_t)nt * sizeof(unsigned long long) : 0, st, &o);
  if (rc != KTF_OK) return rc;
  if (top1_score == nullptr)
    return ktf::tc_gemm_nt(o.A, nt, K, o.B, ne, K, K, /*fp16=*/1, o.Ai, o.Bj, scores, ld, scores_bf16, st);
  unsigned long long* keys = reinterpret_cast<unsigned long long*>(o.extra);
  KTF_CUDA(cudaMemsetAsync(keys, 0, (size_t)nt * sizeof(unsigned long long), st));
  if ((rc = ktf::tc_gemm_nt(o.A, nt, K, o.B, ne, K, K, /*fp16=*/1, o.Ai, o.Bj, nullptr, ne, 0, st, keys)) != KTF_OK)
    return rc;
  plda_top1_decode_kernel<<<(unsigned)((nt + 255) / 256), 256, 0, st>>>(keys, nt, top1_score, top1_index);
  KTF_LAUNCH_OK();
  return KTF_OK;
}

// The k best enrolled columns of every test row: the score GEMM leaves partial lists (one per n-range and column quarter
// of a row) in the workspace, topk_merge reduces them to (nt, k).
int score_tc_topk(const ktf_plda* p, const float* ut, int64_t nt, const float* ue, int64_t ne, int k, float* score,
                  long long* index, cudaStream_t st) {
  const long long K = 3LL * p->dim;
  const int lists = ktf::tc_topk_lists(nt, ne, K);
  if (lists == 0) return topk_merge(nullptr, nullptr, 0, nt, k, k, score, index, st);   // no enrolled vector
  const size_t n_part = (size_t)lists * nt * k;
  const size_t s_bytes = (n_part * sizeof(float) + 255) & ~(size_t)255;
  TcOperands o;
  int rc = tc_operands(p, ut, nt, ue, ne, s_bytes + n_part * sizeof(long long), st, &o);
  if (rc != KTF_OK) return rc;
  float* part_s = reinterpret_cast<float*>(o.extra);
  long long* part_i = reinterpret_cast<long long*>(o.extra + s_bytes);
  if ((rc = ktf::tc_gemm_topk(o.A, nt, K, o.B, ne, K, K, /*fp16=*/1, o.Ai, o.Bj, k, part_s, part_i, st)) != KTF_OK)
    return rc;
  return topk_merge(part_s, part_i, lists, nt, k, k, score, index, st);
}

template <typename T>
int upload_as(void** dst, const std::vector<double>& v) {
  std::vector<T> tmp(v.size());
  for (size_t i = 0; i < v.size(); ++i) tmp[i] = (T)v[i];
  return ktf::upload((T**)dst, tmp.data(), tmp.size());
}

template <typename T>
int transform_impl(const ktf_plda* p, const float* x, int64_t n, T* u, cudaStream_t st) {
  const int dim = p->dim;
  CastLoad<T> al{x, (long long)dim};
  ktf::DenseLoad<T> bl{(const T*)p->d_T, (long long)dim};
  OffsetEpi<T> epi{u, (const T*)p->d_offset, dim};
  dim3 grid((unsigned)((n + ktf::kTileM - 1) / ktf::kTileM), (unsigned)((dim + ktf::kTileN - 1) / ktf::kTileN));
  ktf::gemm_nt_kernel<T><<<grid, ktf::kGemmThreads, 0, st>>>((long long)n, (long long)dim, dim, al, bl, epi);
  KTF_LAUNCH_OK();
  if (p->normalize_length) {
    plda_norm_kernel<T><<<(unsigned)((n + 7) / 8), 256, 0, st>>>(u, n, dim, (const T*)p->d_psi,
                                                                 p->simple_length_norm, (T)(1.0 / p->num_examples));
    KTF_LAUNCH_OK();
  }
  return KTF_OK;
}

template <typename T>
int score_impl(const ktf_plda* p, const T* ut, int64_t nt, const T* ue, int64_t ne, T* scores, int64_t ld,
               cudaStream_t st) {
  const int dim = p->dim;
  ktf::Scratch scratch(st);            // released on every exit path
  T* ab = nullptr;
  KTF_CUDA(scratch.take(&ab, (size_t)(nt + ne) * sizeof(T)));
  T* A = ab;
  T* B = ab + nt;
  plda_quad_kernel<T><<<(unsigned)((nt + 7) / 8), 256, 0, st>>>(ut, nt, dim, (const T*)p->d_wa,
                                                                (T)p->logdet_term, A);
  KTF_LAUNCH_OK();
  plda_quad_kernel<T><<<(unsigned)((ne + 7) / 8), 256, 0, st>>>(ue, ne, dim, (const T*)p->d_wb, T(0), B);
  KTF_LAUNCH_OK();
  ScaledLoad<T> al{ut, (const T*)p->d_c, (long long)dim};
  ktf::DenseLoad<T> bl{ue, (long long)dim};
  ScoreEpi<T> epi{scores, A, B, (long long)ld};
  dim3 grid((unsigned)((nt + ktf::kTileM - 1) / ktf::kTileM), (unsigned)((ne + ktf::kTileN - 1) / ktf::kTileN));
  ktf::gemm_nt_kernel<T><<<grid, ktf::kGemmThreads, 0, st>>>((long long)nt, (long long)ne, dim, al, bl, epi);
  KTF_LAUNCH_OK();
  return KTF_OK;
}

}  // namespace

extern "C" {

int ktf_plda_create(int32_t dim, const double* mean_host, const double* transform_host,
                    const double* psi_host, int32_t normalize_length, int32_t simple_length_norm,
                    int32_t dtype_bytes, ktf_plda** out) {
  return ktf_plda_create_ex(dim, mean_host, transform_host, psi_host, normalize_length, simple_length_norm,
                            dtype_bytes, 1.0, out);
}

int ktf_plda_create_ex(int32_t dim, const double* mean_host, const double* transform_host,
                       const double* psi_host, int32_t normalize_length, int32_t simple_length_norm,
                       int32_t dtype_bytes, double num_examples, ktf_plda** out) {
  KTF_CHECK_ARG(mean_host && transform_host && psi_host && out, "ktf_plda_create: null argument");
  KTF_CHECK_ARG(num_examples > 0.0, "num_examples must be greater than 0");
  KTF_CHECK_ARG(dim > 0, "dim must be > 0");
  KTF_CHECK_ARG(dtype_bytes == 4 || dtype_bytes == 8, "dtype_bytes must be 4 or 8");
  ktf_plda* p = new ktf_plda();
  p->dim = dim;
  p->normalize_length = normalize_length;
  p->simple_length_norm = simple_length_norm;
  p->dtype_bytes = dtype_bytes;
  p->num_examples = num_examples;
  const double ne = num_examples;
  const bool f32 = dtype_bytes == 4;
  // Parameters are first rounded to the layer dtype, like tf.constant(..., dtype) (plda.py:103-105).
  auto rnd = [&](double v) { return f32 ? (double)(float)v : v; };
  std::vector<double> Tm((size_t)dim * dim), off(dim), psi(dim), c(dim), wa(dim), wb(dim);
  for (size_t i = 0; i < Tm.size(); ++i) Tm[i] = rnd(transform_host[i]);
  double ld1 = 0.0, ld0 = 0.0;
  for (int r = 0; r < dim; ++r) {
    double acc = 0.0;
    for (int k = 0; k < dim; ++k) acc += Tm[(size_t)r * dim + k] * rnd(mean_host[k]);
    off[r] = rnd(-acc);                                        // plda.py:116
    psi[r] = rnd(psi_host[r]);
    const double rr = ne * psi[r] / (ne * psi[r] + 1.0);       // plda.py:228-231: mean = rr * u_enrolled
    const double v1 = 1.0 + psi[r] / (ne * psi[r] + 1.0), v0 = 1.0 + psi[r];
    c[r] = rr / v1;
    wa[r] = 0.5 / v0 - 0.5 / v1;
    wb[r] = -0.5 * rr * rr / v1;
    ld1 += log(v1);
    ld0 += log(v0);
  }
  p->logdet_term = -0.5 * (ld1 - ld0);
  int rc;
  auto fail = [&](int code) { ktf_plda_destroy(p); return code; };
#define UP(dst, vec)                                                          \
  if ((rc = f32 ? upload_as<float>(&p->dst, vec) : upload_as<double>(&p->dst, vec)) != KTF_OK) return fail(rc)
  UP(d_T, Tm);
  UP(d_offset, off);
  UP(d_psi, psi);
  UP(d_c, c);
  UP(d_wa, wa);
  UP(d_wb, wb);
#undef UP
  // tensor-core path: fp32 handle, sm_100 device, K = 3*dim a multiple of 8, and operands that stay far
  // inside the fp16 range: after length normalisation |u_d| <= sqrt(dim * (psi_d + 1)).
  if (f32 && dim % 8 == 0 && normalize_length && ktf_device_arch() >= 100) {
    double bound = 0.0;
    for (int r = 0; r < dim; ++r) bound = std::max(bound, sqrt((double)dim * (psi[r] + 1.0 / ne)));
    p->use_tc = bound < 3.0e4;
  }
  *out = p;
  return KTF_OK;
}

void ktf_plda_destroy(ktf_plda* p) {
  if (!p) return;
  p->ws.release();
  cudaFree(p->d_T);
  cudaFree(p->d_offset);
  cudaFree(p->d_psi);
  cudaFree(p->d_c);
  cudaFree(p->d_wa);
  cudaFree(p->d_wb);
  delete p;
}

int ktf_plda_transform(const ktf_plda* p, const float* x_dev, int64_t n, void* u_dev, void* stream) {
  KTF_CHECK_ARG(p && x_dev && u_dev, "ktf_plda_transform: null argument");
  if (n <= 0) return KTF_OK;
  cudaStream_t st = (cudaStream_t)stream;
  return p->dtype_bytes == 4 ? transform_impl<float>(p, x_dev, n, (float*)u_dev, st)
                             : transform_impl<double>(p, x_dev, n, (double*)u_dev, st);
}

int ktf_plda_score_ex(const ktf_plda* p, const void* u_test_dev, int64_t n_test, const void* u_enroll_dev,
                      int64_t n_enroll, void* scores_dev, int64_t ld, int32_t score_format, void* stream) {
  KTF_CHECK_ARG(p && u_test_dev && u_enroll_dev && scores_dev, "ktf_plda_score: null argument");
  KTF_CHECK_ARG(ld >= n_enroll, "ld must be >= n_enroll");
  KTF_CHECK_ARG(score_format == KTF_SCORES_NATIVE || score_format == KTF_SCORES_BF16, "bad score_format");
  if (score_format == KTF_SCORES_BF16) {
    KTF_CHECK_ARG(p->use_tc, "KTF_SCORES_BF16 needs a float32 handle (the tcgen05 score GEMM)");
    if (n_test <= 0 || n_enroll <= 0) return KTF_OK;
    return score_tc(p, (const float*)u_test_dev, n_test, (const float*)u_enroll_dev, n_enroll, scores_dev, ld, 1,
                    (cudaStream_t)stream);
  }
  return ktf_plda_score(p, u_test_dev, n_test, u_enroll_dev, n_enroll, scores_dev, ld, stream);
}

int ktf_plda_score_top1(const ktf_plda* p, const void* u_test_dev, int64_t n_test, const void* u_enroll_dev,
                        int64_t n_enroll, float* best_score_dev, int64_t* best_index_dev, void* stream) {
  KTF_CHECK_ARG(p && u_test_dev && u_enroll_dev && best_score_dev && best_index_dev, "ktf_plda_score_top1: null argument");
  KTF_CHECK_ARG(p->use_tc, "ktf_plda_score_top1 needs a float32 PLDA handle on an sm_100 device");
  KTF_CHECK_ARG(n_enroll < (1LL << 32), "ktf_plda_score_top1: more than 2^32 enrolled vectors");
  if (n_test <= 0) return KTF_OK;
  return score_tc(p, (const float*)u_test_dev, n_test, (const float*)u_enroll_dev, n_enroll, nullptr, n_enroll, 0,
                  (cudaStream_t)stream, best_score_dev, (long long*)best_index_dev);
}

int ktf_plda_score_topk(const ktf_plda* p, const void* u_test_dev, int64_t n_test, const void* u_enroll_dev,
                        int64_t n_enroll, int32_t k, float* scores_dev, int64_t* index_dev, void* stream) {
  KTF_CHECK_ARG(p, "ktf_plda_score_topk: null handle");
  KTF_CHECK_ARG(k >= 1 && k <= KTF_PLDA_TOPK_MAX, "ktf_plda_score_topk: k = %d, must be 1 .. %d (KTF_PLDA_TOPK_MAX)", k,
                KTF_PLDA_TOPK_MAX);
  KTF_CHECK_ARG(p->use_tc, "ktf_plda_score_topk needs a float32 PLDA handle on an sm_100 device");
  KTF_CHECK_ARG(n_enroll >= 0 && n_enroll < (1LL << 32), "ktf_plda_score_topk: n_enroll must be in 0 .. 2^32 - 1");
  if (n_test <= 0) return KTF_OK;
  KTF_CHECK_ARG(u_test_dev && scores_dev && index_dev && (u_enroll_dev || n_enroll == 0),
                "ktf_plda_score_topk: null argument");
  return score_tc_topk(p, (const float*)u_test_dev, n_test, (const float*)u_enroll_dev, n_enroll, k, scores_dev,
                       (long long*)index_dev, (cudaStream_t)stream);
}

int ktf_topk_merge(const float* scores_in_dev, const int64_t* index_in_dev, int32_t num_lists, int64_t n_rows,
                   int32_t k_in, int32_t k, float* scores_dev, int64_t* index_dev, void* stream) {
  KTF_CHECK_ARG(k >= 1 && k <= KTF_PLDA_TOPK_MAX, "ktf_topk_merge: k = %d, must be 1 .. %d (KTF_PLDA_TOPK_MAX)", k,
                KTF_PLDA_TOPK_MAX);
  KTF_CHECK_ARG(num_lists >= 0 && k_in >= 1 && (long long)num_lists * k_in < (1LL << 31),
                "ktf_topk_merge: bad num_lists / k_in");
  if (n_rows <= 0) return KTF_OK;
  KTF_CHECK_ARG(scores_dev && index_dev && (num_lists == 0 || (scores_in_dev && index_in_dev)),
                "ktf_topk_merge: null argument");
  return topk_merge(scores_in_dev, (const long long*)index_in_dev, num_lists, n_rows, k_in, k, scores_dev,
                    (long long*)index_dev, (cudaStream_t)stream);
}

int ktf_plda_score(const ktf_plda* p, const void* u_test_dev, int64_t n_test, const void* u_enroll_dev,
                   int64_t n_enroll, void* scores_dev, int64_t ld, void* stream) {
  KTF_CHECK_ARG(p && u_test_dev && u_enroll_dev && scores_dev, "ktf_plda_score: null argument");
  KTF_CHECK_ARG(ld >= n_enroll, "ld must be >= n_enroll");
  if (n_test <= 0 || n_enroll <= 0) return KTF_OK;
  cudaStream_t st = (cudaStream_t)stream;
  if (p->use_tc)
    return score_tc(p, (const float*)u_test_dev, n_test, (const float*)u_enroll_dev, n_enroll, scores_dev, ld, 0, st);
  return p->dtype_bytes == 4
             ? score_impl<float>(p, (const float*)u_test_dev, n_test, (const float*)u_enroll_dev, n_enroll,
                                 (float*)scores_dev, ld, st)
             : score_impl<double>(p, (const double*)u_test_dev, n_test, (const double*)u_enroll_dev,
                                  n_enroll, (double*)scores_dev, ld, st);
}

}  // extern "C"

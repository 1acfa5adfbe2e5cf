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
#include <assert.h>
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

// Decodes the best-entry keys of tc_gemm_score(row_best): score and column of every test row (-1: no enrolled vector).
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

// ---- AS-norm: per-vector statistics of the top-N cohort scores, normalised score matrix ----
constexpr int kSelThreads = 512;
constexpr int kSelBins = 4096;                    // histogram bins of the first radix pass (12 bits); the others use 10
constexpr long long kSelSmemRowMax = 48 * 1024;   // rows up to this long are held in shared memory as keys (208 KB)
constexpr double kCohortChunkBytes = 64e6;        // raw cohort scores per chunk: written by the GEMM, read from L2
// Score chunk of the k > 32 top-k path: 512 rows at 50 000 columns.  Twice the cohort chunk halves the selection's
// tail wave (256 -> 512 CTAs on 148 SMs); measured 15 % faster at 50 000 columns (DESIGN K5 (vi)).
constexpr double kTopkChunkBytes = 128e6;

__device__ __forceinline__ unsigned order_key(float v) {   // unsigned order = float order
  const unsigned b = __float_as_uint(v);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float key_value(unsigned k) {
  return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

// f(c, key(c)) for c = tid, tid + kSelThreads, ... < n in increasing c, with eight key loads in flight per thread (a
// row that is not in shared memory is read from L2, and one dependent load per iteration would leave the CTA waiting).
template <typename KeyFn, typename F>
__device__ __forceinline__ void for_each_key(const KeyFn& key, long long n, const F& f) {
  constexpr int kIlp = 8;
  long long c = threadIdx.x;
  for (; c + (kIlp - 1) * kSelThreads < n; c += kIlp * kSelThreads) {
    unsigned k[kIlp];
#pragma unroll
    for (int u = 0; u < kIlp; ++u) k[u] = key(c + u * kSelThreads);
#pragma unroll
    for (int u = 0; u < kIlp; ++u) f(c + u * kSelThreads, k[u]);
  }
  for (; c < n; c += kSelThreads) f(c, key(c));
}

// Exact need-th largest of the keys key(c), c < n, of one row (need >= 1; key 0 is not counted -- order_key gives it
// only to the NaN 0xffffffff): radix select, three passes of 12 + 10 + 10 bits, each a shared-memory histogram (hist:
// kSelBins) of the keys under the prefix found so far.  Returns that key (thr), how many keys equal to it are among the
// need largest (eq), how many there are (n_eq) and count = need; with fewer than need counted keys thr = eq = n_eq = 0
// and count = the number of counted keys.  Called by all kSelThreads threads of the CTA.
struct Selected {
  unsigned thr, eq, n_eq, count;
};
template <typename KeyFn>
__device__ Selected radix_select(KeyFn key, long long n, unsigned need, unsigned* hist) {
  __shared__ unsigned s_warp[kSelThreads / 32];
  __shared__ unsigned s_digit, s_need, s_neq;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const unsigned n_want = need;
  unsigned prefix = 0, pmask = 0;   // need: rank of the target among the keys under the prefix
  for (int pass = 0; pass < 3; ++pass) {
    const int shift = pass == 0 ? 20 : (pass == 1 ? 10 : 0);
    const unsigned nb = pass == 0 ? 4096u : 1024u, per = nb / kSelThreads;
    for (unsigned b = tid; b < nb; b += kSelThreads) hist[b] = 0;
    __syncthreads();                              // (first pass: the keys may be in shared memory too)
    for_each_key(key, n, [&](long long, unsigned k) {
      if (k != 0 && (k & pmask) == prefix) atomicAdd(&hist[(k >> shift) & (nb - 1)], 1u);
    });
    __syncthreads();
    // the digit d with #(keys above d) < need <= #(keys at or above d); thread t owns bins [t per, (t + 1) per)
    unsigned loc = 0;
    for (unsigned i = 0; i < per; ++i) loc += hist[tid * per + i];
    unsigned incl = loc;                          // sum over this and the higher lanes of the warp
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned v = __shfl_down_sync(0xffffffffu, incl, o);
      if (lane + o < 32) incl += v;
    }
    if (lane == 0) s_warp[warp] = incl;
    __syncthreads();
    unsigned above = incl - loc;
    for (int w = warp + 1; w < kSelThreads / 32; ++w) above += s_warp[w];
    if (pass == 0) {
      unsigned total = 0;
      for (int w = 0; w < kSelThreads / 32; ++w) total += s_warp[w];
      if (total < need) {                         // CTA-uniform: every counted key is listed
        __syncthreads();                          // hist / s_warp are rewritten by the caller or the next call
        return Selected{0u, 0u, 0u, total};
      }
    }
    if (above < need && need <= above + loc) {    // exactly one thread
      unsigned acc = above;
      for (int i = (int)per - 1; i >= 0; --i) {
        const unsigned h = hist[tid * per + i];
        if (need <= acc + h) {
          s_digit = tid * per + (unsigned)i;
          s_need = need - acc;
          s_neq = h;
          break;
        }
        acc += h;
      }
    }
    __syncthreads();
    prefix |= s_digit << shift;
    pmask |= (nb - 1) << shift;
    need = s_need;
    const unsigned n_eq = s_neq;
    __syncthreads();                              // hist / s_warp / s_digit are rewritten by the next pass
    if (pass == 2) return Selected{prefix, need, n_eq, n_want};
  }
  return Selected{};
}

// One CTA per row of a chunk of raw cohort accumulators x (pitch ld).  The score is (x + first) + second: column addend
// then row addend for the test role (B of the cohort vector, A of the test vector), row addend then column addend for
// the enrolled role (B of the enrolled vector, A of the cohort vector) -- the association of the score GEMM's epilogue,
// so every score is bit-equal to its logLikelihoodRatio entry.
// Exact top_n-th largest score: radix select on order keys, three passes of 12 + 10 + 10 bits, each a shared-memory
// histogram of the keys under the prefix found so far.  Mean and std of the top_n multiset in float64, relative to that
// threshold t: the keys above it contribute x - t and (x - t)^2, the (top_n - count above) copies of t contribute 0.
// Every thread sums its columns in index order and the CTA adds the threads' sums in a fixed tree, so the statistics
// depend on the row alone (not on its batch-mates or the chunking).
__global__ void __launch_bounds__(kSelThreads) cohort_select_kernel(const float* __restrict__ x, long long ld,
                                                                    long long nc, const float* __restrict__ row_add,
                                                                    const float* __restrict__ col_add, int row_first,
                                                                    unsigned top_n, int in_smem, float* __restrict__ mean,
                                                                    float* __restrict__ stdev, float* __restrict__ nth) {
  extern __shared__ unsigned sel_smem[];
  unsigned* hist = sel_smem;                  // [kSelBins]
  unsigned* keys = sel_smem + kSelBins;       // [nc] when in_smem
  __shared__ double s_sum[kSelThreads / 32], s_sq[kSelThreads / 32];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const long long row = blockIdx.x;
  const float* xr = x + row * ld;
  const float ra = row_add[row];
  auto key_at = [&](long long c) {
    return order_key(row_first ? (xr[c] + ra) + col_add[c] : (xr[c] + col_add[c]) + ra);
  };
  if (in_smem)
    for (long long c = tid; c < nc; c += kSelThreads) keys[c] = key_at(c);
  auto key = [&](long long c) { return in_smem ? keys[c] : key_at(c); };

  // top_n <= nc finite scores: the threshold always exists
  const unsigned prefix = radix_select(key, nc, top_n, hist).thr;
  const double thr = (double)key_value(prefix);
  double sum = 0.0, sq = 0.0;
  for (long long c = tid; c < nc; c += kSelThreads) {
    const unsigned k = key(c);
    if (k > prefix) {
      const double d = (double)key_value(k) - thr;
      sum += d;
      sq += d * d;
    }
  }
  for (int o = 16; o > 0; o >>= 1) {
    sum += __shfl_xor_sync(0xffffffffu, sum, o);
    sq += __shfl_xor_sync(0xffffffffu, sq, o);
  }
  if (lane == 0) {
    s_sum[warp] = sum;
    s_sq[warp] = sq;
  }
  __syncthreads();
  if (tid == 0) {
    double S = 0.0, Q = 0.0;
    for (int w = 0; w < kSelThreads / 32; ++w) {
      S += s_sum[w];
      Q += s_sq[w];
    }
    const double m = S / (double)top_n;
    mean[row] = (float)(thr + m);
    stdev[row] = (float)sqrt(fmax(Q / (double)top_n - m * m, 0.0));
    if (nth != nullptr) nth[row] = (float)thr;
  }
}

// Per-row (A_i, 0.5 / sigma_t, mu_t, 0) and per-column 0.5 / sigma_e of the normalising epilogue (IEEE divisions: a
// sigma of 0 gives inf, and the score the IEEE quotient; 0.5 / sigma is exactly half of 1 / sigma).
__global__ void asnorm_prep_kernel(const float* __restrict__ Ai, const float* __restrict__ t_mean,
                                   const float* __restrict__ t_std, long long nt, const float* __restrict__ e_std,
                                   long long ne, float4* __restrict__ row, float* __restrict__ e_half_inv) {
  const long long items = nt > ne ? nt : ne;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < items; i += (long long)gridDim.x * blockDim.x) {
    if (i < nt) row[i] = make_float4(Ai[i], 0.5f / t_std[i], t_mean[i], 0.0f);
    if (i < ne) e_half_inv[i] = 0.5f / e_std[i];
  }
}

// Statistics of the normalising epilogue: the caller's per-vector mean and std of both sides (device, float32).
struct AsnormStats {
  const float* t_mean;
  const float* t_std;
  const float* e_mean;
  const float* e_std;
};

// Operands of the tensor-core score GEMM, in the handle's workspace: the fp16 hi/lo splits of both sides (K = 3 dim) and
// A_i / B_j; for AS-norm scores the per-row float4 and per-column 0.5 / sigma_e of asnorm_prep_kernel; then `extra`
// bytes of the caller's.  The GEMM's rows are normally the test vectors (c-scaled split, A addend) and its columns the
// enrolled ones (plain split, B addend).  With `enrolled_rows` (raw scores) the roles swap sides: the rows (ut) are
// enrolled vectors and get the plain split and the B addend, the columns (ue) play the test role.  The cross term is
// symmetric and the three partial products meet the same K positions, so the accumulator is the transpose of the normal
// one; Ai / Bj are then the row / column addends (B of the rows, A of the columns).
struct TcOperands {
  const __half* A;
  const __half* B;
  long long K;
  const float* Ai;
  const float* Bj;
  const float* row;          // the GEMM's per-row addend: Ai, or for AS-norm scores (nt) float4
  const float* e_half_inv;   // AS-norm: (ne); otherwise null
  const float* e_mean;       // AS-norm: the caller's; otherwise null
  char* extra;

  // The score GEMM of rows [r0, r0 + rows) against n columns, rows output C (null for the other outputs).
  ktf::TcScore gemm(long long r0, long long rows, long long n, const float* row_add, const float* col_add, void* C,
                    long long ldc, int c_bf16 = 0) const {
    return ktf::TcScore{A + r0 * K, rows, K, B, n, K, K, /*fp16=*/1,
                        row_add == nullptr ? nullptr : row_add + (e_half_inv ? 4 : 1) * r0, col_add, e_half_inv, e_mean,
                        C, ldc, c_bf16};
  }
};

int tc_operands(const ktf_plda* p, const float* ut, int64_t nt, const float* ue, int64_t ne, const AsnormStats* norm,
                size_t extra, cudaStream_t st, TcOperands* o, bool enrolled_rows = false) {
  const int dim = p->dim;
  const long long K = 3LL * dim;
  ktf::Carver cv;
  const size_t o_a = cv.take((size_t)nt * K * sizeof(__half));
  const size_t o_b = cv.take((size_t)ne * K * sizeof(__half));
  const size_t o_ai = cv.take((size_t)nt * sizeof(float));
  const size_t o_bj = cv.take((size_t)ne * sizeof(float));
  const size_t o_row = cv.take(norm ? (size_t)nt * sizeof(float4) : 0);
  const size_t o_half_inv = cv.take(norm ? (size_t)ne * sizeof(float) : 0);
  const size_t o_extra = cv.take(extra);
  int rc = p->ws.ensure(cv.off);
  if (rc != KTF_OK) return rc;
  char* base = static_cast<char*>(p->ws.ptr);
  __half* As = reinterpret_cast<__half*>(base + o_a);
  __half* Bs = reinterpret_cast<__half*>(base + o_b);
  float* Ai = reinterpret_cast<float*>(base + o_ai);
  float* Bj = reinterpret_cast<float*>(base + o_bj);
  const float* wa = (const float*)p->d_wa;
  const float* wb = (const float*)p->d_wb;
  const float* c = (const float*)p->d_c;
  const float ld = (float)p->logdet_term;
  plda_quad_kernel<float><<<(unsigned)((nt + 7) / 8), 256, 0, st>>>(ut, nt, dim, enrolled_rows ? wb : wa,
                                                                    enrolled_rows ? 0.0f : ld, Ai);
  KTF_LAUNCH_OK();
  plda_quad_kernel<float><<<(unsigned)((ne + 7) / 8), 256, 0, st>>>(ue, ne, dim, enrolled_rows ? wa : wb,
                                                                    enrolled_rows ? ld : 0.0f, Bj);
  KTF_LAUNCH_OK();
  auto blocks = [](long long items) {
    return (unsigned)std::min<long long>((items + 255) / 256, (long long)ktf::num_sms() * 16);
  };
  plda_split_kernel<<<blocks(nt * dim), 256, 0, st>>>(ut, nt, dim, enrolled_rows ? nullptr : c, enrolled_rows ? 1 : 0,
                                                      As);
  KTF_LAUNCH_OK();
  plda_split_kernel<<<blocks(ne * dim), 256, 0, st>>>(ue, ne, dim, enrolled_rows ? c : nullptr, enrolled_rows ? 0 : 1,
                                                      Bs);
  KTF_LAUNCH_OK();
  *o = TcOperands{As, Bs, K, Ai, Bj, Ai, nullptr, nullptr, base + o_extra};
  if (norm != nullptr) {
    float4* row = reinterpret_cast<float4*>(base + o_row);
    float* e_half_inv = reinterpret_cast<float*>(base + o_half_inv);
    asnorm_prep_kernel<<<blocks(std::max<long long>(nt, ne)), 256, 0, st>>>(Ai, norm->t_mean, norm->t_std, nt,
                                                                           norm->e_std, ne, row, e_half_inv);
    KTF_LAUNCH_OK();
    o->row = reinterpret_cast<const float*>(row);
    o->e_half_inv = e_half_inv;
    o->e_mean = norm->e_mean;
  }
  return KTF_OK;
}

// Rows of a chunk of n rows of pitch ld floats: at most `bytes`, whole pair tiles when there are enough.
long long chunk_rows(long long ld, long long n, double bytes) {
  long long chunk = std::max(1LL, (long long)(bytes / (double)(ld * (long long)sizeof(float))));
  if (chunk >= 256) chunk = chunk / 256 * 256;
  return std::min<long long>(chunk, n);
}

// Cohort statistics of n vectors: the raw score GEMM against the cohort runs in row chunks of at most
// kCohortChunkBytes into the workspace, each chunk is selected while it is still in L2.
int cohort_stats_tc(const ktf_plda* p, const float* u, int64_t n, const float* uc, int64_t nc, long long top_n,
                    bool enrolled, float* mean, float* stdev, float* nth, cudaStream_t st) {
  const long long K = 3LL * p->dim;
  const long long ld = (nc + 3) / 4 * 4;          // 16-byte row pitch: the GEMM's boxed stores
  const long long chunk = chunk_rows(ld, n, kCohortChunkBytes);
  TcOperands o;
  int rc = tc_operands(p, u, n, uc, nc, nullptr, (size_t)chunk * ld * sizeof(float), st, &o, enrolled);
  if (rc != KTF_OK) return rc;
  float* raw = reinterpret_cast<float*>(o.extra);
  const int in_smem = nc <= kSelSmemRowMax;
  const size_t smem = (size_t)(kSelBins + (in_smem ? nc : 0)) * sizeof(unsigned);
  static unsigned long long attr_done = 0;
  if (ktf::first_use_on_device(&attr_done))
    KTF_CUDA(cudaFuncSetAttribute(cohort_select_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)((kSelBins + kSelSmemRowMax) * sizeof(unsigned))));
  for (long long r0 = 0; r0 < n; r0 += chunk) {
    const long long rows = std::min(chunk, (long long)n - r0);
    if ((rc = ktf::tc_gemm_score(o.gemm(r0, rows, nc, nullptr, nullptr, raw, ld), st)) != KTF_OK) return rc;
    cohort_select_kernel<<<(unsigned)rows, kSelThreads, smem, st>>>(raw, ld, nc, o.Ai + r0, o.Bj, enrolled ? 1 : 0,
                                                                     (unsigned)top_n, in_smem, mean + r0, stdev + r0,
                                                                     nth ? nth + r0 : nullptr);
    KTF_LAUNCH_OK();
  }
  return KTF_OK;
}

// ---- the k best of a row for k up to KTF_PLDA_TOPK_LARGE_MAX: radix select, ordered emit, bitonic sort ----
// Built with -DKTF_SELECT_CHECKS, topk_select_kernel asserts every shared-memory index and the global candidate it
// reads and writes against the bounds the launch gives it (a bounds-checked build of the selection); otherwise the
// checks compile to nothing.
#ifdef KTF_SELECT_CHECKS
#define KTF_SEL_CHECK(cond) assert(cond)
#else
#define KTF_SEL_CHECK(cond) ((void)0)
#endif

__device__ __forceinline__ unsigned listed_key(float v) {   // NaN and -inf are never listed: key 0
  return (isnan(v) || v == -INFINITY) ? 0u : order_key(v);
}

// Candidates of a row of a score chunk (pitch ld): candidate c is column c.
struct MatrixRows {
  const float* x;
  long long ld;
  __device__ __forceinline__ unsigned key(long long row, long long c) const {
    KTF_SEL_CHECK(row >= 0 && c >= 0 && c < ld);
    return listed_key(x[row * ld + c]);
  }
  __device__ __forceinline__ long long index(long long, long long c) const { return c; }
};

// Candidates of a row of ktf_topk_merge_large's (num_lists, n_rows, k_in) lists: candidate c is entry c % k_in of list
// c / k_in; an entry with index < 0 is none.
struct ListRows {
  const float* s;
  const long long* i;
  long long n_rows;
  int k_in;
  __device__ __forceinline__ long long at(long long row, long long c) const {
    KTF_SEL_CHECK(row >= 0 && row < n_rows && c >= 0);
    return (c / k_in * n_rows + row) * k_in + c % k_in;
  }
  __device__ __forceinline__ unsigned key(long long row, long long c) const {
    const long long o = at(row, c);
    return i[o] < 0 ? 0u : listed_key(s[o]);
  }
  __device__ __forceinline__ long long index(long long row, long long c) const { return i[at(row, c)]; }
};

// Sort entry of a listed candidate: the larger key first, then the lower candidate number (c < 2^32); 0 is none.
__device__ __forceinline__ unsigned long long cand_entry(unsigned key, long long c) {
  return ((unsigned long long)key << 32) | (0xffffffffu - (unsigned)c);
}

// One CTA per row (grid-stride): the k best of the row's n candidates -- the first k of a stable descending sort of
// their values without NaN and -inf -- best first, padded with (-inf, -1).  radix_select finds the k-th largest key;
// every key above it is emitted (shared-memory atomics: the order does not matter, the sort below fixes it), and so
// are the keys equal to it when all of them are listed; otherwise the first `eq` equal keys in candidate order follow
// (a CTA prefix count per tile of kSelThreads candidates, so equal keys are taken lowest candidate first whatever the
// scheduling).  A bitonic sort of the <= k entries in shared memory puts them in order.  Keys are held in shared memory when in_smem (n <= kSelSmemRowMax), otherwise re-read (from L2) by
// each pass.
template <typename Rows>
__global__ void __launch_bounds__(kSelThreads) topk_select_kernel(Rows rows, long long n_rows, long long n, int k,
                                                                  int in_smem, float* __restrict__ s_out,
                                                                  long long* __restrict__ i_out) {
  extern __shared__ __align__(16) unsigned topk_smem[];
  unsigned* hist = topk_smem;                                           // [kSelBins] during the select
  unsigned long long* cand = reinterpret_cast<unsigned long long*>(topk_smem);   // [k] after it (8 KB <= 16 KB)
  unsigned* keys = topk_smem + kSelBins;                                // [n] when in_smem
  __shared__ unsigned s_above, s_warp_eq[kSelThreads / 32];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
#ifdef KTF_SELECT_CHECKS
  unsigned smem_bytes;
  asm("mov.u32 %0, %%dynamic_smem_size;" : "=r"(smem_bytes));
  KTF_SEL_CHECK(blockDim.x == kSelThreads && k >= 1 && k <= KTF_PLDA_TOPK_LARGE_MAX &&
                (!in_smem || n <= kSelSmemRowMax) &&
                (kSelBins + (in_smem ? n : 0)) * sizeof(unsigned) <= smem_bytes &&
                KTF_PLDA_TOPK_LARGE_MAX * sizeof(unsigned long long) <= kSelBins * sizeof(unsigned));
#endif
  for (long long row = blockIdx.x; row < n_rows; row += gridDim.x) {
    auto row_key = [&](long long c) { return rows.key(row, c); };
    if (in_smem) for_each_key(row_key, n, [&](long long c, unsigned kc) { keys[c] = kc; });
    auto key = [&](long long c) {
      KTF_SEL_CHECK(c >= 0 && c < n);
      return in_smem ? keys[c] : rows.key(row, c);
    };
    const Selected sel = radix_select(key, n, (unsigned)k, hist);
    const unsigned thr = sel.thr, eq = sel.eq, count = sel.count;
    if (tid == 0) s_above = 0;
    __syncthreads();
    // every key equal to thr listed (no tie across rank k, or fewer than k keys): one unordered pass; otherwise the keys
    // above thr unordered, then the first eq equal ones in candidate order
    const bool all_eq = eq == sel.n_eq;
    const unsigned lo = all_eq && thr != 0 ? thr : thr + 1;            // thr < 0xffffffff: NaN keys are 0
    for_each_key(key, n, [&](long long c, unsigned kc) {
      if (kc >= lo) {
        const unsigned slot = atomicAdd(&s_above, 1u);
        KTF_SEL_CHECK(slot < (all_eq ? count : count - eq));
        cand[slot] = cand_entry(kc, c);
      }
    });
    const unsigned n_above = count - eq;
    unsigned taken = all_eq ? eq : 0u;                                  // equal keys seen so far (CTA-uniform)
    for (long long c0 = 0; c0 < n && taken < eq; c0 += kSelThreads) {  // thr > 0 here: kc == thr means c < n
      const long long c = c0 + tid;
      const unsigned kc = c < n ? key(c) : 0u;
      const unsigned ball = __ballot_sync(0xffffffffu, kc == thr);
      if (lane == 0) s_warp_eq[warp] = __popc(ball);
      __syncthreads();
      unsigned before = taken + __popc(ball & ((1u << lane) - 1u)), tile = 0;
      for (int w = 0; w < kSelThreads / 32; ++w) {
        const unsigned v = s_warp_eq[w];
        before += w < warp ? v : 0u;
        tile += v;
      }
      if (kc == thr && before < eq) {
        KTF_SEL_CHECK(n_above + before < count);
        cand[n_above + before] = cand_entry(kc, c);
      }
      taken += tile;
      __syncthreads();                                                  // s_warp_eq is rewritten by the next tile
    }
    unsigned P = 1;
    while (P < count) P <<= 1;
    KTF_SEL_CHECK(count <= (unsigned)k && P <= KTF_PLDA_TOPK_LARGE_MAX);
    for (unsigned i = count + tid; i < P; i += kSelThreads) cand[i] = 0ull;
    __syncthreads();
    for (unsigned size = 2; size <= P; size <<= 1)
      for (unsigned stride = size >> 1; stride > 0; stride >>= 1) {
        for (unsigned i = tid; i < P / 2; i += kSelThreads) {
          const unsigned lo = 2 * i - (i & (stride - 1)), hi = lo + stride;
          KTF_SEL_CHECK(hi < P);
          const unsigned long long a = cand[lo], b = cand[hi];
          if ((a < b) == ((lo & size) == 0)) {                          // descending where lo & size == 0
            cand[lo] = b;
            cand[hi] = a;
          }
        }
        __syncthreads();
      }
    for (int i = tid; i < k; i += kSelThreads) {
      float s = -INFINITY;
      long long idx = -1;
      if ((unsigned)i < count) {
        const unsigned long long e = cand[i];
        KTF_SEL_CHECK(e != 0ull && (long long)(0xffffffffu - (unsigned)e) < n);
        s = key_value((unsigned)(e >> 32));
        idx = rows.index(row, (long long)(0xffffffffu - (unsigned)e));
      }
      s_out[row * k + i] = s;
      i_out[row * k + i] = idx;
    }
    __syncthreads();                                                    // cand / keys are rewritten by the next row
  }
}

template <typename Rows>
int topk_select(const Rows& rows, long long n_rows, long long n, int k, float* s_out, long long* i_out, cudaStream_t st) {
  if (n_rows <= 0) return KTF_OK;
  const int in_smem = n <= kSelSmemRowMax;
  const size_t smem = (size_t)(kSelBins + (in_smem ? n : 0)) * sizeof(unsigned);
  static unsigned long long attr_done = 0;
  if (ktf::first_use_on_device(&attr_done))
    KTF_CUDA(cudaFuncSetAttribute(topk_select_kernel<Rows>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)((kSelBins + kSelSmemRowMax) * sizeof(unsigned))));
  topk_select_kernel<Rows><<<(unsigned)std::min<long long>(n_rows, 1LL << 20), kSelThreads, smem, st>>>(
      rows, n_rows, n, k, in_smem, s_out, i_out);
  KTF_LAUNCH_OK();
  return KTF_OK;
}

// What a tensor-core score call writes: the score matrix (row pitch ld, fp32 or bf16), the best column of every test
// row (top-1), or its k best columns (1 <= k <= KTF_PLDA_TOPK_LARGE_MAX) as (nt, k) scores and indexes, best first.
struct ScoreOut {
  enum Kind { kMatrix, kTop1, kTopk } kind;
  void* scores;
  long long* index;
  int64_t ld;
  int bf16;
  int k;
};

// The raw scores of test rows ut against enrolled columns ue, or (norm != nullptr) their AS-norm scores, as `out` asks:
// - the matrix: one GEMM;
// - top-1: the GEMM keeps a best-entry key per row (row_best), plda_top1_decode_kernel decodes the keys;
// - k <= KTF_PLDA_TOPK_MAX: the GEMM's top-k epilogue leaves partial lists (one per n-range and column quarter of a row)
//   in the workspace, topk_merge reduces them to (nt, k);
// - larger k: the GEMM writes the scores in row chunks of at most kTopkChunkBytes into the workspace -- the epilogue of
//   the matrix, so the values are bit-equal -- and topk_select selects every chunk while it is still in L2.
int score_tc(const ktf_plda* p, const float* ut, int64_t nt, const float* ue, int64_t ne, const AsnormStats* norm,
             const ScoreOut& out, cudaStream_t st) {
  const int k = out.k;
  float* score = static_cast<float*>(out.scores);
  const bool top_small = out.kind == ScoreOut::kTopk && k <= KTF_PLDA_TOPK_MAX;
  const bool top_large = out.kind == ScoreOut::kTopk && k > KTF_PLDA_TOPK_MAX;
  int lists = 0;
  long long ld = 0, chunk = 0;
  size_t extra = 0, s_bytes = 0;
  if (out.kind == ScoreOut::kTop1) extra = (size_t)nt * sizeof(unsigned long long);
  if (top_small) {
    lists = ktf::tc_topk_lists(nt, ne, 3LL * p->dim);
    if (lists == 0) return topk_merge(nullptr, nullptr, 0, nt, k, k, score, out.index, st);   // no enrolled vector
    const size_t n_part = (size_t)lists * nt * k;
    s_bytes = (n_part * sizeof(float) + 255) & ~(size_t)255;
    extra = s_bytes + n_part * sizeof(long long);
  }
  if (top_large) {
    if (ne == 0) return topk_select(MatrixRows{nullptr, 0}, nt, 0, k, score, out.index, st);   // padding only
    ld = (ne + 3) / 4 * 4;          // 16-byte row pitch: the GEMM's boxed stores
    chunk = chunk_rows(ld, nt, kTopkChunkBytes);
    extra = (size_t)chunk * ld * sizeof(float);
  }
  TcOperands o;
  int rc = tc_operands(p, ut, nt, ue, ne, norm, extra, st, &o);
  if (rc != KTF_OK) return rc;
  if (out.kind == ScoreOut::kMatrix)
    return ktf::tc_gemm_score(o.gemm(0, nt, ne, o.row, o.Bj, out.scores, out.ld, out.bf16), st);
  if (out.kind == ScoreOut::kTop1) {
    unsigned long long* keys = reinterpret_cast<unsigned long long*>(o.extra);
    KTF_CUDA(cudaMemsetAsync(keys, 0, (size_t)nt * sizeof(unsigned long long), st));
    ktf::TcScore g = o.gemm(0, nt, ne, o.row, o.Bj, nullptr, ne);
    g.row_best = keys;
    if ((rc = ktf::tc_gemm_score(g, st)) != KTF_OK) return rc;
    plda_top1_decode_kernel<<<(unsigned)((nt + 255) / 256), 256, 0, st>>>(keys, nt, score, out.index);
    KTF_LAUNCH_OK();
    return KTF_OK;
  }
  if (top_small) {
    float* part_s = reinterpret_cast<float*>(o.extra);
    long long* part_i = reinterpret_cast<long long*>(o.extra + s_bytes);
    ktf::TcScore g = o.gemm(0, nt, ne, o.row, o.Bj, nullptr, 0);
    g.k = k;
    g.part_score = part_s;
    g.part_index = part_i;
    if ((rc = ktf::tc_gemm_score(g, st)) != KTF_OK) return rc;
    return topk_merge(part_s, part_i, lists, nt, k, k, score, out.index, st);
  }
  float* buf = reinterpret_cast<float*>(o.extra);
  for (long long r0 = 0; r0 < nt; r0 += chunk) {
    const long long rows = std::min(chunk, (long long)nt - r0);
    if ((rc = ktf::tc_gemm_score(o.gemm(r0, rows, ne, o.row, o.Bj, buf, ld), st)) != KTF_OK) return rc;
    if ((rc = topk_select(MatrixRows{buf, ld}, rows, ne, k, score + r0 * k, out.index + r0 * k, st)) != KTF_OK) return rc;
  }
  return KTF_OK;
}

// Row i of a within-group score: the group g with offs[g] <= i < offs[g + 1] (offs relative to the first row; the last
// such g skips empty groups), its columns and the packed position of entry (i, 0): base[g] + (i - offs[g]) n_g - offs[g],
// so entry (i, j) lands at base[g] + (i - offs[g]) n_g + (j - offs[g]).
__global__ void within_rows_kernel(const long long* __restrict__ offs, const long long* __restrict__ base, int num_groups,
                                   long long n, ktf::WithinRow* __restrict__ rows) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= n) return;
  int lo = 0, hi = num_groups - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (offs[mid] <= i) lo = mid;
    else hi = mid - 1;
  }
  const long long c0 = offs[lo], c1 = offs[lo + 1];
  rows[i] = ktf::WithinRow{base[lo] + (i - c0) * (c1 - c0) - c0, (int)c0, (int)c1};
}

// Within-group scores of the rows u (offsets relative to offsets[0]) in one pair-kernel launch: the GEMM's rows are the
// enrolled side and its columns the test side (tc_operands' enrolled_rows), so row i of the accumulator is column i of
// the normal one and (acc + B_i) + A_j keeps the association of the normal epilogue (acc + B_i) + A_j: every entry is
// bit-equal to logLikelihoodRatio(u_g, u_g)[j, i].  The group table and the tile list are copied into the workspace with
// one cudaMemcpyAsync from pageable memory, which returns once the host buffer has been staged (no device
// synchronisation), so `host` may die at return.
int score_within_tc(const ktf_plda* p, const float* u, const int64_t* offsets, int num_groups, float* scores,
                    cudaStream_t st) {
  const long long n = offsets[num_groups] - offsets[0];
  const long long num_tiles = ktf::tc_within_tiles(offsets, num_groups, nullptr);
  // host: offsets (G + 1), packed bases (G), then the tiles
  std::vector<long long> host((size_t)(2 * num_groups + 1) + (size_t)num_tiles);
  long long acc = 0;
  for (int g = 0; g <= num_groups; ++g) host[g] = offsets[g] - offsets[0];
  for (int g = 0; g < num_groups; ++g) {
    host[num_groups + 1 + g] = acc;
    acc += (offsets[g + 1] - offsets[g]) * (offsets[g + 1] - offsets[g]);
  }
  int2* tiles_host = reinterpret_cast<int2*>(host.data() + 2 * num_groups + 1);
  ktf::tc_within_tiles(offsets, num_groups, tiles_host);
  const size_t table_bytes = host.size() * sizeof(long long);
  const size_t rows_at = (table_bytes + 255) & ~(size_t)255;
  TcOperands o;
  int rc = tc_operands(p, u, n, u, n, nullptr, rows_at + (size_t)n * sizeof(ktf::WithinRow), st, &o, /*enrolled_rows=*/true);
  if (rc != KTF_OK) return rc;
  long long* table = reinterpret_cast<long long*>(o.extra);
  ktf::WithinRow* rows = reinterpret_cast<ktf::WithinRow*>(o.extra + rows_at);
  KTF_CUDA(cudaMemcpyAsync(table, host.data(), table_bytes, cudaMemcpyHostToDevice, st));
  within_rows_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(table, table + num_groups + 1, num_groups, n, rows);
  KTF_LAUNCH_OK();
  const ktf::TcWithin w{reinterpret_cast<const int2*>(table + 2 * num_groups + 1), num_tiles, rows};
  ktf::TcScore g = o.gemm(0, n, n, o.Ai, o.Bj, scores, 0);
  g.within = &w;
  return ktf::tc_gemm_score(g, st);
}

// Argument checks of the k-best entry points `fn`, one order for all: k (1 .. k_max, named k_max_name), the handle,
// float32 / sm_100, n_enroll; n_test <= 0 is then a no-op, and the pointers are checked last.  Scores when they pass.
int score_topk_checked(const char* fn, int k_max, const char* k_max_name, const ktf_plda* p, const void* u_test,
                       int64_t n_test, const void* u_enroll, int64_t n_enroll, const AsnormStats* norm, int k,
                       float* scores, int64_t* index, void* stream) {
  KTF_CHECK_ARG(k >= 1 && k <= k_max, "%s: k = %d, must be 1 .. %d (%s)", fn, k, k_max, k_max_name);
  KTF_CHECK_ARG(p, "%s: null handle", fn);
  KTF_CHECK_ARG(p->use_tc, "%s needs a float32 PLDA handle on an sm_100 device", fn);
  KTF_CHECK_ARG(n_enroll >= 0 && n_enroll < (1LL << 32), "%s: n_enroll must be in 0 .. 2^32 - 1", fn);
  if (n_test <= 0) return KTF_OK;
  KTF_CHECK_ARG(u_test && scores && index && (n_enroll == 0 || u_enroll) &&
                    (norm == nullptr ||
                     (norm->t_mean && norm->t_std && (n_enroll == 0 || (norm->e_mean && norm->e_std)))),
                "%s: null argument", fn);
  return score_tc(p, (const float*)u_test, n_test, (const float*)u_enroll, n_enroll, norm,
                  ScoreOut{ScoreOut::kTopk, scores, (long long*)index, 0, 0, k}, (cudaStream_t)stream);
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
    return score_tc(p, (const float*)u_test_dev, n_test, (const float*)u_enroll_dev, n_enroll, nullptr,
                    ScoreOut{ScoreOut::kMatrix, scores_dev, nullptr, ld, 1, 0}, (cudaStream_t)stream);
  }
  return ktf_plda_score(p, u_test_dev, n_test, u_enroll_dev, n_enroll, scores_dev, ld, stream);
}

int ktf_plda_score_top1(const ktf_plda* p, const void* u_test_dev, int64_t n_test, const void* u_enroll_dev,
                        int64_t n_enroll, float* best_score_dev, int64_t* best_index_dev, void* stream) {
  KTF_CHECK_ARG(p && u_test_dev && u_enroll_dev && best_score_dev && best_index_dev, "ktf_plda_score_top1: null argument");
  KTF_CHECK_ARG(p->use_tc, "ktf_plda_score_top1 needs a float32 PLDA handle on an sm_100 device");
  KTF_CHECK_ARG(n_enroll < (1LL << 32), "ktf_plda_score_top1: more than 2^32 enrolled vectors");
  if (n_test <= 0) return KTF_OK;
  return score_tc(p, (const float*)u_test_dev, n_test, (const float*)u_enroll_dev, n_enroll, nullptr,
                  ScoreOut{ScoreOut::kTop1, best_score_dev, (long long*)best_index_dev, n_enroll, 0, 1},
                  (cudaStream_t)stream);
}

int ktf_plda_score_topk(const ktf_plda* p, const void* u_test_dev, int64_t n_test, const void* u_enroll_dev,
                        int64_t n_enroll, int32_t k, float* scores_dev, int64_t* index_dev, void* stream) {
  return score_topk_checked("ktf_plda_score_topk", KTF_PLDA_TOPK_MAX, "KTF_PLDA_TOPK_MAX", p, u_test_dev, n_test,
                            u_enroll_dev, n_enroll, nullptr, k, scores_dev, index_dev, stream);
}

int ktf_plda_cohort_stats(const ktf_plda* p, const void* u_dev, int64_t n, const void* u_cohort_dev, int64_t n_cohort,
                          int64_t top_n, int32_t role, float* mean_dev, float* std_dev, float* nth_dev, void* stream) {
  KTF_CHECK_ARG(p, "ktf_plda_cohort_stats: null handle");
  KTF_CHECK_ARG(role == KTF_COHORT_AS_TEST || role == KTF_COHORT_AS_ENROLLED,
                "ktf_plda_cohort_stats: role must be KTF_COHORT_AS_TEST or KTF_COHORT_AS_ENROLLED");
  KTF_CHECK_ARG(p->use_tc, "ktf_plda_cohort_stats needs a float32 PLDA handle on an sm_100 device");
  KTF_CHECK_ARG(top_n >= 2 && top_n <= n_cohort && n_cohort < (1LL << 32),
                "ktf_plda_cohort_stats: top_n = %lld, n_cohort = %lld: needs 2 <= top_n <= n_cohort < 2^32",
                (long long)top_n, (long long)n_cohort);
  if (n <= 0) return KTF_OK;
  KTF_CHECK_ARG(u_dev && u_cohort_dev && mean_dev && std_dev, "ktf_plda_cohort_stats: null argument");
  return cohort_stats_tc(p, (const float*)u_dev, n, (const float*)u_cohort_dev, n_cohort, top_n,
                         role == KTF_COHORT_AS_ENROLLED, mean_dev, std_dev, nth_dev, (cudaStream_t)stream);
}

int ktf_plda_score_asnorm(const ktf_plda* p, const void* u_test_dev, int64_t n_test, const void* u_enroll_dev,
                          int64_t n_enroll, const float* test_mean_dev, const float* test_std_dev,
                          const float* enroll_mean_dev, const float* enroll_std_dev, float* scores_dev, int64_t ld,
                          void* stream) {
  return ktf_plda_score_asnorm_ex(p, u_test_dev, n_test, u_enroll_dev, n_enroll, test_mean_dev, test_std_dev,
                                  enroll_mean_dev, enroll_std_dev, scores_dev, ld, KTF_SCORES_NATIVE, stream);
}

int ktf_plda_score_asnorm_ex(const ktf_plda* p, const void* u_test_dev, int64_t n_test, const void* u_enroll_dev,
                             int64_t n_enroll, const float* test_mean_dev, const float* test_std_dev,
                             const float* enroll_mean_dev, const float* enroll_std_dev, void* scores_dev, int64_t ld,
                             int32_t score_format, void* stream) {
  KTF_CHECK_ARG(score_format == KTF_SCORES_NATIVE || score_format == KTF_SCORES_BF16,
                "ktf_plda_score_asnorm: bad score_format %d", score_format);
  KTF_CHECK_ARG(p, "ktf_plda_score_asnorm: null handle");
  KTF_CHECK_ARG(p->use_tc, "ktf_plda_score_asnorm needs a float32 PLDA handle on an sm_100 device");
  KTF_CHECK_ARG(ld >= n_enroll, "ld must be >= n_enroll");
  if (n_test <= 0 || n_enroll <= 0) return KTF_OK;
  KTF_CHECK_ARG(u_test_dev && u_enroll_dev && test_mean_dev && test_std_dev && enroll_mean_dev && enroll_std_dev &&
                    scores_dev,
                "ktf_plda_score_asnorm: null argument");
  const AsnormStats s{test_mean_dev, test_std_dev, enroll_mean_dev, enroll_std_dev};
  return score_tc(p, (const float*)u_test_dev, n_test, (const float*)u_enroll_dev, n_enroll, &s,
                  ScoreOut{ScoreOut::kMatrix, scores_dev, nullptr, ld, score_format == KTF_SCORES_BF16 ? 1 : 0, 0},
                  (cudaStream_t)stream);
}

int ktf_plda_score_asnorm_topk(const ktf_plda* p, const void* u_test_dev, int64_t n_test, const void* u_enroll_dev,
                               int64_t n_enroll, const float* test_mean_dev, const float* test_std_dev,
                               const float* enroll_mean_dev, const float* enroll_std_dev, int32_t k, float* scores_dev,
                               int64_t* index_dev, void* stream) {
  const AsnormStats s{test_mean_dev, test_std_dev, enroll_mean_dev, enroll_std_dev};
  return score_topk_checked("ktf_plda_score_asnorm_topk", KTF_PLDA_TOPK_MAX, "KTF_PLDA_TOPK_MAX", p, u_test_dev, n_test,
                            u_enroll_dev, n_enroll, &s, k, scores_dev, index_dev, stream);
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

int ktf_plda_score_topk_large(const ktf_plda* p, const void* u_test_dev, int64_t n_test, const void* u_enroll_dev,
                              int64_t n_enroll, int32_t k, float* scores_dev, int64_t* index_dev, void* stream) {
  return score_topk_checked("ktf_plda_score_topk_large", KTF_PLDA_TOPK_LARGE_MAX, "KTF_PLDA_TOPK_LARGE_MAX", p,
                            u_test_dev, n_test, u_enroll_dev, n_enroll, nullptr, k, scores_dev, index_dev, stream);
}

int ktf_plda_score_asnorm_topk_large(const ktf_plda* p, const void* u_test_dev, int64_t n_test,
                                     const void* u_enroll_dev, int64_t n_enroll, const float* test_mean_dev,
                                     const float* test_std_dev, const float* enroll_mean_dev,
                                     const float* enroll_std_dev, int32_t k, float* scores_dev, int64_t* index_dev,
                                     void* stream) {
  const AsnormStats s{test_mean_dev, test_std_dev, enroll_mean_dev, enroll_std_dev};
  return score_topk_checked("ktf_plda_score_asnorm_topk_large", KTF_PLDA_TOPK_LARGE_MAX, "KTF_PLDA_TOPK_LARGE_MAX", p,
                            u_test_dev, n_test, u_enroll_dev, n_enroll, &s, k, scores_dev, index_dev, stream);
}

int ktf_topk_merge_large(const float* scores_in_dev, const int64_t* index_in_dev, int32_t num_lists, int64_t n_rows,
                         int32_t k_in, int32_t k, float* scores_dev, int64_t* index_dev, void* stream) {
  KTF_CHECK_ARG(k >= 1 && k <= KTF_PLDA_TOPK_LARGE_MAX,
                "ktf_topk_merge_large: k = %d, must be 1 .. %d (KTF_PLDA_TOPK_LARGE_MAX)", k, KTF_PLDA_TOPK_LARGE_MAX);
  KTF_CHECK_ARG(num_lists >= 0 && k_in >= 1 && (long long)num_lists * k_in < (1LL << 31),
                "ktf_topk_merge_large: bad num_lists / k_in");
  if (n_rows <= 0) return KTF_OK;
  KTF_CHECK_ARG(scores_dev && index_dev && (num_lists == 0 || (scores_in_dev && index_in_dev)),
                "ktf_topk_merge_large: null argument");
  return topk_select(ListRows{scores_in_dev, (const long long*)index_in_dev, n_rows, k_in}, n_rows,
                     (long long)num_lists * k_in, k, scores_dev, (long long*)index_dev, (cudaStream_t)stream);
}

int ktf_plda_score_within(const ktf_plda* p, const void* u_dev, const int64_t* offsets_host, int32_t num_groups,
                          float* scores_dev, void* stream) {
  KTF_CHECK_ARG(p, "ktf_plda_score_within: null handle");
  KTF_CHECK_ARG(p->use_tc, "ktf_plda_score_within needs a float32 PLDA handle on an sm_100 device");
  KTF_CHECK_ARG(num_groups >= 0, "ktf_plda_score_within: num_groups = %d, must be >= 0", num_groups);
  if (num_groups == 0) return KTF_OK;
  KTF_CHECK_ARG(offsets_host, "ktf_plda_score_within: null offsets");
  KTF_CHECK_ARG(offsets_host[0] >= 0, "ktf_plda_score_within: offsets[0] = %lld, must be >= 0",
                (long long)offsets_host[0]);
  for (int32_t g = 0; g < num_groups; ++g)
    KTF_CHECK_ARG(offsets_host[g + 1] >= offsets_host[g], "ktf_plda_score_within: group %d has a negative length", g);
  KTF_CHECK_ARG(offsets_host[num_groups] - offsets_host[0] < (1LL << 31),
                "ktf_plda_score_within: more than 2^31 - 1 rows");
  if (offsets_host[num_groups] == offsets_host[0]) return KTF_OK;
  KTF_CHECK_ARG(u_dev && scores_dev, "ktf_plda_score_within: null argument");
  return score_within_tc(p, (const float*)u_dev + offsets_host[0] * p->dim, offsets_host, num_groups, scores_dev,
                         (cudaStream_t)stream);
}

int ktf_plda_score(const ktf_plda* p, const void* u_test_dev, int64_t n_test, const void* u_enroll_dev,
                   int64_t n_enroll, void* scores_dev, int64_t ld, void* stream) {
  KTF_CHECK_ARG(p && u_test_dev && u_enroll_dev && scores_dev, "ktf_plda_score: null argument");
  KTF_CHECK_ARG(ld >= n_enroll, "ld must be >= n_enroll");
  if (n_test <= 0 || n_enroll <= 0) return KTF_OK;
  cudaStream_t st = (cudaStream_t)stream;
  if (p->use_tc)
    return score_tc(p, (const float*)u_test_dev, n_test, (const float*)u_enroll_dev, n_enroll, nullptr,
                    ScoreOut{ScoreOut::kMatrix, scores_dev, nullptr, ld, 0, 0}, st);
  return p->dtype_bytes == 4
             ? score_impl<float>(p, (const float*)u_test_dev, n_test, (const float*)u_enroll_dev, n_enroll,
                                 (float*)scores_dev, ld, st)
             : score_impl<double>(p, (const double*)u_test_dev, n_test, (const double*)u_enroll_dev,
                                  n_enroll, (double*)scores_dev, ld, st);
}

}  // extern "C"

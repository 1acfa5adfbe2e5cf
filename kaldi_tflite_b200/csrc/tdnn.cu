// TDNN affine layer (frame splice with edge clamp + contraction + bias + ReLU + BatchNorm),
// statistics pooling and the LDA / length-norm back-end.
//
// Replaces (file:line under /root/reference/kaldi_tflite/lib/):
//   layers/tdnn/tdnn.py:224-280 (+ utils.py:22-28 weight layout), keras ReLU
//   (models/kaldi/sequential.py:71-72), layers/normalization/batchnorm.py:81-88,
//   layers/stats/stats_pooling.py:179-316, models/kaldi/xvector_extractor.py:174-181.
//
// Two contraction engines sit behind ktf_affine_forward:
//   KTF_PREC_F32  -- exact fp32 SIMT tiles (this file), the precision reference;
//   KTF_PREC_BF16 -- tcgen05/TMEM implicit GEMM (tdnn_tc.cu), the throughput path.
#include <algorithm>
#include <vector>

#include "common.cuh"
#include "gemm_simt.cuh"
#include "tdnn_internal.cuh"

namespace {

struct RowInfo {
  long long in_base;  // first input row of the utterance
  int t_in;           // input time step the output row is centred on
  int T;              // utterance length (input rows)
};

__global__ void row_info_kernel(const long long* __restrict__ in_offs, const long long* __restrict__ out_offs,
                                long long batch, long long total_out, int start, int sub,
                                RowInfo* __restrict__ info, int* __restrict__ row_utt) {
  for (long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x; r < total_out;
       r += (long long)gridDim.x * blockDim.x) {
    long long lo = 0, hi = batch;
    while (hi - lo > 1) {
      const long long mid = (lo + hi) >> 1;
      if (out_offs[mid] <= r) lo = mid; else hi = mid;
    }
    RowInfo ri;
    ri.in_base = in_offs[lo];
    ri.T = (int)(in_offs[lo + 1] - in_offs[lo]);
    ri.t_in = start + (int)(r - out_offs[lo]) * sub;
    info[r] = ri;
    if (row_utt) row_utt[r] = (int)lo;
  }
}

struct SpliceLoad {  // tdnn.py:244-247, 258: gather with edge clamp (SAME) or plain shift (VALID)
  const float* x;
  const RowInfo* info;
  int D;
  int ctx[KTF_MAX_CONTEXT];
  __device__ __forceinline__ float operator()(long long row, int k) const {
    const RowInfo ri = info[row];
    const int kc = k / D, d = k - kc * D;
    int t = ri.t_in + ctx[kc];
    t = max(min(t, ri.T - 1), 0);      // rows past the last utterance (upper-bound row counts) stay in range
    return x[(ri.in_base + t) * D + d];
  }
};

struct AffineEpi {  // tdnn.py:275 bias, ReLU, batchnorm.py:81-88 as scale/offset
  float* y;
  const float* bias;
  const float* scale;
  const float* offset;
  int U;
  int relu;
  __device__ __forceinline__ void operator()(long long row, long long col, float acc) const {
    float v = acc;
    if (bias) v += bias[col];
    if (relu) v = fmaxf(v, 0.0f);
    if (scale) v = fmaf(v, scale[col], offset[col]);
    y[row * U + col] = v;
  }
};

__global__ void relu_kernel(const float* __restrict__ x, long long n, float* __restrict__ y) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
       i += (long long)gridDim.x * blockDim.x)
    y[i] = fmaxf(x[i], 0.0f);
}

__global__ void scale_offset_kernel(const float* __restrict__ x, long long n, int dim,
                                    const float* __restrict__ scale, const float* __restrict__ offset,
                                    float* __restrict__ y) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
       i += (long long)gridDim.x * blockDim.x) {
    const int d = (int)(i % dim);
    y[i] = fmaf(x[i], scale[d], offset ? offset[d] : 0.0f);
  }
}

// grid (batch, ceil(dim/128)); thread = column; fp64 accumulation, fp32 sums out.
__global__ void stats_sum_kernel(const float* __restrict__ x, const long long* __restrict__ offs, int dim,
                                 int period, float* __restrict__ sums) {
  const int d = blockIdx.y * blockDim.x + threadIdx.x;
  if (d >= dim) return;
  const long long b = blockIdx.x;
  const long long r0 = offs[b], r1 = offs[b + 1];
  double s = 0.0, s2 = 0.0;
  for (long long r = r0; r < r1; r += period) {
    const double v = (double)x[r * dim + d];
    s += v;
    s2 += v * v;
  }
  sums[(b * 2 + 0) * dim + d] = (float)s;
  sums[(b * 2 + 1) * dim + d] = (float)s2;
}

__global__ void stats_finalize_kernel(const float* __restrict__ sums, const long long* __restrict__ offs,
                                      int dim, int include_std, float eps, int period,
                                      float* __restrict__ out) {
  const int d = blockIdx.y * blockDim.x + threadIdx.x;
  if (d >= dim) return;
  const long long b = blockIdx.x;
  const long long T = offs[b + 1] - offs[b];
  const float n = (float)((T + period - 1) / period);
  const float mean = sums[(b * 2 + 0) * dim + d] / n;            // stats_pooling.py:231
  const int od = include_std ? 2 * dim : dim;
  out[b * od + d] = mean;
  if (include_std) {
    const float var = sums[(b * 2 + 1) * dim + d] / n - __fmul_rn(mean, mean);  // :236-238
    out[b * od + dim + d] = sqrtf(fmaxf(var, 0.0f) + eps);
  }
}

// one thread per (b, eval step j, feature d)
__global__ void stats_windows_kernel(const float* __restrict__ x, long long batch, long long T, int dim,
                                     int left, int right_excl, int in_period, long long t_start,
                                     long long num_eval, int out_period, int repeat, int include_std,
                                     float eps, float* __restrict__ out) {
  const long long total = batch * num_eval * dim;
  const int od = include_std ? 2 * dim : dim;
  const long long T_out = num_eval * repeat;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const int d = (int)(idx % dim);
    const long long bj = idx / dim;
    const long long j = bj % num_eval, b = bj / num_eval;
    const long long t = t_start + j * out_period;
    float s = 0.0f, s2 = 0.0f, n = 0.0f;
    for (int o = left; o < right_excl; o += in_period) {     // stats_pooling.py:192-209
      const long long u = t + o;
      if (u >= 0 && u < T) {
        const float v = x[(b * T + u) * dim + d];
        s += v;
        s2 += __fmul_rn(v, v);
        n += 1.0f;
      }
    }
    const float mean = s / n;
    const float var = s2 / n - __fmul_rn(mean, mean);
    const float sd = sqrtf(fmaxf(var, 0.0f) + eps);
    for (int r = 0; r < repeat; ++r) {                        // tf.repeat for SAME (:305-310)
      float* o = out + (b * T_out + j * repeat + r) * od;
      o[d] = mean;
      if (include_std) o[dim + d] = sd;
    }
  }
}

// One CTA (256 threads) per x-vector: y = (x - mean) @ L^T + o, then y *= sqrt(out)/||y||.
__global__ void lda_kernel(const float* __restrict__ x, int in_dim, int out_dim,
                           const float* __restrict__ mean, const float* __restrict__ tr, int length_norm,
                           float* __restrict__ y) {
  extern __shared__ float sm[];
  float* xs = sm;             // in_dim
  float* ys = sm + in_dim;    // out_dim
  __shared__ float s_norm;
  const long long b = blockIdx.x;
  for (int i = threadIdx.x; i < in_dim; i += blockDim.x) xs[i] = x[b * in_dim + i] - (mean ? mean[i] : 0.0f);
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  const int ld = in_dim + 1;
  for (int u = warp; u < out_dim; u += nw) {
    const float* row = tr + (long long)u * ld;
    float acc = 0.0f;
    for (int i = lane; i < in_dim; i += 32) acc = fmaf(xs[i], row[i], acc);
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) ys[u] = acc + row[in_dim];
  }
  __syncthreads();
  if (warp == 0) {
    float ss = 0.0f;
    for (int u = lane; u < out_dim; u += 32) ss = fmaf(ys[u], ys[u], ss);
    for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
    if (lane == 0) s_norm = sqrtf(ss);
  }
  __syncthreads();
  float ratio = 1.0f;
  if (length_norm) ratio = s_norm / sqrtf((float)out_dim);   // xvector_extractor.py:178-181
  for (int u = threadIdx.x; u < out_dim; u += blockDim.x) y[b * out_dim + u] = ys[u] / ratio;
}

inline unsigned grid_for(long long n, int threads) {
  return (unsigned)std::min<long long>((n + threads - 1) / threads, (long long)ktf::num_sms() * 32);
}

}  // namespace

namespace ktf {
int stats_sums_f32(const float* y_dev, const int64_t* offsets_dev, int64_t batch, int dim, float* sums_dev,
                   cudaStream_t st) {
  dim3 g((unsigned)batch, (unsigned)((dim + 127) / 128));
  stats_sum_kernel<<<g, 128, 0, st>>>(y_dev, (const long long*)offsets_dev, dim, 1, sums_dev);
  KTF_LAUNCH_OK();
  return KTF_OK;
}
}  // namespace ktf

extern "C" {

int ktf_affine_create(const ktf_affine_cfg* cfg, const float* weights_host, const float* bias_host,
                      const float* bn_scale_host, const float* bn_offset_host, ktf_affine** out) {
  KTF_CHECK_ARG(cfg && weights_host && out, "ktf_affine_create: null argument");
  KTF_CHECK_ARG(cfg->in_dim > 0 && cfg->out_dim > 0, "in_dim and out_dim must be > 0");
  KTF_CHECK_ARG(cfg->num_context >= 1 && cfg->num_context <= KTF_MAX_CONTEXT,
                "num_context must be in [1, %d]", KTF_MAX_CONTEXT);
  KTF_CHECK_ARG(cfg->subsampling_factor > 0, "subsampling_factor should be > 0");
  KTF_CHECK_ARG((bn_scale_host == nullptr) == (bn_offset_host == nullptr),
                "bn_scale_host and bn_offset_host must be given together");
  KTF_CHECK_ARG(cfg->precision == KTF_PREC_F32 || cfg->precision == KTF_PREC_BF16, "bad precision");
  for (int k = 1; k < cfg->num_context; ++k)
    KTF_CHECK_ARG(cfg->context[k] >= cfg->context[k - 1], "context must be sorted");
  ktf_affine* a = new ktf_affine();
  a->cfg = *cfg;
  const size_t K = (size_t)cfg->num_context * cfg->in_dim, U = cfg->out_dim;
  int rc;
  auto fail = [&](int code) { ktf_affine_destroy(a); return code; };
  if ((rc = ktf::upload(&a->d_w, weights_host, U * K)) != KTF_OK) return fail(rc);
  if (bias_host && (rc = ktf::upload(&a->d_bias, bias_host, U)) != KTF_OK) return fail(rc);
  if (bn_scale_host) {
    if ((rc = ktf::upload(&a->d_scale, bn_scale_host, U)) != KTF_OK) return fail(rc);
    if ((rc = ktf::upload(&a->d_offset, bn_offset_host, U)) != KTF_OK) return fail(rc);
  }
  if (cfg->precision == KTF_PREC_BF16) {
    if ((rc = ktf::affine_tc_prepare(a, weights_host, bn_scale_host, bn_offset_host)) != KTF_OK) return fail(rc);
  }
  *out = a;
  return KTF_OK;
}

void ktf_affine_destroy(ktf_affine* a) {
  if (!a) return;
  ktf::affine_tc_release(a);
  cudaFree(a->d_w);
  cudaFree(a->d_bias);
  cudaFree(a->d_scale);
  cudaFree(a->d_offset);
  delete a;
}

int64_t ktf_affine_out_rows(const ktf_affine* a, int64_t T) {
  if (!a || T <= 0) return 0;
  const ktf_affine_cfg& c = a->cfg;
  int64_t start = 0, end = T;                                 // tdnn.py:224-234
  if (c.padding_valid) {
    if (c.context[0] < 0) start = -c.context[0];
    if (c.context[c.num_context - 1] > 0) end = T - c.context[c.num_context - 1];
  }
  if (end <= start) return 0;
  return (end - start + c.subsampling_factor - 1) / c.subsampling_factor;
}

int ktf_affine_forward(const ktf_affine* a, const float* x_dev, const int64_t* in_offsets_dev,
                       const int64_t* out_offsets_dev, int64_t batch, int64_t total_in_rows,
                       int64_t total_out_rows, float* y_dev, float* stats_dev, void* stream) {
  KTF_CHECK_ARG(a && x_dev && in_offsets_dev && out_offsets_dev, "ktf_affine_forward: null argument");
  KTF_CHECK_ARG(y_dev || stats_dev, "nothing to compute: y_dev and stats_dev are both NULL");
  (void)total_in_rows;
  if (batch <= 0 || total_out_rows <= 0) return KTF_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const ktf_affine_cfg& c = a->cfg;

  if (c.precision == KTF_PREC_BF16)
    return ktf::affine_tc_forward(a, x_dev, in_offsets_dev, out_offsets_dev, batch, total_in_rows,
                                  total_out_rows, y_dev, stats_dev, st);

  const int K = c.num_context * c.in_dim, U = c.out_dim;
  ktf::Scratch scratch(st);            // released on every exit path
  RowInfo* info = nullptr;
  KTF_CUDA(scratch.take(&info, total_out_rows * sizeof(RowInfo)));
  const int start = (c.padding_valid && c.context[0] < 0) ? -c.context[0] : 0;
  row_info_kernel<<<grid_for(total_out_rows, 256), 256, 0, st>>>(
      (const long long*)in_offsets_dev, (const long long*)out_offsets_dev, batch, total_out_rows, start,
      c.subsampling_factor, info, nullptr);
  KTF_LAUNCH_OK();

  float* y = y_dev;
  if (y == nullptr) KTF_CUDA(scratch.take(&y, (size_t)total_out_rows * U * sizeof(float)));

  SpliceLoad al;
  al.x = x_dev;
  al.info = info;
  al.D = c.in_dim;
  for (int k = 0; k < KTF_MAX_CONTEXT; ++k) al.ctx[k] = k < c.num_context ? c.context[k] : 0;
  ktf::DenseLoad<float> bl{a->d_w, (long long)K};
  AffineEpi epi{y, a->d_bias, a->d_scale, a->d_offset, U, c.activation == KTF_ACT_RELU};
  dim3 grid((unsigned)((total_out_rows + ktf::kTileM - 1) / ktf::kTileM),
            (unsigned)((U + ktf::kTileN - 1) / ktf::kTileN));
  ktf::gemm_nt_kernel<float><<<grid, ktf::kGemmThreads, 0, st>>>((long long)total_out_rows, (long long)U, K,
                                                                al, bl, epi);
  KTF_LAUNCH_OK();
  if (stats_dev) {
    dim3 g2((unsigned)batch, (unsigned)((U + 127) / 128));
    stats_sum_kernel<<<g2, 128, 0, st>>>(y, (const long long*)out_offsets_dev, U, 1, stats_dev);
    KTF_LAUNCH_OK();
  }
  return KTF_OK;
}

int ktf_relu_forward(const float* x_dev, int64_t n, float* y_dev, void* stream) {
  KTF_CHECK_ARG(x_dev && y_dev, "ktf_relu_forward: null argument");
  if (n <= 0) return KTF_OK;
  relu_kernel<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(x_dev, n, y_dev);
  KTF_LAUNCH_OK();
  return KTF_OK;
}

int ktf_scale_offset_forward(const float* x_dev, int64_t rows, int32_t dim, const float* scale_dev,
                             const float* offset_dev, float* y_dev, void* stream) {
  KTF_CHECK_ARG(x_dev && y_dev && scale_dev, "ktf_scale_offset_forward: null argument");
  const long long n = (long long)rows * dim;
  if (n <= 0) return KTF_OK;
  scale_offset_kernel<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(x_dev, n, dim, scale_dev,
                                                                         offset_dev, y_dev);
  KTF_LAUNCH_OK();
  return KTF_OK;
}

int ktf_stats_finalize(const float* sums_dev, const int64_t* offsets_dev, int64_t batch, int32_t dim,
                       int32_t include_std, float epsilon, int32_t input_period, float* out_dev,
                       void* stream) {
  KTF_CHECK_ARG(sums_dev && offsets_dev && out_dev, "ktf_stats_finalize: null argument");
  KTF_CHECK_ARG(input_period > 0, "'input_period' and 'output_period' must be > 0");
  if (batch <= 0) return KTF_OK;
  dim3 g((unsigned)batch, (unsigned)((dim + 127) / 128));
  stats_finalize_kernel<<<g, 128, 0, (cudaStream_t)stream>>>(sums_dev, (const long long*)offsets_dev, dim,
                                                             include_std, epsilon, input_period, out_dev);
  KTF_LAUNCH_OK();
  return KTF_OK;
}

int ktf_stats_reduce(const float* x_dev, const int64_t* offsets_dev, int64_t batch, int32_t dim,
                     int32_t input_period, int32_t include_std, float epsilon, float* out_dev,
                     void* stream) {
  KTF_CHECK_ARG(x_dev && offsets_dev && out_dev, "ktf_stats_reduce: null argument");
  KTF_CHECK_ARG(input_period > 0, "'input_period' and 'output_period' must be > 0");
  if (batch <= 0) return KTF_OK;
  cudaStream_t st = (cudaStream_t)stream;
  ktf::Scratch scratch(st);
  float* sums = nullptr;
  KTF_CUDA(scratch.take(&sums, (size_t)batch * 2 * dim * sizeof(float)));
  dim3 g((unsigned)batch, (unsigned)((dim + 127) / 128));
  stats_sum_kernel<<<g, 128, 0, st>>>(x_dev, (const long long*)offsets_dev, dim, input_period, sums);
  KTF_LAUNCH_OK();
  stats_finalize_kernel<<<g, 128, 0, st>>>(sums, (const long long*)offsets_dev, dim, include_std, epsilon,
                                           input_period, out_dev);
  KTF_LAUNCH_OK();
  return KTF_OK;
}

int ktf_stats_windows(const float* x_dev, int64_t batch, int64_t T, int32_t dim, int32_t left,
                      int32_t right_excl, int32_t input_period, int64_t t_start, int64_t num_eval,
                      int32_t output_period, int32_t repeat, int32_t include_std, float epsilon,
                      float* out_dev, void* stream) {
  KTF_CHECK_ARG(x_dev && out_dev, "ktf_stats_windows: null argument");
  KTF_CHECK_ARG(input_period > 0 && output_period > 0 && repeat > 0,
                "'input_period' and 'output_period' must be > 0");
  const long long total = (long long)batch * num_eval * dim;
  if (total <= 0) return KTF_OK;
  stats_windows_kernel<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(
      x_dev, batch, T, dim, left, right_excl, input_period, t_start, num_eval, output_period, repeat,
      include_std, epsilon, out_dev);
  KTF_LAUNCH_OK();
  return KTF_OK;
}

int ktf_lda_forward(const float* x_dev, int64_t batch, int32_t in_dim, int32_t out_dim,
                    const float* mean_dev, const float* transform_dev, int32_t length_norm,
                    float* y_dev, void* stream) {
  KTF_CHECK_ARG(x_dev && transform_dev && y_dev, "ktf_lda_forward: null argument");
  KTF_CHECK_ARG(in_dim > 0 && out_dim > 0, "bad dimensions");
  if (batch <= 0) return KTF_OK;
  const size_t smem = (size_t)(in_dim + out_dim) * sizeof(float);
  KTF_CHECK_ARG(smem <= 48 * 1024, "in_dim + out_dim too large for ktf_lda_forward");
  lda_kernel<<<(unsigned)batch, 256, smem, (cudaStream_t)stream>>>(x_dev, in_dim, out_dim, mean_dev,
                                                                   transform_dev, length_norm, y_dev);
  KTF_LAUNCH_OK();
  return KTF_OK;
}

}  // extern "C"

// Fused front-end for long frames: real FFT lengths N = 1024, 2048, 4096 (complex length C = N/2 = 512 .. 2048),
// i.e. 25 ms frames at 32 to 96 kHz and up to 85 ms at 48 kHz.  Same math and the same reference lines as
// frontend.cu (framing.py:243-265, windowing.py:180-209, filterbank.py:225-242, dct.py:175-176, mfcc.py:197-244),
// in one launch; frames, spectra and mel energies never touch HBM.
//
// Work decomposition:
//   * a warp owns a group of 4 consecutive frames of one utterance (decode_item), stages the group's sample span
//     (3*shift + width samples, float32 or int16 PCM) once in shared memory, and runs the 4 frames one after the other
//     with all 32 lanes (the 8-lanes-per-frame geometry of frontend.cu would need 64..256 complex values per lane).
//   * windowing writes the frame as C complex pairs (x[2n], x[2n+1]) into the warp's tile; pre-emphasis takes the
//     neighbouring sample from a shuffle.
//   * the C-point complex FFT runs as in-place radix-P decimation-in-frequency passes over the tile, P <= 32 values
//     per lane in registers (compile-time inner twiddles, one table twiddle per output):
//       C =  512: 16 x 8 x 4      C = 1024: 32 x 32      C = 2048: 32 x 8 x 8
//     Every pass is a group of consecutive radix-2 DIF stages, so the result is in bit-reversed order whatever the
//     radices.  The tile is padded by one complex value per 16, which keeps the strided accesses of the passes and
//     of the bit-reversed reads mostly free of bank conflicts.
//   * real-FFT untangling pairs bins k and C - k (lane k = lane + 32 t); the powers are parked in registers until every
//     lane has read the tile, then written over it as the power spectrum.
//   * mel bank: every filter is cut into units of at most kUnitChunks 4-bin chunks, units are dealt to the 32 lanes
//     longest-first (the balancing of frontend_r16.cu), partial sums land in fixed slots and each filter adds its own
//     slots in a fixed order -- so the result does not depend on the batch and is reproducible bit for bit.
//   * log, DCT (lane c = coefficient c), lifter, C0 <- log-energy; each frame's row is stored directly (coalesced).
// All synchronisation inside the item loop is __syncwarp; CTAs only share the constant tables.
#include <math.h>

#include <algorithm>
#include <numeric>
#include <vector>

#include "frontend_internal.cuh"

using namespace ktf_fe;
using namespace ktf_fe::radix2;

namespace {

constexpr int kWideMaxWarps = 4;
constexpr int kUnitChunks = 8;   // 4-bin chunks per mel unit (a filter at 48 kHz / 80 mels spans up to ~40 chunks)
constexpr int kSmemLimit = 227 * 1024;

// tile index (complex units) of element n: one complex value of padding after every 16
__device__ __forceinline__ int pidx(int n) { return n + (n >> 4); }
__host__ __device__ constexpr int tile_floats(int C) { return 2 * (C + C / 16); }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// W_C^e for 0 <= e < C from the table tw[t] = W_{2C}^t, t < C
template <int C>
__device__ __forceinline__ float2 twc(const float2* tw, int e) {
  const int t = 2 * e;
  const float2 w = tw[t & (C - 1)];
  return (t & C) ? make_float2(-w.x, -w.y) : w;
}

// d * W_64^j (j a compile-time constant once the caller's loops are unrolled)
__device__ __forceinline__ float2 tw64(float2 d, int j) {
  j &= 63;
  const float c = 0.70710678118654752440f;
  if (j == 0) return d;
  if (j == 16) return make_float2(d.y, -d.x);                        // -i
  if (j == 32) return make_float2(-d.x, -d.y);
  if (j == 48) return make_float2(-d.y, d.x);                        // +i
  if (j == 8) return make_float2((d.x + d.y) * c, (d.y - d.x) * c);  // (1 - i)/sqrt2
  if (j == 24) return make_float2((d.y - d.x) * c, -(d.x + d.y) * c);
  const float wr = KTF_COS64[j], wi = -KTF_SIN64[j];
  return make_float2(fmaf(d.x, wr, -d.y * wi), fmaf(d.x, wi, d.y * wr));
}

// In-register DIF FFT of x[OFF .. OFF+N), N <= 64, output bit-reversed: the same result as fft_dif, computed with
// radix-4 butterflies (one radix-2 stage first when log2 N is odd).  A radix-4 stage rounds one twiddle product per
// output where two radix-2 stages round two, which keeps the float32 noise floor of the long transforms at or below
// that of a float32 library FFT.
template <int N, int OFF, int TOT>
__device__ __forceinline__ void fft_dif4(float2 (&x)[TOT]) {
  if constexpr (N == 2) {
    const float2 a = x[OFF], b = x[OFF + 1];
    x[OFF] = cadd(a, b);
    x[OFF + 1] = csub(a, b);
  } else if constexpr (N >= 4 && (ilog2(N) & 1)) {
    constexpr int H = N / 2;
#pragma unroll
    for (int i = 0; i < H; ++i) {
      const float2 a = x[OFF + i], b = x[OFF + i + H];
      x[OFF + i] = cadd(a, b);
      x[OFF + i + H] = tw64(csub(a, b), i * (64 / N));
    }
    fft_dif4<H, OFF, TOT>(x);
    fft_dif4<H, OFF + H, TOT>(x);
  } else if constexpr (N >= 4) {
    constexpr int Q = N / 4;
#pragma unroll
    for (int i = 0; i < Q; ++i) {
      const float2 a0 = x[OFF + i], a1 = x[OFF + i + Q], a2 = x[OFF + i + 2 * Q], a3 = x[OFF + i + 3 * Q];
      const float2 b0 = cadd(a0, a2), b1 = csub(a0, a2), b2 = cadd(a1, a3), d = csub(a1, a3);
      const float2 b3 = make_float2(d.y, -d.x);                       // (a1 - a3) * -i
      x[OFF + i] = cadd(b0, b2);
      x[OFF + i + Q] = tw64(csub(b0, b2), 2 * i * (64 / N));
      x[OFF + i + 2 * Q] = tw64(cadd(b1, b3), i * (64 / N));
      x[OFF + i + 3 * Q] = tw64(csub(b1, b3), 3 * i * (64 / N));
    }
    fft_dif4<Q, OFF, TOT>(x);
    fft_dif4<Q, OFF + Q, TOT>(x);
    fft_dif4<Q, OFF + 2 * Q, TOT>(x);
    fft_dif4<Q, OFF + 3 * Q, TOT>(x);
  }
}

// One in-place radix-P DIF pass over blocks of LB elements: log2(P) consecutive radix-2 stages at once.
// Group g = (block, i0) holds x[block*LB + i0 + m*LB/P], m < P; its P-point DFT bin k' (register brev(k')) is scaled by
// W_LB^(i0 k') and stored back to the slot of register index r.
template <int C, int P, int LB>
__device__ __forceinline__ void dif_pass(float2* tile, const float2* tw, int lane) {
  constexpr int S = LB / P;
  constexpr int G = C / P;
  constexpr int LOGP = ilog2(P);
  constexpr int LOGS = ilog2(S);
  constexpr int TWS = C / LB;
  static_assert(G % 32 == 0, "every lane owns the same number of groups");
#pragma unroll 1
  for (int t = 0; t < G / 32; ++t) {
    const int g = lane + 32 * t;
    const int i0 = g & (S - 1);
    const int base = (g >> LOGS) * LB + i0;
    float2 v[P];
#pragma unroll
    for (int m = 0; m < P; ++m) v[m] = tile[pidx(base + m * S)];
    fft_dif4<P, 0, P>(v);
#pragma unroll
    for (int r = 0; r < P; ++r) {
      const int kp = brev(r, LOGP);
      float2 y = v[r];
      if (S > 1 && kp != 0) y = cmul(y, twc<C>(tw, TWS * i0 * kp));
      tile[pidx(base + r * S)] = y;
    }
  }
  __syncwarp();
}

template <int C>
__device__ __forceinline__ void fft_passes(float2* tile, const float2* tw, int lane) {
  if constexpr (C == 512) {
    dif_pass<C, 16, 512>(tile, tw, lane);
    dif_pass<C, 8, 32>(tile, tw, lane);
    dif_pass<C, 4, 4>(tile, tw, lane);
  } else if constexpr (C == 1024) {
    dif_pass<C, 32, 1024>(tile, tw, lane);
    dif_pass<C, 32, 32>(tile, tw, lane);
  } else {
    static_assert(C == 2048, "complex FFT length 512, 1024 or 2048");
    dif_pass<C, 32, 2048>(tile, tw, lane);
    dif_pass<C, 8, 64>(tile, tw, lane);
    dif_pass<C, 8, 8>(tile, tw, lane);
  }
}

template <bool PCM16>
__device__ __forceinline__ float sample(const float* fr, const short* fr16, int i) {
  if constexpr (PCM16) return (float)fr16[i];
  else return fr[i];
}

template <int C, bool PCM16>
__global__ void __launch_bounds__(kWideMaxWarps * 32, 3) frontend_wide_kernel(const FrontendArgs a) {
  constexpr int L = ilog2(C);
  constexpr int NT = C / 32;   // complex pairs per lane in the windowing loops
  constexpr int NP = C / 64;   // (k, C - k) pairs per lane in the untangling
  extern __shared__ __align__(16) float smem[];
  const int nwarps = blockDim.x >> 5;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  // ---- CTA-shared tables (one blob) --------------------------------------------------------------
  const float* s_window = smem;
  const float2* s_tw = reinterpret_cast<const float2*>(smem + a.wide_off_tw);
  const int* s_ustart = reinterpret_cast<const int*>(smem + a.wide_off_ustart);
  const int4* s_units = reinterpret_cast<const int4*>(smem + a.wide_off_units);
  const int2* s_fslot = reinterpret_cast<const int2*>(smem + a.wide_off_fslot);
  const float* s_melw = smem + a.wide_off_melw;
  const float* s_dct = smem + a.wide_off_dct;
  const float* s_lifter = smem + a.wide_off_lifter;
  // ---- per-warp regions ----------------------------------------------------------------------------
  const int span_p = (a.span + 3) & ~3;
  float* s_span = smem + a.wide_blob_floats + warp * a.wide_warp_floats;
  float2* s_tile = reinterpret_cast<float2*>(s_span + span_p);
  float* s_Q = reinterpret_cast<float*>(s_tile);           // power spectrum, aliases the tile
  float* s_LM = s_span + span_p + tile_floats(C);          // log-mel row
  int* s_part = reinterpret_cast<int*>(s_LM + a.wide_lm_floats);   // mel unit partial sums (float64 as int pairs)

  const long long warp_stride = (long long)gridDim.x * nwarps;
  long long item = (long long)blockIdx.x * nwarps + warp;
  Item cur;
  if (item < a.total_groups) {             // start fetching the first span while the tables load
    cur = decode_item(a, item);
    if constexpr (PCM16) stage_span16(a, cur, reinterpret_cast<short*>(s_span), lane);
    else stage_span(a, cur, s_span, lane);
  }
  {
    const float4* src = reinterpret_cast<const float4*>(a.wide_blob);
    float4* dst = reinterpret_cast<float4*>(smem);
    for (int i = threadIdx.x; i < (a.wide_blob_floats >> 2); i += blockDim.x) dst[i] = src[i];
  }
  __syncthreads();

  const bool dithered = a.dither != 0.0f;
  const float pc = a.preemph > 0.0f ? a.preemph : 0.0f;
  const int W = a.W;

  for (; item < a.total_groups; item += warp_stride) {
    cp_async_wait_all();
    __syncwarp();
    const Item me = cur;

    for (int f = 0; f < me.nvalid; ++f) {
      const long long row = me.out_row0 + me.frame0 + f;   // global frame index: the dither counter
      const float* fr = s_span + f * a.shift;
      const short* fr16 = reinterpret_cast<const short*>(s_span) + f * a.shift;

      // ---- windowing (windowing.py:180-209), pass 1: samples (+ dither) into the tile, DC sum ----------
      float sum = 0.0f;
#pragma unroll 4
      for (int t = 0; t < NT; ++t) {
        const int n = lane + 32 * t, i0 = 2 * n;
        float x0 = 0.0f, x1 = 0.0f;
        if (i0 < W) {
          x0 = sample<PCM16>(fr, fr16, i0);
          if (i0 + 1 < W) x1 = sample<PCM16>(fr, fr16, i0 + 1);
          if (dithered) {                                        // windowing.py:182-183
            const float2 nz = dither_pair(a.dither_seed, row, n);
            x0 = fmaf(a.dither, nz.x, x0);
            if (i0 + 1 < W) x1 = fmaf(a.dither, nz.y, x1);
          }
        }
        s_tile[pidx(n)] = make_float2(x0, x1);
        sum += x0 + x1;
      }
      if (f == me.nvalid - 1) {          // the span is consumed: prefetch the next item's into the same buffer
        __syncwarp();
        const long long nxt = item + warp_stride;
        if (nxt < a.total_groups) {
          cur = decode_item(a, nxt);
          if constexpr (PCM16) stage_span16(a, cur, reinterpret_cast<short*>(s_span), lane);
          else stage_span(a, cur, s_span, lane);
        }
      }
      const float mean = a.remove_dc ? warp_sum(sum) / (float)W : 0.0f;

      // ---- pass 2 (own slots only): DC removal, energy, pre-emphasis, window --------------------------
      const bool windowed_out = a.output == KTF_OUT_WINDOWED;
      float* wdst = a.out + row * (long long)W;
      float esum = 0.0f, carry = 0.0f;   // carry: x[64 t - 1], lane 31's odd sample of the previous trip
#pragma unroll 4
      for (int t = 0; t < NT; ++t) {
        const int n = lane + 32 * t, i0 = 2 * n;
        const float2 v = s_tile[pidx(n)];
        float prev = __shfl_up_sync(0xffffffffu, v.y, 1);
        if (lane == 0) prev = carry;
        carry = __shfl_sync(0xffffffffu, v.y, 31);
        float y0 = 0.0f, y1 = 0.0f;
        if (i0 < W) {
          const bool has1 = i0 + 1 < W;
          const float x0 = v.x - mean;
          const float x1 = has1 ? v.y - mean : 0.0f;
          const float xm1 = i0 > 0 ? prev - mean : x0;
          if (a.raw_energy) esum = fmaf(x0, x0, fmaf(x1, x1, esum));
          y0 = (x0 - pc * xm1) * s_window[i0];
          y1 = has1 ? (x1 - pc * x0) * s_window[i0 + 1] : 0.0f;
          if (!a.raw_energy) esum = fmaf(y0, y0, fmaf(y1, y1, esum));
          if (windowed_out) {
            wdst[i0] = y0;
            if (has1) wdst[i0 + 1] = y1;
          }
        }
        s_tile[pidx(n)] = make_float2(y0, y1);
      }

      float log_e = 0.0f;
      if (a.use_energy) {
        esum = warp_sum(esum);
        log_e = logf(fmaxf(esum, 0.0f) + a.eps);
        log_e = fminf(fmaxf(log_e, a.energy_floor), 3.402823466e+38f);
      }
      __syncwarp();
      if (windowed_out) {
        if (a.use_energy && a.energy_out != nullptr && lane == 0) a.energy_out[row] = log_e;
        continue;
      }

      // ---- C-point complex FFT, bit-reversed result ---------------------------------------------------
      fft_passes<C>(s_tile, s_tw, lane);

      // ---- real-FFT untangling and |X|^2 (x4: the 1/4 is in the mel weights) ----------------------------
      float qa[NP], qb[NP];
#pragma unroll
      for (int t = 0; t < NP; ++t) {
        const int k = lane + 32 * t;
        const int kc = (C - k) & (C - 1);
        const float2 zk = s_tile[pidx((int)(__brev((unsigned)k) >> (32 - L)))];
        float2 zp = s_tile[pidx((int)(__brev((unsigned)kc) >> (32 - L)))];
        zp.y = -zp.y;
        const float2 w = s_tw[k];                              // W_N^k
        const float2 post = make_float2(w.y, -w.x);             // -i W_N^k
        const float2 S = cadd(zk, zp), D = csub(zk, zp);
        const float2 Gt = cmul(post, D);
        qa[t] = cnorm(cadd(S, Gt));                             // bin k
        qb[t] = cnorm(csub(S, Gt));                             // bin C - k (k = 0: the Nyquist bin C)
      }
      float qmid = 0.0f;                                        // bin C/2 pairs with itself: X = conj(Z[C/2])
      if (lane == 0) qmid = 4.0f * cnorm(s_tile[pidx(1)]);      // brev(C/2) == 1
      __syncwarp();   // tile fully consumed
#pragma unroll
      for (int t = 0; t < NP; ++t) {
        const int k = lane + 32 * t;
        float v1 = qa[t], v2 = qb[t];
        if (!a.use_power) { v1 = sqrtf(v1); v2 = sqrtf(v2); }
        s_Q[k] = v1;
        s_Q[C - k] = v2;
      }
      if (lane == 0) {
        s_Q[C / 2] = a.use_power ? qmid : sqrtf(qmid);
        s_Q[C + 1] = 0.0f;
        s_Q[C + 2] = 0.0f;
        s_Q[C + 3] = 0.0f;
      }
      __syncwarp();

      // ---- mel bank (filterbank.py:238-240): units -> slots, then each filter adds its slots ------------
      {
        const int u1 = s_ustart[lane + 1];
        for (int u = s_ustart[lane]; u < u1; ++u) {
          const int4 d = s_units[u];                            // (first chunk, #chunks, weight offset, slot)
          const float4* qv = reinterpret_cast<const float4*>(s_Q) + d.x;
          const float4* wv = reinterpret_cast<const float4*>(s_melw + d.z);
          double acc = 0.0;   // float64 sums: the mel and DCT stages add no rounding noise of their own (they cost
          for (int c = 0; c < d.y; ++c) {   // a few percent of the frame's time at these lengths)
            const float4 q = qv[c], w = wv[c];
            acc = fma((double)w.x, (double)q.x, acc);
            acc = fma((double)w.y, (double)q.y, acc);
            acc = fma((double)w.z, (double)q.z, acc);
            acc = fma((double)w.w, (double)q.w, acc);
          }
          s_part[2 * d.w] = __double2hiint(acc);
          s_part[2 * d.w + 1] = __double2loint(acc);
        }
      }
      __syncwarp();
      for (int i = lane; i < a.M; i += 32) {
        const int2 fs = s_fslot[i];
        double sum = 0.0;
        for (int p = 0; p < fs.y; ++p) sum += __hiloint2double(s_part[2 * (fs.x + p)], s_part[2 * (fs.x + p) + 1]);
        float acc = (float)sum;
        if (a.use_log) acc = __logf(fmaxf(acc, 0.0f) + a.eps);   // as frontend.cu
        if (a.output == KTF_OUT_FBANK) a.out[row * a.M + i] = acc;
        else s_LM[i] = acc;
      }

      if (a.output == KTF_OUT_MFCC) {
        __syncwarp();
        // ---- DCT (dct.py:176), lifter (mfcc.py:212), C0 <- energy (mfcc.py:219-228): lane c = coefficient c
        if (lane < a.Kc) {
          double sum = 0.0;
          for (int i = 0; i < a.M; ++i) sum = fma((double)s_LM[i], (double)s_dct[i * 32 + lane], sum);
          float acc = (float)sum;
          if (a.apply_lifter) acc *= s_lifter[lane];
          if (lane == 0 && a.use_energy) acc = log_e;
          a.out[row * a.Kc + lane] = acc;
        }
      }
      __syncwarp();   // the next frame overwrites the tile and the log-mel row
    }
  }
}

template <int C, bool PCM16>
int launch_wide(const ktf_frontend* fe, FrontendArgs& a, cudaStream_t st) {
  const int threads = fe->wide_warps * 32;
  const size_t smem = ((size_t)fe->wide_blob_floats + (size_t)fe->wide_warps * fe->wide_warp_floats) * sizeof(float);
  auto kern = frontend_wide_kernel<C, PCM16>;
  KTF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)std::max<size_t>(smem, 48 * 1024)));
  int occ = 0;
  KTF_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, threads, smem));
  if (occ < 1) occ = 1;
  const long long ctas_needed = (a.total_groups + fe->wide_warps - 1) / fe->wide_warps;
  const long long grid = std::min<long long>(ctas_needed, (long long)ktf::num_sms() * occ);
  if (grid <= 0) return KTF_OK;
  kern<<<(unsigned)grid, threads, smem, st>>>(a);
  KTF_LAUNCH_OK();
  return KTF_OK;
}

}  // namespace

namespace ktf_fe {

int wide_build(ktf_frontend* fe, const float* window_host, const float* mel_bank_host, const float* dct_host,
               const float* lifter_host) {
  const ktf_frontend_cfg& c = fe->cfg;
  const int W = c.frame_width, N = c.fft_length, C = N / 2;
  const bool need_mel = c.output != KTF_OUT_WINDOWED;
  const int M = need_mel ? c.num_mels : 0, Kc = c.num_ceps;

  // ---- mel filters -> units of <= kUnitChunks chunks, dealt to the 32 lanes longest-first --------------
  struct Unit { int filt, c0, n, slot; };
  std::vector<Unit> units;
  std::vector<int> fslot((size_t)2 * std::max(M, 1), 0);
  for (int i = 0; i < M; ++i) {
    int lo = -1, hi = -1;
    for (int k = 0; k <= C; ++k)
      if (mel_bank_host[(size_t)k * M + i] != 0.0f) { if (lo < 0) lo = k; hi = k; }
    fslot[2 * i] = (int)units.size();
    if (lo >= 0) {
      const int c0 = lo >> 2, n = (hi >> 2) - c0 + 1;
      for (int cc = 0; cc < n; cc += kUnitChunks)
        units.push_back({i, c0 + cc, std::min(kUnitChunks, n - cc), (int)units.size()});
    }
    fslot[2 * i + 1] = (int)units.size() - fslot[2 * i];
  }
  const int NU = (int)units.size();
  std::vector<int> order((size_t)NU);
  std::iota(order.begin(), order.end(), 0);
  std::stable_sort(order.begin(), order.end(), [&](int x, int y) { return units[x].n > units[y].n; });
  std::vector<std::vector<int>> lanes(32);
  int load[32] = {0};
  for (int u : order) {
    int best = 0;
    for (int l = 1; l < 32; ++l)
      if (load[l] < load[best]) best = l;
    lanes[best].push_back(u);
    load[best] += units[u].n;
  }

  // ---- blob layout -----------------------------------------------------------------------------------
  auto pad4 = [](int x) { return (x + 3) & ~3; };
  const int off_tw = pad4(W);
  const int off_ustart = off_tw + 2 * C;
  const int off_units = off_ustart + 36;
  const int off_fslot = off_units + 4 * NU;
  const int off_melw = off_fslot + pad4(2 * std::max(M, 1));
  int melw_floats = 0;
  for (const Unit& u : units) melw_floats += 4 * u.n;
  const int off_dct = off_melw + melw_floats;
  const int dct_floats = c.output == KTF_OUT_MFCC ? M * 32 : 0;
  const int off_lifter = off_dct + dct_floats;
  const int blob_floats = pad4(off_lifter + 32);
  std::vector<float> blob((size_t)blob_floats, 0.0f);

  for (int i = 0; i < W; ++i) blob[i] = window_host[i];
  const double PI = 3.14159265358979323846;
  for (int t = 0; t < C; ++t) {    // W_N^t
    const double th = -2.0 * PI * (double)t / (double)N;
    blob[off_tw + 2 * t] = (float)cos(th);
    blob[off_tw + 2 * t + 1] = (float)sin(th);
  }
  int* ustart = reinterpret_cast<int*>(blob.data() + off_ustart);
  int4* ud = reinterpret_cast<int4*>(blob.data() + off_units);
  float* mw = blob.data() + off_melw;
  const float scale = c.use_power ? 0.25f : 0.5f;   // the kernel stores 4|X|^2 (or 2|X|)
  std::vector<int> woff((size_t)NU, 0);
  {
    int w = 0;
    for (int u = 0; u < NU; ++u) {   // weights in slot (filter-major) order
      woff[u] = w;
      const Unit& un = units[u];
      for (int cc = 0; cc < un.n; ++cc)
        for (int b = 0; b < 4; ++b) {
          const int k = 4 * (un.c0 + cc) + b;
          mw[w++] = k <= C ? mel_bank_host[(size_t)k * M + un.filt] * scale : 0.0f;
        }
    }
  }
  int pos = 0;
  for (int l = 0; l < 32; ++l) {
    ustart[l] = pos;
    for (int u : lanes[l]) ud[pos++] = make_int4(units[u].c0, units[u].n, woff[u], units[u].slot);
  }
  ustart[32] = pos;
  int* fs = reinterpret_cast<int*>(blob.data() + off_fslot);
  for (int i = 0; i < 2 * M; ++i) fs[i] = fslot[i];
  if (c.output == KTF_OUT_MFCC) {
    float* dp = blob.data() + off_dct;
    for (int i = 0; i < M; ++i)
      for (int cc = 0; cc < Kc; ++cc) dp[(size_t)i * 32 + cc] = dct_host[(size_t)i * Kc + cc];
    float* lf = blob.data() + off_lifter;
    for (int cc = 0; cc < 32; ++cc) lf[cc] = (c.apply_lifter && cc < Kc) ? lifter_host[cc] : 1.0f;
  }

  // ---- CTA size: the most warps (<= 4) whose regions fit next to the tables --------------------------------
  const int span_p = pad4(fe->span);
  const int lm_floats = pad4(std::max(M, 1));
  const int warp_floats = span_p + tile_floats(C) + lm_floats + pad4(2 * std::max(NU, 1));
  int warps = kWideMaxWarps;
  while (warps > 1 && ((size_t)blob_floats + (size_t)warps * warp_floats) * sizeof(float) > (size_t)kSmemLimit) warps /= 2;
  const size_t bytes = ((size_t)blob_floats + (size_t)warps * warp_floats) * sizeof(float);
  if (bytes > (size_t)kSmemLimit) {
    ktf::set_error("front-end configuration (frame_width %d, frame_shift %d, fft_length %d) needs %zu bytes of shared "
                   "memory (> 227 KB)", W, c.frame_shift, N, bytes);
    return KTF_EINVAL;
  }
  fe->smem_bytes = bytes;
  fe->wide_warps = warps;
  fe->wide_blob_floats = blob_floats;
  fe->wide_warp_floats = warp_floats;
  fe->wide_lm_floats = lm_floats;
  fe->wide_off_tw = off_tw;
  fe->wide_off_ustart = off_ustart;
  fe->wide_off_units = off_units;
  fe->wide_off_fslot = off_fslot;
  fe->wide_off_melw = off_melw;
  fe->wide_off_dct = off_dct;
  fe->wide_off_lifter = off_lifter;
  return ktf::upload(&fe->d_wide, blob.data(), blob.size());
}

int wide_launch(const ktf_frontend* fe, FrontendArgs& a, cudaStream_t st) {
  a.wide_blob = fe->d_wide;
  a.wide_blob_floats = fe->wide_blob_floats;
  a.wide_warp_floats = fe->wide_warp_floats;
  a.wide_lm_floats = fe->wide_lm_floats;
  a.wide_off_tw = fe->wide_off_tw;
  a.wide_off_ustart = fe->wide_off_ustart;
  a.wide_off_units = fe->wide_off_units;
  a.wide_off_fslot = fe->wide_off_fslot;
  a.wide_off_melw = fe->wide_off_melw;
  a.wide_off_dct = fe->wide_off_dct;
  a.wide_off_lifter = fe->wide_off_lifter;
  const bool pcm = a.wav16 != nullptr;
  switch (fe->C) {
    case 512: return pcm ? launch_wide<512, true>(fe, a, st) : launch_wide<512, false>(fe, a, st);
    case 1024: return pcm ? launch_wide<1024, true>(fe, a, st) : launch_wide<1024, false>(fe, a, st);
    case 2048: return pcm ? launch_wide<2048, true>(fe, a, st) : launch_wide<2048, false>(fe, a, st);
    default: break;
  }
  ktf::set_error("wide front-end: unsupported complex FFT length %d", fe->C);
  return KTF_EINVAL;
}

}  // namespace ktf_fe

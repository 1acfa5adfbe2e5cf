// Fused Kaldi-compatible front-end for sm_100a:
//   framing -> DC removal -> log-energy -> pre-emphasis -> window -> zero-pad -> real FFT
//   -> power spectrum -> sparse mel filterbank -> log -> DCT-II -> lifter -> C0 <- energy
// in ONE kernel; frames, spectra and mel energies never touch HBM.
//
// Replaces (file:line under /root/reference/kaldi_tflite/lib/layers/dsp/):
//   framing.py:243-265, windowing.py:180-209, filterbank.py:225-242, dct.py:175-176,
//   mfcc.py:197-244.
//
// Work decomposition (HBM traffic = wav once + features once):
//   * a warp owns 4 consecutive frames of one utterance ("frame group"); 8 lanes per frame.
//   * the group's sample span (3*shift + width floats) is staged once in shared memory with
//     fully coalesced loads; the 2.5x frame overlap is served from there.
//   * real FFT of length NFFT = 2C as a C-point complex FFT, C = R x 8:
//       lane l holds z[l + 8m], m < R  -> R-point FFT in registers (compile-time twiddles)
//       -> twiddle W_C^(l*k1) -> 8xR transpose through a conflict-free smem tile
//       -> 8-point FFTs in registers.  The k1 columns a lane receives are closed under
//       k -> C-k, so the real-FFT untangling and |X|^2 need no further exchange.
//   * mel bank is applied in its sparse form: every FFT bin feeds <= 2 adjacent filters, so
//     bins are walked once with two running sums per "segment" (mel_i = U_i + D_{i-1}).
//   * log, DCT (30x30-ish, from smem), lifter, C0 <- log-energy, coalesced store.
// All synchronisation is __syncwarp; CTAs only share the constant tables.
#include <math.h>
#include <stdlib.h>

#include <algorithm>
#include <vector>

#include "common.cuh"

#include "frontend_internal.cuh"

using namespace ktf_fe;
using namespace ktf_fe::radix2;

namespace {

template <int R>
struct Geo {
  static constexpr int C = 8 * R;          // complex FFT length
  static constexpr int NSLOT = R / 8;      // k1 columns a lane owns after the transpose
  static constexpr int RS = R + 2;         // complex row stride of the transpose tile / twiddle table
  static constexpr int TFS = ((8 * RS * 2 + 31) / 32) * 32 + 16;  // floats per frame tile (== 16 mod 32)
  // floats per frame of the power buffer.  The chunk swizzle of qidx() sends the Nyquist chunk C/4 to C/4 ^ ((C/32) & 7):
  // itself for C = 256, but chunk 36 for C = 128 -- the 256-point FFT needs 16 more floats per frame (without them the
  // Nyquist power of frame f landed on bins 8..11 of frame f + 1)
  static constexpr int QS = C + (R == 16 ? 24 : 8);
};

// Power-buffer index of bin k: 4-bin chunks are XOR-swizzled so that the eight lanes of a frame,
// which read chunks of different filters with LDS.128, spread over all banks.
__device__ __forceinline__ int qidx(int k) {
  const int c = k >> 2;
  return ((c ^ ((c >> 3) & 7)) << 2) | (k & 3);
}
__device__ __forceinline__ int qchunk(int c) { return (c ^ ((c >> 3) & 7)) << 2; }

// R = complex FFT length / 8.  MV > 0: frame width is exactly 16*MV and frame_shift is even, so the
// windowing loop has compile-time bounds and 64-bit loads; MV == 0: any width <= 16R (runtime checks).
template <int R, int MV>
__global__ void __launch_bounds__(kThreads, 3) frontend_kernel(const FrontendArgs a) {
  using G = Geo<R>;
  constexpr int C = G::C;
  constexpr int NSLOT = G::NSLOT;
  constexpr int RS = G::RS;
  constexpr int LOGR = ilog2(R);

  extern __shared__ __align__(16) float smem[];
  // ---- CTA-shared tables -------------------------------------------------------------
  float* s_window = smem;                                        // W (padded to 4)
  const int Wp = (a.W + 3) & ~3;
  float2* s_tw = reinterpret_cast<float2*>(s_window + Wp);       // 8*RS complex
  int4* s_filt = reinterpret_cast<int4*>(s_tw + 8 * RS);         // M filters (padded to kMaxMels)
  float* s_melw = reinterpret_cast<float*>(s_filt + kMaxMels);   // mel_w_len (multiple of 4)
  float* s_dct = s_melw + a.mel_w_len;                           // M*32
  float* s_lifter = s_dct + a.M * 32;                            // 32
  float* s_warp0 = s_lifter + 32;
  // ---- per-warp regions ----------------------------------------------------------------
  const int span_p = (a.span + 3) & ~3;
  const int LMS = ((a.M + 3) & ~3) + 4;                          // log-mel row stride (== 4 mod 8)
  const int out_sz = 4 * ((a.out_dim + 3) & ~3);
  const int warp_floats = span_p + 4 * G::TFS + 4 * LMS + out_sz;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* s_span = s_warp0 + warp * warp_floats;
  float* s_T = s_span + span_p;            // transpose tile, later aliased by the power buffer
  float* s_LM = s_T + 4 * G::TFS;          // logmel[f][LMS]
  float* s_out = s_LM + 4 * LMS;           // out tile [f][out_dim]

  const long long warp_global = (long long)blockIdx.x * kWarpsPerCta + warp;
  const long long warp_stride = (long long)gridDim.x * kWarpsPerCta;

  Item cur;
  long long item = warp_global;
  if (item < a.total_groups) {             // start fetching the first span while the tables load
    cur = decode_item(a, item);
    stage_span(a, cur, s_span, lane);
  }

  for (int i = threadIdx.x; i < a.W; i += kThreads) s_window[i] = a.window[i];
  for (int i = threadIdx.x; i < 8 * RS; i += kThreads) s_tw[i] = a.stage_tw[i];
  if (a.output != KTF_OUT_WINDOWED) {
    for (int i = threadIdx.x; i < a.M; i += kThreads) s_filt[i] = a.mel_filt[i];
    for (int i = threadIdx.x; i < a.mel_w_len; i += kThreads) s_melw[i] = a.mel_w[i];
    if (a.output == KTF_OUT_MFCC) {
      for (int i = threadIdx.x; i < a.M * 32; i += kThreads) s_dct[i] = a.dct[i];
      for (int i = threadIdx.x; i < 32; i += kThreads) s_lifter[i] = a.lifter[i];
    }
  }
  __syncthreads();

  const int f = lane >> 3;  // frame within the group
  const int j = lane & 7;   // lane within the frame (FFT lane / mel group)
  const bool j0 = (j == 0);

  // k1 columns owned after the transpose, arranged as (a, b) pairs with a + b == R (mod R):
  //   lanes j >= 1: (j, R-j) [, (R/2-j, R/2+j)];  lane 0: (R/2, R/2) [, (R/4, 3R/4)] + column 0.
  int ka[NSLOT / 2], kb[NSLOT / 2];
  float2 base[NSLOT / 2];
  ka[0] = j0 ? R / 2 : j;
  kb[0] = j0 ? R / 2 : R - j;
  if constexpr (NSLOT == 4) {
    ka[1] = j0 ? R / 4 : R / 2 - j;
    kb[1] = j0 ? 3 * R / 4 : R / 2 + j;
  }
#pragma unroll
  for (int p = 0; p < NSLOT / 2; ++p) base[p] = a.post_tw[ka[p]];

  for (; item < a.total_groups; item += warp_stride) {
    cp_async_wait_all();
    __syncwarp();

    // ---- windowing (windowing.py:180-209) ------------------------------------------------
    const float* fr = s_span + f * a.shift;
    const bool fvalid = f < cur.nvalid;
    const bool dithered = a.dither != 0.0f;                       // warp-uniform
    const long long gframe = cur.out_row0 + cur.frame0 + f;      // global frame index: the dither counter
    float2 z[R];
    float sum = 0.0f;
    if constexpr (MV > 0) {
#pragma unroll
      for (int m = 0; m < R; ++m) {
        if (m < MV) {
          z[m] = *reinterpret_cast<const float2*>(fr + 2 * (j + 8 * m));
          if (dithered) {                                         // windowing.py:182-183
            const float2 nz = dither_pair(a.dither_seed, gframe, j + 8 * m);
            z[m].x = fmaf(a.dither, nz.x, z[m].x);
            z[m].y = fmaf(a.dither, nz.y, z[m].y);
          }
          sum += z[m].x + z[m].y;
        } else {
          z[m] = make_float2(0.0f, 0.0f);
        }
      }
    } else {
#pragma unroll
      for (int m = 0; m < R; ++m) {
        const int i0 = 2 * (j + 8 * m);
        float x0 = 0.0f, x1 = 0.0f;
        if (i0 < a.W) {
          x0 = fr[i0];
          if (i0 + 1 < a.W) x1 = fr[i0 + 1];
          if (dithered) {                                         // windowing.py:182-183
            const float2 nz = dither_pair(a.dither_seed, gframe, j + 8 * m);
            x0 = fmaf(a.dither, nz.x, x0);
            if (i0 + 1 < a.W) x1 = fmaf(a.dither, nz.y, x1);
          }
        }
        z[m] = make_float2(x0, x1);
        sum += x0 + x1;
      }
    }
    float mean = 0.0f;
    if (a.remove_dc) mean = group_sum8(sum) / (float)a.W;
    float esum = 0.0f;
    const float pc = a.preemph > 0.0f ? a.preemph : 0.0f;
    if constexpr (MV > 0) {
#pragma unroll
      for (int m = 0; m < MV; ++m) {
        const int i0 = 2 * (j + 8 * m);
        const float x0 = z[m].x - mean, x1 = z[m].y - mean;
        float xm1;
        if (m == 0 && j0) {
          xm1 = x0;
        } else {
          float prev = fr[i0 - 1];          // the neighbour lane's sample: its dither is recomputed, not exchanged
          if (dithered) prev = fmaf(a.dither, dither_pair(a.dither_seed, gframe, j + 8 * m - 1).y, prev);
          xm1 = prev - mean;
        }
        const float2 w = *reinterpret_cast<const float2*>(s_window + i0);
        if (a.raw_energy) esum = fmaf(x0, x0, fmaf(x1, x1, esum));
        const float y0 = (x0 - pc * xm1) * w.x;
        const float y1 = (x1 - pc * x0) * w.y;
        if (!a.raw_energy) esum = fmaf(y0, y0, fmaf(y1, y1, esum));
        z[m] = make_float2(y0, y1);
      }
    } else {
#pragma unroll
      for (int m = 0; m < R; ++m) {
        const int i0 = 2 * (j + 8 * m);
        float y0 = 0.0f, y1 = 0.0f;
        if (i0 < a.W) {
          const float x0 = z[m].x - mean;
          const bool has1 = (i0 + 1 < a.W);
          const float x1 = has1 ? z[m].y - mean : 0.0f;
          float xm1 = x0;
          if (i0 > 0) {
            float prev = fr[i0 - 1];
            if (dithered) prev = fmaf(a.dither, dither_pair(a.dither_seed, gframe, j + 8 * m - 1).y, prev);
            xm1 = prev - mean;
          }
          if (a.raw_energy) esum = fmaf(x0, x0, fmaf(x1, x1, esum));
          y0 = (x0 - pc * xm1) * s_window[i0];
          y1 = has1 ? (x1 - pc * x0) * s_window[i0 + 1] : 0.0f;
          if (!a.raw_energy) esum = fmaf(y0, y0, fmaf(y1, y1, esum));
        }
        z[m] = make_float2(y0, y1);
      }
    }
    __syncwarp();  // every lane is done with the span buffer

    // ---- prefetch the next item's span into the same buffer ----------------------------
    const Item me = cur;
    {
      const long long nxt = item + warp_stride;
      if (nxt < a.total_groups) {
        cur = decode_item(a, nxt);
        stage_span(a, cur, s_span, lane);
      }
    }

    float log_e = 0.0f;
    if (a.use_energy) {
      esum = group_sum8(esum);
      log_e = logf(fmaxf(esum, 0.0f) + a.eps);
      log_e = fminf(fmaxf(log_e, a.energy_floor), 3.402823466e+38f);
    }

    if (a.output == KTF_OUT_WINDOWED) {
      if (fvalid) {
        float* dst = a.out + (me.out_row0 + me.frame0 + f) * (long long)a.W;
#pragma unroll
        for (int m = 0; m < R; ++m) {
          const int i0 = 2 * (j + 8 * m);
          if (i0 < a.W) dst[i0] = z[m].x;
          if (i0 + 1 < a.W) dst[i0 + 1] = z[m].y;
        }
        if (a.use_energy && a.energy_out != nullptr && j0) a.energy_out[me.out_row0 + me.frame0 + f] = log_e;
      }
      continue;
    }

    // ---- stage 1: R-point FFT over m (registers), twiddle, transpose tile write ---------
    fft_dif<R, 0, R>(z);
    {
      float* tile = s_T + f * G::TFS + j * (RS * 2);
      const float2* twr = s_tw + j * RS;
#pragma unroll
      for (int k1 = 0; k1 < R; k1 += 2) {
        const float4 tw = *reinterpret_cast<const float4*>(twr + k1);
        const float2 y0 = cmul(z[brev(k1, LOGR)], make_float2(tw.x, tw.y));
        const float2 y1 = cmul(z[brev(k1 + 1, LOGR)], make_float2(tw.z, tw.w));
        *reinterpret_cast<float4*>(tile + 2 * k1) = make_float4(y0.x, y0.y, y1.x, y1.y);
      }
    }
    __syncwarp();

    // ---- stage 2: 8-point FFTs over l, real-FFT untangling, |X|^2 (x4: the 1/4 is in the mel
    //      weights).  Results are parked in registers until every lane has read the tile, which the
    //      power buffer aliases.
    float qa[NSLOT / 2][8], qb[NSLOT / 2][8];
#pragma unroll
    for (int p = 0; p < NSLOT / 2; ++p) {
      float2 va[8], vb[8];
      const float* cola = s_T + f * G::TFS + 2 * ka[p];
      const float* colb = s_T + f * G::TFS + 2 * kb[p];
#pragma unroll
      for (int l = 0; l < 8; ++l) {
        va[l] = *reinterpret_cast<const float2*>(cola + l * (RS * 2));
        vb[l] = *reinterpret_cast<const float2*>(colb + l * (RS * 2));
      }
      fft_dif<8, 0, 8>(va);
      fft_dif<8, 0, 8>(vb);
#pragma unroll
      for (int k2 = 0; k2 < 8; ++k2) {   // bin k = ka + R k2 pairs with C - k = kb + R (7 - k2)
        const float2 zk = va[brev(k2, 3)];
        float2 zp = vb[brev(7 - k2, 3)];
        zp.y = -zp.y;
        const float2 c16 = make_float2(KTF_COS64[4 * k2], -KTF_SIN64[4 * k2]);
        const float2 wk = (k2 == 0) ? base[p] : cmul(base[p], c16);
        const float2 S = cadd(zk, zp), Dd = csub(zk, zp);
        const float2 Gt = cmul(wk, Dd);
        qa[p][k2] = cnorm(cadd(S, Gt));
        qb[p][7 - k2] = cnorm(csub(S, Gt));
      }
    }
    // column k1 = 0 (bins 0, R, 2R, ...; partner of k2 is (8 - k2) & 7) and the Nyquist bin: lane 0 only
    float q0[8], qny = 0.0f;
    if (j0) {
      float2 v0[8];
      const float* col0 = s_T + f * G::TFS;
#pragma unroll
      for (int l = 0; l < 8; ++l) v0[l] = *reinterpret_cast<const float2*>(col0 + l * (RS * 2));
      fft_dif<8, 0, 8>(v0);
      const float2 w0 = a.post_tw[0];
#pragma unroll
      for (int k2 = 0; k2 < 8; ++k2) {
        const float2 zk = v0[brev(k2, 3)];
        float2 zp = v0[brev((8 - k2) & 7, 3)];
        zp.y = -zp.y;
        const float2 c16 = make_float2(KTF_COS64[4 * k2], -KTF_SIN64[4 * k2]);
        const float2 wk = (k2 == 0) ? w0 : cmul(w0, c16);
        const float2 S = cadd(zk, zp), Dd = csub(zk, zp);
        q0[k2] = cnorm(cadd(S, cmul(wk, Dd)));
      }
      const float t = 2.0f * v0[0].x - 2.0f * v0[0].y;   // X[C] = Re Z[0] - Im Z[0]
      qny = t * t;
    }
    __syncwarp();  // tile fully consumed

    float* Q = s_T + f * G::QS;
#pragma unroll
    for (int p = 0; p < NSLOT / 2; ++p) {
#pragma unroll
      for (int k2 = 0; k2 < 8; ++k2) {
        float v1 = qa[p][k2], v2 = qb[p][k2];
        if (!a.use_power) { v1 = sqrtf(v1); v2 = sqrtf(v2); }
        Q[qidx(ka[p] + R * k2)] = v1;
        Q[qidx(kb[p] + R * k2)] = v2;
      }
    }
    if (j0) {
#pragma unroll
      for (int k2 = 0; k2 < 8; ++k2) Q[qidx(R * k2)] = a.use_power ? q0[k2] : sqrtf(q0[k2]);
      Q[qidx(C)] = a.use_power ? qny : sqrtf(qny);
    }
    __syncwarp();

    // ---- mel bank (filterbank.py:238-240): lane (f, g=j) owns filters g, g+8, ... -------------
    for (int i = j; i < a.M; i += kGroups) {
      const int4 fl = s_filt[i];
      const float* wp = s_melw + fl.z;
      float acc = 0.0f;
      for (int c = 0; c < fl.y; ++c) {
        const float4 qv = *reinterpret_cast<const float4*>(Q + qchunk(fl.x + c));
        const float4 w = *reinterpret_cast<const float4*>(wp + 4 * c);
        acc = fmaf(w.x, qv.x, acc);
        acc = fmaf(w.y, qv.y, acc);
        acc = fmaf(w.z, qv.z, acc);
        acc = fmaf(w.w, qv.w, acc);
      }
      // __logf (MUFU.LG2 * ln2): absolute error <= ~2e-6 on log-mel values of magnitude ~20, two orders below
      // the float32 noise of the spectrum itself; the frame log-energy (VAD input) keeps the exact logf
      if (a.use_log) acc = __logf(fmaxf(acc, 0.0f) + a.eps);
      if (a.output == KTF_OUT_FBANK) s_out[f * a.M + i] = acc; else s_LM[f * LMS + i] = acc;
    }
    __syncwarp();

    if (a.output == KTF_OUT_MFCC) {
      // ---- DCT (dct.py:176), lifter (mfcc.py:212), C0 <- energy (mfcc.py:219-228) ---------
      float acc[4] = {0.0f, 0.0f, 0.0f, 0.0f};
      const float* lmrow = s_LM + f * LMS;
      const int M4 = a.M & ~3;
      for (int i = 0; i < M4; i += 4) {
        const float4 lm = *reinterpret_cast<const float4*>(lmrow + i);
        const float lmv[4] = {lm.x, lm.y, lm.z, lm.w};
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const float4 d = *reinterpret_cast<const float4*>(s_dct + (i + u) * 32 + j * 4);
          acc[0] = fmaf(lmv[u], d.x, acc[0]);
          acc[1] = fmaf(lmv[u], d.y, acc[1]);
          acc[2] = fmaf(lmv[u], d.z, acc[2]);
          acc[3] = fmaf(lmv[u], d.w, acc[3]);
        }
      }
      for (int i = M4; i < a.M; ++i) {
        const float lm = lmrow[i];
        const float4 d = *reinterpret_cast<const float4*>(s_dct + i * 32 + j * 4);
        acc[0] = fmaf(lm, d.x, acc[0]);
        acc[1] = fmaf(lm, d.y, acc[1]);
        acc[2] = fmaf(lm, d.z, acc[2]);
        acc[3] = fmaf(lm, d.w, acc[3]);
      }
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const int c = j + 8 * r;
        if (c < a.Kc) {
          float v = acc[r];
          if (a.apply_lifter) v *= s_lifter[c];
          if (c == 0 && a.use_energy) v = log_e;
          s_out[f * a.Kc + c] = v;
        }
      }
      __syncwarp();
    }

    // ---- coalesced store of the group's nvalid x out_dim tile -----------------------------
    {
      float* dst = a.out + (me.out_row0 + me.frame0) * (long long)a.out_dim;
      const int n = me.nvalid * a.out_dim;
      if (((n & 3) == 0) && ((reinterpret_cast<unsigned long long>(dst) & 15ull) == 0)) {
        const int n4 = n >> 2;
        for (int i = lane; i < n4; i += 32)
          reinterpret_cast<float4*>(dst)[i] = reinterpret_cast<const float4*>(s_out)[i];
      } else {
        for (int i = lane; i < n; i += 32) dst[i] = s_out[i];
      }
    }
    __syncwarp();
  }
}

__global__ void framing_kernel(const float* __restrict__ wav, long long wav_stride, long long T,
                               int W, int shift, float* __restrict__ out, long long total) {
  // total = batch * T * W elements; out[b][t][i] = wav[b][t*shift + i]  (framing.py:248-265)
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const int i = (int)(idx % W);
    const long long bt = idx / W;
    const long long t = bt % T, b = bt / T;
    out[idx] = wav[b * wav_stride + t * shift + i];
  }
}

}  // namespace


namespace {

template <int R>
size_t smem_for(const ktf_frontend* fe) {
  using G = Geo<R>;
  const int W = fe->cfg.frame_width, M = fe->cfg.num_mels > 0 ? fe->cfg.num_mels : 1;
  size_t fl = 0;
  fl += (W + 3) & ~3;
  fl += 2 * 8 * G::RS;
  fl += 4 * kMaxMels;
  fl += fe->mel_w_len;
  fl += (size_t)M * 32 + 32;
  const int span_p = (fe->span + 3) & ~3;
  const int LMS = ((M + 3) & ~3) + 4;
  const int out_sz = 4 * ((fe->out_dim + 3) & ~3);
  const size_t warp_floats = span_p + 4 * G::TFS + 4 * LMS + out_sz;
  fl += kWarpsPerCta * warp_floats;
  return fl * sizeof(float);
}

template <int R, int MV>
int launch(const ktf_frontend* fe, FrontendArgs& a, cudaStream_t st) {
  const size_t smem = smem_for<R>(fe);
  KTF_CUDA(cudaFuncSetAttribute(frontend_kernel<R, MV>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)std::max<size_t>(smem, 48 * 1024)));
  int occ = 0;
  KTF_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, frontend_kernel<R, MV>, kThreads, smem));
  if (occ < 1) occ = 1;
  const long long ctas_needed = (a.total_groups + kWarpsPerCta - 1) / kWarpsPerCta;
  const long long grid = std::min<long long>(ctas_needed, (long long)ktf::num_sms() * occ);
  if (grid <= 0) return KTF_OK;
  frontend_kernel<R, MV><<<(unsigned)grid, kThreads, smem, st>>>(a);
  KTF_LAUNCH_OK();
  return KTF_OK;
}

int dispatch(const ktf_frontend* fe, FrontendArgs& a, cudaStream_t st) {
  if (fe->d_wide != nullptr) return wide_launch(fe, a, st);
  if (fe->d_r16 != nullptr) return r16_launch(fe, a, st);
  const int W = fe->cfg.frame_width;
  const bool even_shift = (fe->cfg.frame_shift & 1) == 0;
  if (fe->R == 32) {
    if (W == 400 && even_shift) return launch<32, 25>(fe, a, st);
    if (W == 512 && even_shift) return launch<32, 32>(fe, a, st);
    return launch<32, 0>(fe, a, st);
  }
  if (W == 256 && even_shift) return launch<16, 16>(fe, a, st);
  if (W == 200 && even_shift) return launch<16, 0>(fe, a, st);
  return launch<16, 0>(fe, a, st);
}

void fill_args(const ktf_frontend* fe, FrontendArgs& a) {
  const ktf_frontend_cfg& c = fe->cfg;
  a.window = fe->d_window;
  a.stage_tw = fe->d_stage_tw;
  a.post_tw = fe->d_post_tw;
  a.mel_filt = fe->d_mel_filt;
  a.mel_w = fe->d_mel_w;
  a.mel_w_len = fe->mel_w_len;
  a.dct = fe->d_dct;
  a.lifter = fe->d_lifter;
  a.W = c.frame_width;
  a.shift = c.frame_shift;
  a.span = fe->span;
  a.M = c.num_mels > 0 ? c.num_mels : 1;
  a.Kc = c.num_ceps;
  a.out_dim = fe->out_dim;
  a.output = c.output;
  a.remove_dc = c.remove_dc_offset;
  a.raw_energy = c.raw_energy;
  a.use_energy = c.use_energy;
  a.use_power = c.use_power;
  a.use_log = c.use_log_fbank;
  a.apply_lifter = c.apply_lifter;
  a.preemph = c.preemphasis;
  a.energy_floor = c.energy_floor;
  a.eps = c.epsilon;
  a.dither = c.dither;
  a.dither_seed = c.dither != 0.0f ? 0x9E3779B97F4A7C15ull * (ktf::next_dither_stream() + 1) : 0ull;
  a.r16_blob = fe->d_r16;
  a.r16_blob_floats = fe->r16_blob_floats;
  a.r16_nf = fe->r16_nf;
  a.r16_melw_floats = fe->r16_melw_floats;
}

}  // namespace

extern "C" {

int ktf_frontend_create(const ktf_frontend_cfg* cfg, const float* window_host,
                        const float* mel_bank_host, const float* dct_host,
                        const float* lifter_host, ktf_frontend** out) {
  KTF_CHECK_ARG(cfg && out && window_host, "ktf_frontend_create: null argument");
  const int W = cfg->frame_width, N = cfg->fft_length;
  KTF_CHECK_ARG(W > 0 && cfg->frame_shift > 0, "frame_width and frame_shift must be > 0");
  KTF_CHECK_ARG(N >= W && (N & (N - 1)) == 0, "fft_length must be a power of two >= frame_width");
  KTF_CHECK_ARG(N <= 4096, "fft_length %d (frame_width %d) is too long for the fused front-end: the maximum is 4096 "
                "(frame_width <= 4096)", N, W);
  KTF_CHECK_ARG(N == 256 || N == 512 || N == 1024 || N == 2048 || N == 4096,
                "fft_length %d not supported by the fused front-end (supported: 256, 512, 1024, 2048, 4096)", N);
  KTF_CHECK_ARG(cfg->frame_shift <= 2 * N, "frame_shift %d too large", cfg->frame_shift);
  KTF_CHECK_ARG(cfg->output >= KTF_OUT_MFCC && cfg->output <= KTF_OUT_WINDOWED, "bad output kind");
  const bool need_mel = cfg->output != KTF_OUT_WINDOWED;
  const int M = cfg->num_mels, Kc = cfg->num_ceps;
  if (need_mel) {
    KTF_CHECK_ARG(mel_bank_host, "mel_bank_host is required");
    KTF_CHECK_ARG(M >= 1 && M <= kMaxMels, "num_mels must be in [1, %d]", kMaxMels);
  }
  if (cfg->output == KTF_OUT_MFCC) {
    KTF_CHECK_ARG(dct_host, "dct_host is required for MFCC output");
    KTF_CHECK_ARG(Kc >= 1 && Kc <= kMaxCeps && Kc <= M, "num_ceps must be in [1, min(%d, num_mels)]", kMaxCeps);
    KTF_CHECK_ARG(!cfg->apply_lifter || lifter_host, "lifter_host is required when apply_lifter");
  }

  ktf_frontend* fe = new ktf_frontend();
  fe->cfg = *cfg;
  fe->C = N / 2;
  fe->R = fe->C / 8;
  fe->out_dim = cfg->output == KTF_OUT_MFCC ? Kc : (cfg->output == KTF_OUT_FBANK ? M : W);
  fe->span = (kFramesPerWarp - 1) * cfg->frame_shift + W;
  const int C = fe->C, R = fe->R, RS = R + 2;

  int rc = KTF_OK;
  auto fail = [&](int code) { ktf_frontend_destroy(fe); return code; };

  if (N > 512) {   // 1024..4096 points: the one-frame-per-warp kernel of frontend_wide.cu, with its own tables
    if ((rc = wide_build(fe, window_host, mel_bank_host, dct_host, lifter_host)) != KTF_OK) return fail(rc);
    *out = fe;
    return KTF_OK;
  }

  if ((rc = ktf::upload(&fe->d_window, window_host, (size_t)W)) != KTF_OK) return fail(rc);

  const double PI = 3.14159265358979323846;
  std::vector<float2> stw((size_t)8 * RS, make_float2(0.f, 0.f));
  for (int l = 0; l < 8; ++l)
    for (int k1 = 0; k1 < R; ++k1) {
      const double th = -2.0 * PI * (double)((l * k1) % C) / (double)C;
      stw[(size_t)l * RS + k1] = make_float2((float)cos(th), (float)sin(th));
    }
  if ((rc = ktf::upload(&fe->d_stage_tw, stw.data(), stw.size())) != KTF_OK) return fail(rc);

  std::vector<float2> ptw((size_t)C + 1);
  for (int k = 0; k <= C; ++k) {  // -i * exp(-i th) = (-sin th, -cos th)
    const double th = 2.0 * PI * (double)k / (double)N;
    ptw[k] = make_float2((float)(-sin(th)), (float)(-cos(th)));
  }
  if ((rc = ktf::upload(&fe->d_post_tw, ptw.data(), ptw.size())) != KTF_OK) return fail(rc);

  if (need_mel) {
    // Filter-major sparse form of the (C+1) x M bank: filter i covers the 4-bin chunks
    // [first, first + n) of the spectrum; weights are stored chunk-padded with zeros.
    const float scale = cfg->use_power ? 0.25f : 0.5f;  // the kernel stores 4|X|^2 (or 2|X|)
    std::vector<int4> filt((size_t)M);
    std::vector<float> mw;
    for (int i = 0; i < M; ++i) {
      int lo = -1, hi = -1;
      for (int k = 0; k <= C; ++k)
        if (mel_bank_host[(size_t)k * M + i] != 0.0f) { if (lo < 0) lo = k; hi = k; }
      int c0 = 0, n = 0;
      if (lo >= 0) { c0 = lo >> 2; n = (hi >> 2) - c0 + 1; }
      filt[i] = make_int4(c0, n, (int)mw.size(), 0);
      for (int c = c0; c < c0 + n; ++c)
        for (int u = 0; u < 4; ++u) {
          const int k = 4 * c + u;
          mw.push_back(k <= C ? mel_bank_host[(size_t)k * M + i] * scale : 0.0f);
        }
    }
    if (mw.empty()) mw.assign(4, 0.0f);
    fe->mel_w_len = (int)mw.size();
    if ((rc = ktf::upload(&fe->d_mel_filt, filt.data(), filt.size())) != KTF_OK) return fail(rc);
    if ((rc = ktf::upload(&fe->d_mel_w, mw.data(), mw.size())) != KTF_OK) return fail(rc);
  }
  if (cfg->output == KTF_OUT_MFCC) {
    std::vector<float> dp((size_t)M * 32, 0.0f);
    for (int i = 0; i < M; ++i)
      for (int c = 0; c < Kc; ++c) dp[(size_t)i * 32 + (c & 7) * 4 + (c >> 3)] = dct_host[(size_t)i * Kc + c];
    std::vector<float> lf(32, 1.0f);
    if (cfg->apply_lifter)
      for (int c = 0; c < Kc; ++c) lf[c] = lifter_host[c];
    if ((rc = ktf::upload(&fe->d_dct, dp.data(), dp.size())) != KTF_OK) return fail(rc);
    if ((rc = ktf::upload(&fe->d_lifter, lf.data(), lf.size())) != KTF_OK) return fail(rc);
  }
  if (getenv("KTF_FRONTEND_GENERIC") == nullptr && cfg->dither == 0.0f &&   // dither: generic kernel (it draws the noise)
      (rc = r16_build(fe, window_host, mel_bank_host, dct_host, lifter_host)) != KTF_OK) return fail(rc);
  fe->smem_bytes = (R == 32) ? smem_for<32>(fe) : smem_for<16>(fe);
  if (fe->smem_bytes > 227 * 1024) {
    ktf::set_error("front-end configuration needs %zu bytes of shared memory (> 227 KB)", fe->smem_bytes);
    return fail(KTF_EINVAL);
  }
  *out = fe;
  return KTF_OK;
}

void ktf_frontend_destroy(ktf_frontend* fe) {
  if (!fe) return;
  cudaFree(fe->d_window);
  cudaFree(fe->d_stage_tw);
  cudaFree(fe->d_post_tw);
  cudaFree(fe->d_mel_filt);
  cudaFree(fe->d_mel_w);
  cudaFree(fe->d_dct);
  cudaFree(fe->d_lifter);
  cudaFree(fe->d_r16);
  cudaFree(fe->d_wide);
  delete fe;
}

int64_t ktf_frontend_num_frames_ex(const ktf_frontend* fe, int64_t num_samples, int32_t snip_edges) {
  if (!fe || num_samples < fe->cfg.frame_width) return 0;
  if (snip_edges) return 1 + (num_samples - fe->cfg.frame_width) / fe->cfg.frame_shift;
  return (num_samples + fe->cfg.frame_shift / 2) / fe->cfg.frame_shift;   // kaldi_numpy/frame_extraction.py:78-80
}

int64_t ktf_frontend_num_frames(const ktf_frontend* fe, int64_t num_samples) {
  return ktf_frontend_num_frames_ex(fe, num_samples, 1);
}

int32_t ktf_frontend_out_dim(const ktf_frontend* fe) { return fe ? fe->out_dim : 0; }

namespace {

// Common argument checks / setup of the ingest options (sample format, snip-edges).
int set_ingest(const ktf_frontend* fe, FrontendArgs& a, const void* wav_dev, int32_t sample_format,
               int32_t snip_edges) {
  KTF_CHECK_ARG(sample_format == KTF_SAMPLE_F32 || sample_format == KTF_SAMPLE_S16, "unknown sample_format %d",
                sample_format);
  if (sample_format == KTF_SAMPLE_S16) {
    KTF_CHECK_ARG(fe->d_r16 != nullptr || fe->d_wide != nullptr,
                  "int16 input is implemented by the fused 400-sample / 512-point MFCC / fbank kernel and by the "
                  "1024- to 4096-point kernel only");
    a.wav16 = static_cast<const short*>(wav_dev);
  } else {
    a.wav = static_cast<const float*>(wav_dev);
  }
  a.edge_off = snip_edges ? 0 : (fe->cfg.frame_width - fe->cfg.frame_shift) / 2;   // frame_extraction.py:85
  KTF_CHECK_ARG(a.edge_off >= 0, "snip_edges=0 needs frame_width >= frame_shift");
  return KTF_OK;
}

}  // namespace

int ktf_frontend_forward_ex(const ktf_frontend* fe, const void* wav_dev, int32_t sample_format,
                            int32_t snip_edges, int64_t batch, int64_t num_samples, int64_t wav_stride,
                            float* out_dev, float* energy_dev, void* stream) {
  KTF_CHECK_ARG(fe && wav_dev && out_dev, "ktf_frontend_forward: null argument");
  KTF_CHECK_ARG(batch >= 0 && wav_stride >= num_samples, "bad batch / stride");
  KTF_CHECK_ARG(num_samples >= fe->cfg.frame_width,
                "input sample size (%lld) must be >= frame size (%d)", (long long)num_samples,
                fe->cfg.frame_width);
  if (batch == 0) return KTF_OK;
  FrontendArgs a{};
  fill_args(fe, a);
  int rc = set_ingest(fe, a, wav_dev, sample_format, snip_edges);
  if (rc != KTF_OK) return rc;
  a.out = out_dev;
  a.energy_out = energy_dev;
  a.wav_stride = wav_stride;
  a.num_samples = num_samples;
  a.frames_per_utt = ktf_frontend_num_frames_ex(fe, num_samples, snip_edges);
  a.groups_per_utt = (a.frames_per_utt + kFramesPerWarp - 1) / kFramesPerWarp;
  a.batch = batch;
  a.total_groups = a.groups_per_utt * batch;
  // item / groups_per_utt as a multiply-shift: with m = ceil(2^40 / d), floor(n m / 2^40) == floor(n / d) whenever
  // n (m d - 2^40) < 2^40, which holds for n d < 2^40; n m must also fit 64 bits
  a.div_magic = 0;
  if (a.groups_per_utt > 0 && a.total_groups < (1ll << 31) &&
      (double)a.total_groups * (double)a.groups_per_utt < 1.0e12 * 1.0995 &&
      (double)a.total_groups * (double)(((1ull << 40) / (unsigned long long)a.groups_per_utt) + 1) < 1.8e19)
    a.div_magic = ((1ull << 40) + (unsigned long long)a.groups_per_utt - 1) / (unsigned long long)a.groups_per_utt;
  cudaStream_t st = (cudaStream_t)stream;
  return dispatch(fe, a, st);
}

int ktf_frontend_forward(const ktf_frontend* fe, const float* wav_dev, int64_t batch,
                         int64_t num_samples, int64_t wav_stride, float* out_dev,
                         float* energy_dev, void* stream) {
  return ktf_frontend_forward_ex(fe, wav_dev, KTF_SAMPLE_F32, 1, batch, num_samples, wav_stride, out_dev,
                                 energy_dev, stream);
}

int ktf_frontend_forward_ragged_ex(const ktf_frontend* fe, const void* wav_dev, int32_t sample_format,
                                   int32_t snip_edges, int64_t batch, const int64_t* sample_offsets_host,
                                   int64_t* frame_offsets_host, float* out_dev, float* energy_dev,
                                   void* stream) {
  KTF_CHECK_ARG(fe && wav_dev && out_dev && sample_offsets_host && frame_offsets_host,
                "ktf_frontend_forward_ragged: null argument");
  if (batch <= 0) return KTF_OK;
  cudaStream_t st = (cudaStream_t)stream;
  std::vector<long long> host((size_t)3 * (batch + 1));
  long long* so = host.data();
  long long* fo = so + (batch + 1);
  long long* go = fo + (batch + 1);
  fo[0] = 0;
  go[0] = 0;
  for (int64_t b = 0; b < batch; ++b) {
    so[b] = sample_offsets_host[b];
    const int64_t len = sample_offsets_host[b + 1] - sample_offsets_host[b];
    KTF_CHECK_ARG(len >= fe->cfg.frame_width,
                  "utterance %lld: input sample size (%lld) must be >= frame size (%d)",
                  (long long)b, (long long)len, fe->cfg.frame_width);
    const int64_t T = ktf_frontend_num_frames_ex(fe, len, snip_edges);
    fo[b + 1] = fo[b] + T;
    go[b + 1] = go[b] + (T + kFramesPerWarp - 1) / kFramesPerWarp;
  }
  so[batch] = sample_offsets_host[batch];
  for (int64_t b = 0; b <= batch; ++b) frame_offsets_host[b] = fo[b];

  FrontendArgs a{};
  fill_args(fe, a);
  int rc = set_ingest(fe, a, wav_dev, sample_format, snip_edges);
  if (rc != KTF_OK) return rc;

  ktf::Scratch scratch(st);            // released on every exit path
  long long* dev = nullptr;
  KTF_CUDA(scratch.take(&dev, host.size() * sizeof(long long)));
  KTF_CUDA(cudaMemcpyAsync(dev, host.data(), host.size() * sizeof(long long), cudaMemcpyHostToDevice, st));
  KTF_CUDA(cudaStreamSynchronize(st));  // `host` is pageable and dies at return

  a.out = out_dev;
  a.energy_out = energy_dev;
  a.sample_offsets = dev;
  a.frame_offsets = dev + (batch + 1);
  a.group_offsets = dev + 2 * (batch + 1);
  a.batch = batch;
  a.total_groups = go[batch];
  return dispatch(fe, a, st);
}

int ktf_frontend_forward_ragged(const ktf_frontend* fe, const float* wav_dev, int64_t batch,
                                const int64_t* sample_offsets_host, int64_t* frame_offsets_host,
                                float* out_dev, float* energy_dev, void* stream) {
  return ktf_frontend_forward_ragged_ex(fe, wav_dev, KTF_SAMPLE_F32, 1, batch, sample_offsets_host,
                                        frame_offsets_host, out_dev, energy_dev, stream);
}

int ktf_framing_forward(const float* wav_dev, int64_t batch, int64_t num_samples,
                        int64_t wav_stride, int32_t frame_width, int32_t frame_shift,
                        float* out_dev, void* stream) {
  KTF_CHECK_ARG(wav_dev && out_dev, "ktf_framing_forward: null argument");
  KTF_CHECK_ARG(frame_width > 0 && frame_shift > 0, "frame_width and frame_shift must be > 0");
  KTF_CHECK_ARG(num_samples >= frame_width, "input sample size (%lld) must be >= frame size (%d)",
                (long long)num_samples, frame_width);
  const long long T = 1 + (num_samples - frame_width) / frame_shift;
  const long long total = (long long)batch * T * frame_width;
  if (total == 0) return KTF_OK;
  const int threads = 256;
  const long long blocks = std::min<long long>((total + threads - 1) / threads, (long long)ktf::num_sms() * 16);
  framing_kernel<<<(unsigned)blocks, threads, 0, (cudaStream_t)stream>>>(wav_dev, wav_stride, T, frame_width,
                                                                        frame_shift, out_dev, total);
  KTF_LAUNCH_OK();
  return KTF_OK;
}

}  // extern "C"

// Internals shared by the front-end translation units (frontend.cu: generic radix-2 kernel and the
// C-ABI; frontend_r16.cu: the 16 x 16 fast path for 512-point FFTs; frontend_wide.cu: one frame per warp for
// 1024- to 4096-point FFTs).
#pragma once

#include "common.cuh"
#include "twiddles64.h"

namespace ktf_fe {

constexpr int kFramesPerWarp = 4;
constexpr int kWarpsPerCta = 4;
constexpr int kThreads = kWarpsPerCta * 32;
constexpr int kMaxMels = 128;
constexpr int kMaxCeps = 32;
constexpr int kGroups = 8;  // the 8 lanes of a frame cooperate as 8 "groups" in the mel / DCT stages

struct FrontendArgs {
  // data
  const float* wav;       // float32 samples, or
  const short* wav16;     // int16 PCM samples (fast path only); exactly one of the two is non-null
  float* out;
  float* energy_out;
  // uniform batch
  long long wav_stride;
  long long num_samples;
  long long frames_per_utt;
  long long groups_per_utt;
  // ragged batch (all nullptr for uniform)
  const long long* sample_offsets;
  const long long* frame_offsets;
  const long long* group_offsets;
  long long batch;
  long long total_groups;
  int edge_off;           // samples the first frame starts before sample 0 (0 = snip-edges, else mirror padding)
  unsigned long long div_magic;   // ceil(2^40 / groups_per_utt) when item * groups_per_utt < 2^40 for every item, else 0
  // tables (global memory, copied to smem per CTA)
  const float* window;     // [W]
  const float2* stage_tw;  // [8][R+2]
  const float2* post_tw;   // [C+1]  -i * W_{2C}^k
  const int4* mel_filt;    // [M]  (first 4-bin chunk, #chunks, offset into mel_w, 0)
  const float* mel_w;      // [mel_w_len] per-filter weights, chunk padded, prescaled
  const float* dct;        // [M][32] packed as [i][g][r] -> coefficient g + 8r
  const float* lifter;     // [32]
  // config
  int W, shift, span, M, Kc, out_dim, output, mel_w_len;
  int remove_dc, raw_energy, use_energy, use_power, use_log, apply_lifter;
  float preemph, energy_floor, eps;
  float dither;                    // windowing.py:182-183; 0 = off (generic kernel only: the fast path is built without it)
  unsigned long long dither_seed;  // Philox key of this forward call
  // 16 x 16 fast path (frontend_r16.cu): one blob laid out like the CTA's table region
  const float* r16_blob;
  int r16_blob_floats, r16_nf, r16_melw_floats;
  // wide kernel (frontend_wide.cu): one blob laid out like the CTA's table region, and the per-warp region size
  const float* wide_blob;
  int wide_blob_floats, wide_warp_floats;
  int wide_off_tw, wide_off_ustart, wide_off_units, wide_off_fslot, wide_off_melw, wide_off_dct, wide_off_lifter;
  int wide_lm_floats;
};

// Complex helpers and the in-register radix-2 FFT shared by the generic kernel (frontend.cu) and the wide kernel
// (frontend_wide.cu).
namespace radix2 {

__device__ __forceinline__ float2 cadd(float2 a, float2 b) { return make_float2(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ float2 csub(float2 a, float2 b) { return make_float2(a.x - b.x, a.y - b.y); }
__device__ __forceinline__ float2 cmul(float2 a, float2 b) {
  return make_float2(fmaf(a.x, b.x, -a.y * b.y), fmaf(a.x, b.y, a.y * b.x));
}
__device__ __forceinline__ float cnorm(float2 a) { return fmaf(a.x, a.x, a.y * a.y); }

constexpr __host__ __device__ int brev(int v, int bits) {
  int r = 0;
  for (int i = 0; i < bits; ++i) r |= ((v >> i) & 1) << (bits - 1 - i);
  return r;
}
constexpr __host__ __device__ int ilog2(int n) { return n <= 1 ? 0 : 1 + ilog2(n / 2); }

// In-register decimation-in-frequency radix-2 FFT of x[OFF .. OFF+N); output bit-reversed.
// All indices and twiddles are compile-time constants once unrolled.
template <int N, int OFF, int TOT>
__device__ __forceinline__ void fft_dif(float2 (&x)[TOT]) {
  if constexpr (N >= 2) {
    constexpr int H = N / 2;
#pragma unroll
    for (int i = 0; i < H; ++i) {
      const float2 a = x[OFF + i];
      const float2 b = x[OFF + i + H];
      x[OFF + i] = cadd(a, b);
      const float2 d = csub(a, b);
      float2 r;
      if (i == 0) {
        r = d;
      } else if (4 * i == N) {          // W = -i
        r = make_float2(d.y, -d.x);
      } else if (8 * i == N) {          // W = (1 - i)/sqrt2
        const float c = 0.70710678118654752440f;
        r = make_float2((d.x + d.y) * c, (d.y - d.x) * c);
      } else if (8 * i == 3 * N) {      // W = (-1 - i)/sqrt2
        const float c = 0.70710678118654752440f;
        r = make_float2((d.y - d.x) * c, -(d.x + d.y) * c);
      } else {
        const float wr = KTF_COS64[i * (64 / N)];
        const float wi = -KTF_SIN64[i * (64 / N)];
        r = make_float2(fmaf(d.x, wr, -d.y * wi), fmaf(d.x, wi, d.y * wr));
      }
      x[OFF + i + H] = r;
    }
    fft_dif<H, OFF, TOT>(x);
    fft_dif<H, OFF + H, TOT>(x);
  }
}

}  // namespace radix2

__device__ __forceinline__ float group_sum8(float v) {
  v += __shfl_xor_sync(0xffffffffu, v, 1);
  v += __shfl_xor_sync(0xffffffffu, v, 2);
  v += __shfl_xor_sync(0xffffffffu, v, 4);
  return v;
}

__device__ __forceinline__ void cp_async4(unsigned dst_smem, const float* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(dst_smem), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async16(unsigned dst_smem, const float* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(dst_smem), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() {
  asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;\n" ::: "memory");
}

// Counter-based noise for the dither of windowing.py:182-183: Philox4x32 (7 rounds: the fewest that pass BigCrush in
// the Random123 paper) keyed by the call's seed, counter = (global frame index, sample-pair index) -- every FRAMED sample
// has its own draw, so overlapping frames do not share noise, and a neighbour's draw can be recomputed instead of
// exchanged.  Returns two N(0,1) values (Box-Muller on the first two outputs; fast intrinsics are ample for dither).
__device__ __forceinline__ float2 dither_pair(unsigned long long seed, long long frame, int pair) {
  unsigned c0 = (unsigned)frame, c1 = (unsigned)((unsigned long long)frame >> 32), c2 = (unsigned)pair, c3 = 0x6b746621u;
  unsigned k0 = (unsigned)seed, k1 = (unsigned)(seed >> 32);
#pragma unroll
  for (int r = 0; r < 7; ++r) {
    const unsigned hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const unsigned hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    c0 = hi1 ^ c1 ^ k0;
    c1 = lo1;
    c2 = hi0 ^ c3 ^ k1;
    c3 = lo0;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  const float u1 = ((float)(c0 >> 8) + 1.0f) * (1.0f / 16777216.0f);   // (0, 1]
  const float u2 = (float)(c1 >> 8) * (1.0f / 16777216.0f);            // [0, 1)
  const float rad = sqrtf(-2.0f * __logf(u1));
  float sn, cs;
  __sincosf(6.283185307179586f * u2, &sn, &cs);
  return make_float2(rad * cs, rad * sn);
}

struct Item {
  long long utt_base, utt_len, out_row0, frame0;
  int nvalid;
};

// ---- TMA (bulk asynchronous copy) staging of a span: one elected lane issues a single cp.async.bulk of the whole span
// (global -> shared, completion counted in bytes on the warp's mbarrier); no per-lane address arithmetic, no LSU
// wavefronts for the fill.  Requires a 16-byte aligned source and a byte count that is a multiple of 16.
__device__ __forceinline__ void span_mbar_init(unsigned long long* bar) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;\n" ::"r"((unsigned)__cvta_generic_to_shared(bar)) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
}
__device__ __forceinline__ void span_bulk_load(void* smem_dst, const void* src, unsigned bytes, unsigned long long* bar) {
  const unsigned b = (unsigned)__cvta_generic_to_shared(bar);
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(b), "r"(bytes) : "memory");
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::
                   "r"((unsigned)__cvta_generic_to_shared(smem_dst)),
               "l"(src), "r"(bytes), "r"(b)
               : "memory");
}
__device__ __forceinline__ void span_mbar_wait(unsigned long long* bar, unsigned parity) {
  const unsigned b = (unsigned)__cvta_generic_to_shared(bar);
  unsigned ok = 0;
  while (!ok) {
    asm volatile(
        "{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}\n"
        : "=r"(ok)
        : "r"(b), "r"(parity)
        : "memory");
  }
}

__device__ __forceinline__ Item decode_item(const FrontendArgs& a, long long item) {
  Item it;
  long long q, utt_frames;
  if (a.group_offsets == nullptr) {
    long long b;
    if (a.div_magic != 0) b = (long long)(((unsigned long long)item * a.div_magic) >> 40);   // exact, see fill site
    else if (a.total_groups < 0x7fffffffLL) b = (unsigned)item / (unsigned)a.groups_per_utt;  // 32-bit division
    else b = item / a.groups_per_utt;
    q = item - b * a.groups_per_utt;
    it.utt_base = b * a.wav_stride;
    it.utt_len = a.num_samples;
    utt_frames = a.frames_per_utt;
    it.out_row0 = b * a.frames_per_utt;
  } else {
    long long lo = 0, hi = a.batch;  // largest b with group_offsets[b] <= item
    while (hi - lo > 1) {
      const long long mid = (lo + hi) >> 1;
      if (a.group_offsets[mid] <= item) lo = mid; else hi = mid;
    }
    q = item - a.group_offsets[lo];
    it.utt_base = a.sample_offsets[lo];
    it.utt_len = a.sample_offsets[lo + 1] - it.utt_base;
    it.out_row0 = a.frame_offsets[lo];
    utt_frames = a.frame_offsets[lo + 1] - it.out_row0;
  }
  it.frame0 = q * kFramesPerWarp;
  it.nvalid = (int)min((long long)kFramesPerWarp, utt_frames - it.frame0);
  return it;
}

// Source sample index of position `idx` of the (virtually) mirror-padded utterance: Kaldi's snip-edges=false
// reflection (kaldi_numpy/frame_extraction.py:28-51), clamped for utterances shorter than the padding.
__device__ __forceinline__ long long reflect_index(long long idx, long long len) {
  if (idx < 0) idx = -idx - 1;
  if (idx >= len) idx = 2 * len - 1 - idx;
  return idx < 0 ? 0 : (idx >= len ? len - 1 : idx);
}

// Asynchronously stages the item's sample span into the warp's smem buffer.  16-byte copies when the span is inside
// the utterance and aligned; otherwise element copies, zero filled past the end of the utterance (snip-edges) or
// mirrored at both ends (edge_off > 0).
__device__ __forceinline__ void stage_span(const FrontendArgs& a, const Item& it, float* s_span, int lane) {
  const long long s0 = it.frame0 * a.shift - a.edge_off;
  const float* src = a.wav + it.utt_base + s0;
  const long long avail = it.utt_len - s0;
  const unsigned sdst = (unsigned)__cvta_generic_to_shared(s_span);
  if (s0 >= 0 && avail >= a.span && ((reinterpret_cast<unsigned long long>(src) & 15ull) == 0)) {
    const int n4 = a.span >> 2;
    if (n4 == 220) {   // 3 * 160 + 400 samples: the 16 kHz / 25 ms / 10 ms geometry, fully unrolled
#pragma unroll
      for (int t = 0; t < 7; ++t) {
        const int i = lane + 32 * t;
        if (t < 6 || i < 220) cp_async16(sdst + 16u * i, src + 4 * i);
      }
    } else {
      for (int i = lane; i < n4; i += 32) cp_async16(sdst + 16u * i, src + 4 * i);
    }
    for (int i = (n4 << 2) + lane; i < a.span; i += 32) cp_async4(sdst + 4u * i, src + i);
  } else if (a.edge_off == 0) {
    for (int i = lane; i < a.span; i += 32) {
      if (i < avail) cp_async4(sdst + 4u * i, src + i); else s_span[i] = 0.0f;
    }
  } else {
    const float* utt = a.wav + it.utt_base;
    for (int i = lane; i < a.span; i += 32) cp_async4(sdst + 4u * i, utt + reflect_index(s0 + i, it.utt_len));
  }
}

// int16 PCM variant: the smem buffer holds the raw 16-bit samples (converted when the window is applied).
__device__ __forceinline__ void stage_span16(const FrontendArgs& a, const Item& it, short* s_span, int lane) {
  const long long s0 = it.frame0 * a.shift - a.edge_off;
  const short* src = a.wav16 + it.utt_base + s0;
  const long long avail = it.utt_len - s0;
  const unsigned sdst = (unsigned)__cvta_generic_to_shared(s_span);
  if (s0 >= 0 && avail >= a.span && ((reinterpret_cast<unsigned long long>(src) & 15ull) == 0) && (a.span & 7) == 0) {
    const int n8 = a.span >> 3;
    for (int i = lane; i < n8; i += 32)
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(sdst + 16u * i), "l"(src + 8 * i) : "memory");
  } else if (a.edge_off == 0) {
    for (int i = lane; i < a.span; i += 32) s_span[i] = (i < avail) ? src[i] : (short)0;
  } else {
    const short* utt = a.wav16 + it.utt_base;
    for (int i = lane; i < a.span; i += 32) s_span[i] = utt[reflect_index(s0 + i, it.utt_len)];
  }
}

}  // namespace ktf_fe

struct ktf_frontend {
  ktf_frontend_cfg cfg;
  int R = 0;          // complex FFT length / 8
  int C = 0;
  int out_dim = 0;
  int span = 0;
  int mel_w_len = 4;
  size_t smem_bytes = 0;
  float* d_window = nullptr;
  float2* d_stage_tw = nullptr;
  float2* d_post_tw = nullptr;
  int4* d_mel_filt = nullptr;
  float* d_mel_w = nullptr;
  float* d_dct = nullptr;
  float* d_lifter = nullptr;
  // 16 x 16 fast path (frontend_r16.cu); null when the configuration is not eligible
  float* d_r16 = nullptr;
  int r16_blob_floats = 0, r16_nf = 0, r16_melw_floats = 0, r16_dct_sym = 0;
  // wide kernel (frontend_wide.cu, fft_length 1024..4096); null for shorter FFTs
  float* d_wide = nullptr;
  int wide_blob_floats = 0, wide_warp_floats = 0, wide_warps = 0, wide_lm_floats = 0;
  int wide_off_tw = 0, wide_off_ustart = 0, wide_off_units = 0, wide_off_fslot = 0, wide_off_melw = 0,
      wide_off_dct = 0, wide_off_lifter = 0;
};

namespace ktf_fe {
// Builds the fast-path tables when the configuration is eligible (512-point FFT, 400-sample frames, power
// spectrum, log mel, DC removal); leaves fe->d_r16 == nullptr otherwise.  Returns KTF_OK or an error.
int r16_build(ktf_frontend* fe, const float* window_host, const float* mel_bank_host, const float* dct_host,
              const float* lifter_host);
int r16_launch(const ktf_frontend* fe, FrontendArgs& a, cudaStream_t st);
// Builds the wide kernel's tables (fft_length 1024, 2048 or 4096) and picks its CTA size; fails with KTF_EINVAL when
// even a one-warp CTA would need more than 227 KB of shared memory.
int wide_build(ktf_frontend* fe, const float* window_host, const float* mel_bank_host, const float* dct_host,
               const float* lifter_host);
int wide_launch(const ktf_frontend* fe, FrontendArgs& a, cudaStream_t st);
}  // namespace ktf_fe

// tcgen05 / TMEM implicit-GEMM engine for the TDNN stack and PLDA scoring (sm_100a only).
//
// Replaces the tf.gather + tf.nn.conv2d formulation of layers/tdnn/tdnn.py:251-280, the keras
// ReLU / BatchNormalization passes that follow it (models/kaldi/sequential.py:71-76,
// layers/normalization/batchnorm.py:81-88) and the reduce-all branch of
// layers/stats/stats_pooling.py:211-240 with ONE warp-specialised kernel per layer:
//
//   y[r, u] = scale[u] * relu( sum_k sum_d x[r + ctx_k, d] * W[u, k*D + d] + bias[u] ) + offset[u]
//
//   * operands 16-bit (bf16 for the TDNN, fp16 hi/lo splits for PLDA), accumulation fp32 in TMEM (tcgen05.mma kind::f16);
//   * the frame splice is IMPLICIT: tap k is a TMA box load of the activation matrix shifted by ctx_k
//     rows -- the (B, T, K, D) gathered tensor of the reference is never built;
//   * edge clamping (tdnn.py:244-247) is provided by the activation layout: every utterance carries
//     kHalo replicated rows on both sides ("padded rows"); the epilogue of each layer writes the halo
//     replicas the next layer's taps need and skips the halo rows of its own tile;
//   * two kernels share the helpers.  tdnn_tc_pair_kernel (row-storing layers, PLDA scoring): clusters of two CTAs
//     compute 256 x 256 tiles with cta_group::2 (each CTA owns 128 rows and loads half of B), 8 or 16 epilogue warps,
//     a 5- or 4-stage ring of 32 KB k-blocks, rows leave as 32-row x 128-byte TMA store boxes.  tdnn_tc_kernel
//     (single CTA, M128 x N256 x K16, 4-stage ring of 48 KB): the STATS layer, and every launch under KTF_TC_PAIR=0;
//   * warp roles: warp 0 = TMA producer, warp 1 = MMA issuer (one elected lane) + TMEM allocator, the others = epilogue
//     (a thread owns one accumulator row: TMEM load -> per-column vectors -> staging -> boxed / per-row store);
//   * 2 accumulator stages of 256 TMEM columns between MMA and epilogue, persistent CTAs (one per SM);
//   * three outputs: bf16 rows (next layer's operand), fp32 rows (+ per-row / per-column addends:
//     PLDA's A_i + B_j; optionally only the best entry per row), and STATS: the layer that feeds StatsPooling runs
//     with the operands swapped (M = units, N = frames), so a thread owns ONE unit and walks the frames of the tile in
//     its own registers -- per-utterance sum / sum-of-squares need no cross-thread reduction and the widest
//     activation of the network (frames x 1500) is never written to HBM.
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <stdlib.h>

#include <algorithm>
#include <vector>

#include "common.cuh"
#include "tdnn_internal.cuh"

namespace {

constexpr int kHalo = 4;          // replicated rows on each side of every utterance (>= max |context|)
constexpr int BM = 128, BN = 256, BK = 64;
constexpr int kStages = 4;
constexpr int kAccStages = 2;
constexpr int kEpiWarps = 8;                         // 2 per TMEM lane quarter, 128 tile columns each
constexpr int kEpiThreads = kEpiWarps * 32;          // 256
constexpr int kThreadsTc = 64 + kEpiThreads;         // 10 warps
constexpr int kEpiCols = BN / (kEpiWarps / 4);       // 64 columns of the tile per epilogue warp
constexpr int kEpiChunks = kEpiCols / 32;            // 32-column TMEM loads per warp and tile
constexpr int kABytes = BM * BK * 2;                 // 16 KB
constexpr int kBBytes = BN * BK * 2;                 // 32 KB
constexpr int kStageBytes = kABytes + kBBytes;
constexpr int kVecBytes = kAccStages * 3 * BN * 4;   // epilogue vectors (bias / scale / offset)
constexpr int kSegBytes = kAccStages * BN * 4;       // STATS: utterance id of every frame of the tile
constexpr int kRowSeg = 64;                          // bytes of one output row written by one group of lanes
constexpr int kStgPitch = kRowSeg + 16;              // staged row pitch: payload + 16 B (bank spread)
constexpr int kStgBytes = kEpiWarps * 32 * kStgPitch;  // per-warp 32-row transpose buffers for coalesced stores
constexpr int kSmemTc = kStages * kStageBytes + 1024 /*align*/ + 256 /*barriers*/ + kVecBytes + kSegBytes + kStgBytes;
static_assert((kStages * kStageBytes) % 512 == 0 && (32 * kStgPitch) % 512 == 0,
              "staging buffers are TMA-store sources with the 64-byte swizzle: 512-byte aligned");

enum { kModeBf16 = 0, kModeF32 = 1, kModeStats = 2 };
// Pair kernel, per-row top-k (nothing stored, see TcArgs::topk_k): lists of up to 8, 16 or 32 entries per thread.  The
// capacity is part of the mode because it sets the shared-memory layout and with it the number of ring stages.
enum { kModeTopk8 = 3, kModeTopk16 = 4, kModeTopk32 = 5 };
constexpr int topk_cap(int mode) { return mode >= kModeTopk8 ? 8 << (mode - kModeTopk8) : 0; }

// rowmap flags
constexpr int kRowStore = 1, kRowFirst = 2, kRowLast = 4;
constexpr int kRowFlagMask = 7;      // bits above hold splice bookkeeping (build_padded_kernel)
constexpr int kRowEmpty = 8;         // halo row of an empty utterance: the splices write zeros and read nothing

struct TcArgs {
  int num_taps;
  int ctx[KTF_MAX_CONTEXT];
  int kblocks_per_tap;      // ceil(D / 64)
  int tap_cols;             // column distance between taps in the weight matrix (= D)
  int shift_b;              // 0: taps shift the A rows (activations are A); 1: taps shift the B rows (STATS)
  int fp16;                 // operand format: 0 = bf16, 1 = fp16
  long long m_rows;         // rows of the A operand (output rows; STATS: units)
  long long n_rows;         // rows of the B operand (output columns; STATS: frames)
  const int* rowmap;        // per output row flags, or nullptr = store every row < m_rows
  const int* rowseg;        // STATS: per frame utterance id, < 0 for halo rows
  const float* bias;        // per column (STATS: per unit = per row)
  const float* scale;
  const float* offset;
  const float* row_add;     // F32 mode: per-row addend or nullptr
  int relu;
  void* out;                // bf16 or fp32, row-major
  long long out_ld;
  float* sums;              // STATS: (batch, 2, m_rows) sum / sum of squares of relu(acc + bias) - shift
  const float* shift;       // STATS: per unit centre of the sums (TcLayer::d_shift), or nullptr = 0
  const void* act_base;     // activation matrix (the operand that streams from HBM), for the L2 prefetch
  long long act_ld_bytes;   // its row pitch and row count
  long long act_rows;
  const long long* rows_dev;  // optional: the ACTUAL number of activation rows, read on the device (m_rows, or n_rows
                              // when shift_b); the host value is then only an upper bound (VAD-compacted batches: no
                              // host round trip for the kept-row count)
  int group_m;              // > 1: grouped tile walk (see tile_coords)
  int tma_store;            // rows are written with TMA tensor stores (tmC is valid; see store_chunk)
  int l2_stream_out;        // the output is a pure stream much larger than L2 while the operands are re-read by every
                            // tile (PLDA scoring: 10 GB of scores against 76 MB of vectors): operand loads carry an
                            // evict-last L2 policy and the boxed stores evict-first, so the stream does not push the
                            // operands out to HBM (measured without: 3.4-4.3 GB of DRAM reads for 76 MB of inputs)
  int reverse;              // walk the tiles from the last row block to the first (see launch_gemm)
  int debug;                // development knobs (KTF_TC_DEBUG): 1 = skip global stores, 2 = skip the epilogue math,
                            // 4 = stage the boxes but never issue their stores
  long long* trace;         // development (KTF_TC_TRACE=file): clock64 of cluster 0's tile phases, 4 slots per tile
  unsigned long long* row_best;   // pair kernel, optional: instead of storing C, keep the best entry of every row as an
                                  // atomically maximised key (order-preserving float bits << 32 | ~column), see top1_key
  // pair kernel, top-k modes: the tile walk is a sequence of units (one 256-row block x topk_unit_tiles consecutive
  // n-tiles); every (row, column quarter) thread keeps the topk_k best entries of its columns over the unit and writes
  // them, unordered, as one partial list: topk_score / topk_index (num_lists, m_rows, topk_k), list = split * EW / 4 +
  // column quarter, (-inf, -1) for empty entries
  int topk_k;
  int topk_unit_tiles;
  float* topk_score;
  long long* topk_index;
};

__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(unsigned long long* bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned long long* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ unsigned mbar_try_wait(unsigned long long* bar, unsigned parity) {
  unsigned ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok;
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}

__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* map, unsigned long long* bar,
                                            int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];\n" ::
          "r"(smem_u32(smem_dst)),
      "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}

__device__ __forceinline__ void tma_load_2d_hint(void* smem_dst, const CUtensorMap* map, unsigned long long* bar,
                                                 int c0, int c1, unsigned long long policy) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4}], "
      "[%2], %5;\n" ::"r"(smem_u32(smem_dst)),
      "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "l"(policy)
      : "memory");
}
__device__ __forceinline__ unsigned long long l2_policy_evict_last() {
  unsigned long long p;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;\n" : "=l"(p));
  return p;
}
__device__ __forceinline__ unsigned long long l2_policy_evict_first() {
  unsigned long long p;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;\n" : "=l"(p));
  return p;
}

// Pulls a contiguous byte range into L2 (no smem, no barrier).  The smem ring holds 4 k-blocks (~1 us of
// MMA work), less than the HBM latency under load, so the activation rows of a CTA's NEXT tile are
// requested one whole tile ahead with a single bulk prefetch.
__device__ __forceinline__ void bulk_prefetch_l2(const void* p, unsigned bytes) {
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;\n" ::"l"(p), "r"(bytes) : "memory");
}

// TMA tensor store of one staged box (smem -> global) as a bulk async-group; the staging buffer may be rewritten once
// tma_store_wait_read() has returned (the group has finished READING shared memory).
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, const void* smem_src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];\n"
               "cp.async.bulk.commit_group;\n" ::"l"(map), "r"(smem_u32(smem_src)), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void tma_store_2d_hint(const CUtensorMap* map, const void* smem_src, int c0, int c1,
                                                  unsigned long long policy) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group.L2::cache_hint [%0, {%2, %3}], [%1], %4;\n"
               "cp.async.bulk.commit_group;\n" ::"l"(map), "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "l"(policy)
               : "memory");
}
__device__ __forceinline__ void tma_store_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read 0;\n" ::: "memory");
}
// generic-proxy writes to shared memory (the staging STS) -> visible to the async proxy (TMA)
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
}

// K-major, 128B-swizzled operand tile: rows of 64 16-bit elements (128 B), 8-row groups 1024 B apart.
__device__ __forceinline__ unsigned long long umma_desc(unsigned smem_addr) {
  unsigned long long d = 0;
  d |= (unsigned long long)((smem_addr & 0x3FFFF) >> 4);
  d |= (unsigned long long)(1024 >> 4) << 32;   // stride byte offset
  d |= (unsigned long long)1 << 46;             // descriptor version (sm_100)
  d |= (unsigned long long)2 << 61;             // SWIZZLE_128B
  return d;
}

__device__ __forceinline__ void umma_f16(unsigned tmem_d, unsigned long long adesc, unsigned long long bdesc,
                                         unsigned idesc, unsigned accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit(unsigned long long* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n" ::"r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory"); }

// Asynchronous TMEM -> register load of 32 consecutive columns of this thread's lane.  The registers
// may only be read after tmem_ld_wait(), which names them as in/out operands so that the compiler
// cannot move their uses above the wait.
__device__ __forceinline__ void tmem_ld32_issue(unsigned taddr, unsigned (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait(unsigned (&r)[32]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;\n"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
                 "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]),
                 "+r"(r[15]), "+r"(r[16]), "+r"(r[17]), "+r"(r[18]), "+r"(r[19]), "+r"(r[20]), "+r"(r[21]),
                 "+r"(r[22]), "+r"(r[23]), "+r"(r[24]), "+r"(r[25]), "+r"(r[26]), "+r"(r[27]), "+r"(r[28]),
                 "+r"(r[29]), "+r"(r[30]), "+r"(r[31])::"memory");
}

__device__ __forceinline__ unsigned pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<unsigned*>(&h);
}

// One 32-column chunk of a warp's 32 accumulator rows: y = scale * max(acc + bias, relu_lo) + offset (+ radd).
// A thread owns one ROW of the accumulator (TMEM lane), so storing straight from registers would make every
// warp-wide store touch 32 different rows with 16 bytes each (32 partial sectors per instruction -- measured
// as the bottleneck of the K <= 512 layers).  The chunk is therefore transposed through a per-warp staging
// buffer in kRowSeg-byte row segments (32 bf16 / 16 fp32 columns): lanes write their own row, then 4
// consecutive lanes read back one row segment, so a warp store covers 8 rows x 64 contiguous bytes (16 full
// sectors).
// Rows flagged first / last also write their kHalo replicas; rows without kRowStore are skipped.
// VEC = false (ragged right edge, unaligned output): fp32 staging, bounds-checked scalar stores.
// VEC staging layout: row r of the 32 x 64-byte block starts at 64 r and its 16-byte piece g sits at position
// g ^ ((r >> 1) & 3): the eight lanes of a quarter-warp hit 32 different banks both when lanes write their own row
// (STS.128, rows 8q .. 8q+7) and when four consecutive lanes read back one row (LDS.128, rows 2q', 2q'+1).
// `plain` (warp-uniform): every one of the warp's 32 rows is a plain kRowStore row -- no per-row flag traffic.
template <bool OUT_BF16, bool VEC>
__device__ __forceinline__ void store_chunk(const unsigned (&r)[32], const float* vb, float relu_lo, float radd,
                                            unsigned char* stg, int lane, int flags, bool plain, unsigned char* out0,
                                            long long ld_bytes, int cols_left, const CUtensorMap* tmC, int tma_col,
                                            int tma_row, bool& tma_pending, unsigned long long store_policy) {
  const float4* b4 = reinterpret_cast<const float4*>(vb);
  const float4* s4 = reinterpret_cast<const float4*>(vb + BN);
  const float4* o4 = reinterpret_cast<const float4*>(vb + 2 * BN);
  constexpr bool kPacked = OUT_BF16 && VEC;        // staged as bf16 or as fp32
  constexpr int kCols = kRowSeg / (kPacked ? 2 : 4);   // columns per staged row segment
  constexpr int kPieces = kRowSeg / 16;            // 16-byte pieces per row segment
  constexpr int kEs = OUT_BF16 ? 2 : 4;
  constexpr int kPitch = VEC ? kRowSeg : kStgPitch;
  constexpr int kGroups = kCols / 8;               // groups of 8 columns per pass
  const int wsw = (lane >> 1) & 3;                 // swizzle of my own row (VEC): the 64-byte TMA swizzle pattern
  // `plain` VEC blocks (all 32 rows stored, no halo replicas) leave through a TMA tensor store of the staged box:
  // no read-back, no per-lane global stores.  tmC == nullptr: st.global path.
  const bool tma = VEC && plain && tmC != nullptr;
#pragma unroll
  for (int pass = 0; pass < 32 / kCols; ++pass) {
    uint4* mine = reinterpret_cast<uint4*>(stg + lane * kPitch);
    uint4 val[kPacked ? kGroups : 2 * kGroups];    // the math first: it covers the wait for the previous box
#pragma unroll
    for (int g = 0; g < kGroups; ++g) {            // 8 columns per group
      const int c8 = pass * kGroups + g;           // which group of 8 columns of the chunk
      float x[8];
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const float4 bb = b4[2 * c8 + h], ss = s4[2 * c8 + h], oo = o4[2 * c8 + h];
        x[4 * h + 0] = fmaf(fmaxf(__uint_as_float(r[8 * c8 + 4 * h + 0]) + bb.x, relu_lo), ss.x, oo.x);
        x[4 * h + 1] = fmaf(fmaxf(__uint_as_float(r[8 * c8 + 4 * h + 1]) + bb.y, relu_lo), ss.y, oo.y);
        x[4 * h + 2] = fmaf(fmaxf(__uint_as_float(r[8 * c8 + 4 * h + 2]) + bb.z, relu_lo), ss.z, oo.z);
        x[4 * h + 3] = fmaf(fmaxf(__uint_as_float(r[8 * c8 + 4 * h + 3]) + bb.w, relu_lo), ss.w, oo.w);
      }
      if (kPacked) {
        val[g] = make_uint4(pack_bf16x2(x[0] + radd, x[1] + radd), pack_bf16x2(x[2] + radd, x[3] + radd),
                            pack_bf16x2(x[4] + radd, x[5] + radd), pack_bf16x2(x[6] + radd, x[7] + radd));
      } else {
        val[2 * g] = make_uint4(__float_as_uint(x[0] + radd), __float_as_uint(x[1] + radd),
                                __float_as_uint(x[2] + radd), __float_as_uint(x[3] + radd));
        val[2 * g + 1] = make_uint4(__float_as_uint(x[4] + radd), __float_as_uint(x[5] + radd),
                                    __float_as_uint(x[6] + radd), __float_as_uint(x[7] + radd));
      }
    }
    if (tma_pending) {                             // warp-uniform: the previous box still reads the staging buffer
      if (lane == 0) tma_store_wait_read();
      __syncwarp();
      tma_pending = false;
    }
#pragma unroll
    for (int g = 0; g < kGroups; ++g) {
      if (kPacked) {
        mine[g ^ wsw] = val[g];
      } else {
        const int sw = VEC ? wsw : 0;
        mine[(2 * g) ^ sw] = val[2 * g];
        mine[(2 * g + 1) ^ sw] = val[2 * g + 1];
      }
    }
    if (tma) {
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) {
        if (store_policy != 0ull) tma_store_2d_hint(tmC, stg, tma_col + pass * kCols, tma_row, store_policy);
        else tma_store_2d(tmC, stg, tma_col + pass * kCols, tma_row);
      }
      tma_pending = true;
      continue;
    }
    __syncwarp();
    if (VEC) {
#pragma unroll
      for (int j = 0; j < kPieces; ++j) {
        const int q = j * 32 + lane, rr = q / kPieces, part = q % kPieces;
        const uint4 v = *reinterpret_cast<const uint4*>(stg + rr * kRowSeg + ((part ^ ((rr >> 1) & 3)) * 16));
        unsigned char* dst = out0 + rr * ld_bytes + pass * kRowSeg + part * 16;
        if (plain) {
          *reinterpret_cast<uint4*>(dst) = v;
          continue;
        }
        const int f = __shfl_sync(0xffffffffu, flags, rr);
        if (f & kRowStore) {
          *reinterpret_cast<uint4*>(dst) = v;
          if (f & (kRowFirst | kRowLast)) {
            const int lo = (f & kRowFirst) ? kHalo : 0, hi = (f & kRowLast) ? kHalo : 0;
#pragma unroll 1
            for (int h = -lo; h <= hi; ++h)
              if (h != 0) *reinterpret_cast<uint4*>(dst + h * ld_bytes) = v;
          }
        }
      }
    } else {
#pragma unroll 1
      for (int k = lane; k < 32 * kCols; k += 32) {
        const int rr = k / kCols, col = k % kCols;
        const float v = *reinterpret_cast<const float*>(stg + rr * kStgPitch + col * 4);
        const int f = __shfl_sync(0xffffffffu, flags, rr);
        if ((f & kRowStore) && pass * kCols + col < cols_left) {
          const int lo = (f & kRowFirst) ? kHalo : 0, hi = (f & kRowLast) ? kHalo : 0;
          unsigned char* dst = out0 + rr * ld_bytes + (long long)(pass * kCols + col) * kEs;
#pragma unroll 1
          for (int h = -lo; h <= hi; ++h) {
            if (OUT_BF16) *reinterpret_cast<__nv_bfloat16*>(dst + h * ld_bytes) = __float2bfloat16_rn(v);
            else *reinterpret_cast<float*>(dst + h * ld_bytes) = v;
          }
        }
      }
    }
    __syncwarp();
  }
}

// Pair-kernel chunk store through 128-byte-wide staging boxes (32 rows x 128 bytes, the 128-byte TMA swizzle): a 32-column
// chunk of fp32 rows fills a box, a chunk of bf16 rows fills half of one (HALF = chunk & 1) and the box leaves after the
// second half -- one boxed store per 4 KB instead of one per 2 KB, i.e. half the fence / elect / issue sequences per tile.
// A warp has ONE box: before refilling it waits for its previous store to have read the box (issued a whole tile
// earlier for bf16 rows with 16 warps; two boxes per warp measured equal and cost a ring stage).
// EPI: kEpiFull  y = scale * max(acc + bias, lo) + offset      (TDNN + ReLU + BatchNorm; never with a row addend)
//      kEpiLean  y = max(acc + bias, lo) + row addend           (no per-column scale / offset)
//      kEpiAdd   y = (acc + bias) + row addend                  (PLDA scoring: nothing to clamp)
// all three round like the general form with scale 1 / offset 0 / lo = -FLT_MAX, so every path gives the same fp32 value.
constexpr int kEpiFull = 0, kEpiLean = 1, kEpiAdd = 2;

// Key of (value, column) whose unsigned order is: larger value first, then SMALLER column.  0 never occurs for a real value.
__device__ __forceinline__ unsigned long long top1_key(float v, int col) {
  const unsigned b = __float_as_uint(v);
  const unsigned u = (b & 0x80000000u) ? ~b : (b | 0x80000000u);
  return ((unsigned long long)u << 32) | (unsigned long long)(0xffffffffu - (unsigned)col);
}
__device__ __forceinline__ float top1_key_value(unsigned long long key) {
  const unsigned u = (unsigned)(key >> 32);
  return __uint_as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u);
}
constexpr int kBoxRow = 128;                         // bytes per staged row of a box
constexpr int kBoxBytes = 32 * kBoxRow;

template <bool OUT_BF16, int EPI, int VSTRIDE, int HALF>
__device__ __forceinline__ void store_box(const unsigned (&r)[32], const float* vb, float relu_lo, float radd,
                                          unsigned char* stg, int lane, int flags, bool plain,
                                          unsigned char* out_box, long long ld_bytes, const CUtensorMap* tmC, int tma_col,
                                          int tma_row, bool& tma_pending, unsigned long long store_policy, int dbg) {
  const float4* b4 = reinterpret_cast<const float4*>(vb);
  const float4* s4 = reinterpret_cast<const float4*>(vb + VSTRIDE);
  const float4* o4 = reinterpret_cast<const float4*>(vb + 2 * VSTRIDE);
  constexpr int kVals = OUT_BF16 ? 4 : 8;              // 16-byte pieces this chunk contributes to a staged row
  const bool tma = plain && tmC != nullptr;
  uint4 val[kVals];
#pragma unroll
  for (int c8 = 0; c8 < 4; ++c8) {
    float x[8];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const float4 bb = b4[2 * c8 + h];
      const float a0 = __uint_as_float(r[8 * c8 + 4 * h + 0]), a1 = __uint_as_float(r[8 * c8 + 4 * h + 1]);
      const float a2 = __uint_as_float(r[8 * c8 + 4 * h + 2]), a3 = __uint_as_float(r[8 * c8 + 4 * h + 3]);
      if (EPI == kEpiAdd) {
        x[4 * h + 0] = (a0 + bb.x) + radd;
        x[4 * h + 1] = (a1 + bb.y) + radd;
        x[4 * h + 2] = (a2 + bb.z) + radd;
        x[4 * h + 3] = (a3 + bb.w) + radd;
      } else if (EPI == kEpiLean) {
        x[4 * h + 0] = fmaxf(a0 + bb.x, relu_lo) + radd;
        x[4 * h + 1] = fmaxf(a1 + bb.y, relu_lo) + radd;
        x[4 * h + 2] = fmaxf(a2 + bb.z, relu_lo) + radd;
        x[4 * h + 3] = fmaxf(a3 + bb.w, relu_lo) + radd;
      } else {
        const float4 ss = s4[2 * c8 + h], oo = o4[2 * c8 + h];
        x[4 * h + 0] = fmaf(fmaxf(a0 + bb.x, relu_lo), ss.x, oo.x);
        x[4 * h + 1] = fmaf(fmaxf(a1 + bb.y, relu_lo), ss.y, oo.y);
        x[4 * h + 2] = fmaf(fmaxf(a2 + bb.z, relu_lo), ss.z, oo.z);
        x[4 * h + 3] = fmaf(fmaxf(a3 + bb.w, relu_lo), ss.w, oo.w);
      }
    }
    if (OUT_BF16) {
      val[c8] = make_uint4(pack_bf16x2(x[0], x[1]), pack_bf16x2(x[2], x[3]), pack_bf16x2(x[4], x[5]),
                           pack_bf16x2(x[6], x[7]));
    } else {
      val[2 * c8] = make_uint4(__float_as_uint(x[0]), __float_as_uint(x[1]), __float_as_uint(x[2]), __float_as_uint(x[3]));
      val[2 * c8 + 1] = make_uint4(__float_as_uint(x[4]), __float_as_uint(x[5]), __float_as_uint(x[6]), __float_as_uint(x[7]));
    }
  }
  constexpr bool kOpens = !OUT_BF16 || HALF == 0;      // this chunk writes the first bytes of the box
  constexpr bool kCloses = !OUT_BF16 || HALF == 1;     // ... the last ones: the box leaves
  if (kOpens && tma_pending) {                         // the box's previous store has finished reading it
    if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;\n" ::: "memory");
    tma_pending = false;
    __syncwarp();
  }
  uint4* mine = reinterpret_cast<uint4*>(stg + lane * kBoxRow);
  const int wsw = lane & 7;
#pragma unroll
  for (int g = 0; g < kVals; ++g) mine[((OUT_BF16 ? HALF * 4 : 0) + g) ^ wsw] = val[g];
  if (!kCloses) return;
  if (tma) {
    fence_proxy_async_smem();
    __syncwarp();
    if (lane == 0 && !(dbg & 4)) {                     // (ablation bit 4: boxes are filled but never leave)
      if (store_policy != 0ull) tma_store_2d_hint(tmC, stg, tma_col, tma_row, store_policy);
      else tma_store_2d(tmC, stg, tma_col, tma_row);
    }
    tma_pending = true;
    return;
  }
  __syncwarp();
#pragma unroll 2
  for (int j = 0; j < 8; ++j) {                        // 32 rows x 8 pieces, a lane moves one 16-byte piece per step
    const int q = j * 32 + lane, rr = q >> 3, part = q & 7;
    const uint4 v = *reinterpret_cast<const uint4*>(stg + rr * kBoxRow + ((part ^ (rr & 7)) * 16));
    unsigned char* dst = out_box + rr * ld_bytes + part * 16;
    const int f = __shfl_sync(0xffffffffu, flags, rr);
    if (f & kRowStore) {
      *reinterpret_cast<uint4*>(dst) = v;
      if (f & (kRowFirst | kRowLast)) {
        const int lo = (f & kRowFirst) ? kHalo : 0, hi = (f & kRowLast) ? kHalo : 0;
#pragma unroll 1
        for (int h = -lo; h <= hi; ++h)
          if (h != 0) *reinterpret_cast<uint4*>(dst + h * ld_bytes) = v;
      }
    }
  }
  __syncwarp();
}

// Ragged / unaligned chunk of the pair kernel (right edge of the matrix, output pitch not a multiple of 16 bytes): fp32
// staging, bounds-checked scalar stores with the per-row flags.  Same arithmetic (and association) as store_box.
template <bool OUT_BF16, int VSTRIDE>
__device__ __forceinline__ void store_chunk_ragged(const unsigned (&r)[32], const float* vb, bool lean, float relu_lo,
                                                   float radd, unsigned char* stg, int lane, int flags, unsigned char* out0,
                                                   long long ld_bytes, int cols_left) {
  constexpr int kCols = 16;                              // columns per pass (kStgPitch = 80 bytes holds 16 floats + pad)
  constexpr int kEs = OUT_BF16 ? 2 : 4;
#pragma unroll      // (compile-time indices into r[]: a rolled loop would push the accumulator registers to local memory)
  for (int pass = 0; pass < 32 / kCols; ++pass) {
    float* mine = reinterpret_cast<float*>(stg + lane * kStgPitch);
#pragma unroll
    for (int i = 0; i < kCols; ++i) {
      const int c = pass * kCols + i;
      const float b = vb[c], sc = lean ? 1.0f : vb[VSTRIDE + c], of = lean ? 0.0f : vb[2 * VSTRIDE + c];
      const float t = fmaxf(__uint_as_float(r[c]) + b, relu_lo);
      mine[i] = (lean ? t : fmaf(t, sc, of)) + radd;
    }
    __syncwarp();
#pragma unroll 1
    for (int k = lane; k < 32 * kCols; k += 32) {
      const int rr = k / kCols, col = k % kCols;
      const float v = *reinterpret_cast<const float*>(stg + rr * kStgPitch + col * 4);
      const int f = __shfl_sync(0xffffffffu, flags, rr);
      if ((f & kRowStore) && pass * kCols + col < cols_left) {
        const int lo = (f & kRowFirst) ? kHalo : 0, hi = (f & kRowLast) ? kHalo : 0;
        unsigned char* dst = out0 + rr * ld_bytes + (long long)(pass * kCols + col) * kEs;
#pragma unroll 1
        for (int h = -lo; h <= hi; ++h) {
          if (OUT_BF16) *reinterpret_cast<__nv_bfloat16*>(dst + h * ld_bytes) = __float2bfloat16_rn(v);
          else *reinterpret_cast<float*>(dst + h * ld_bytes) = v;
        }
      }
    }
    __syncwarp();
  }
}

// Tile walk: row-storing modes go n-fastest (the n-tiles of one row block run on neighbouring CTAs and
// share the activation rows through L2); STATS goes m-fastest (the unit tiles of one frame block).
template <int MODE>
__device__ __forceinline__ void tile_coords(long long tile64, long long m_tiles64, int n_tiles, int reverse, int group_m,
                                            long long& mt, int& nt) {
  // tile counts fit 32 bits (2^31 tiles of 128 x 256 outputs is 10^14 elements): 32-bit divisions, not 64-bit ones --
  // every epilogue thread runs this twice per tile
  const unsigned m_tiles = (unsigned)m_tiles64, nt_n = (unsigned)n_tiles;
  unsigned tile = (unsigned)tile64;
  if (reverse) tile = m_tiles * nt_n - 1u - tile;
  if (MODE == kModeStats) {
    const unsigned q = tile / m_tiles;
    mt = tile - q * m_tiles;
    nt = (int)q;
  } else if (group_m > 1) {
    // grouped walk for wide outputs (PLDA: 196 n-tiles): the 148 CTAs of a wave cover group_m row blocks x ~148 /
    // group_m column blocks, so a wave re-uses its B tiles group_m times while they are hot and the whole B operand is
    // swept once per group_m row blocks instead of once per row block (it has to survive in L2 against the output stream)
    const unsigned per = (unsigned)group_m * nt_n;
    const unsigned g = tile / per, r = tile - g * per;
    const unsigned m_in = min((unsigned)group_m, m_tiles - g * (unsigned)group_m);
    const unsigned q = r / m_in;
    nt = (int)q;
    mt = g * (unsigned)group_m + (r - q * m_in);
  } else {
    const unsigned q = tile / nt_n;
    mt = q;
    nt = (int)(tile - q * nt_n);
  }
}

template <int MODE>
__global__ void __launch_bounds__(kThreadsTc, 1)
tdnn_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
               const __grid_constant__ CUtensorMap tmC, const TcArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  // 1024-byte alignment for the 128B swizzle; offsetting the __shared__ array (instead of rounding a generic
  // pointer) keeps the address space visible to the compiler, so the epilogue reads are LDS, not generic LD.
  unsigned char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  unsigned char* sA = smem;
  unsigned char* sB = smem + kStages * kABytes;
  unsigned char* s_stg = smem + kStages * kStageBytes;   // [kEpiWarps][32][kStgPitch], 512-byte aligned (TMA store source)
  unsigned long long* bars = reinterpret_cast<unsigned long long*>(smem + kStages * kStageBytes + kStgBytes);
  unsigned long long* full_bar = bars;                       // [kStages]
  unsigned long long* empty_bar = bars + kStages;            // [kStages]
  unsigned long long* tfull_bar = bars + 2 * kStages;        // [kAccStages]
  unsigned long long* tempty_bar = tfull_bar + kAccStages;   // [kAccStages]
  unsigned* tmem_slot = reinterpret_cast<unsigned*>(tempty_bar + kAccStages);
  float* s_vec = reinterpret_cast<float*>(smem + kStages * kStageBytes + kStgBytes + 256);  // [kAccStages][3][BN]
  int* s_seg = reinterpret_cast<int*>(smem + kStages * kStageBytes + kStgBytes + 256 + kVecBytes);  // [kAccStages][BN]

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  long long m_rows = a.m_rows, n_rows = a.n_rows;
  if (a.rows_dev != nullptr) {
    const long long actual = *a.rows_dev;
    if (a.shift_b) n_rows = min(n_rows, actual); else m_rows = min(m_rows, actual);
  }
  const long long act_rows = a.rows_dev != nullptr ? (a.shift_b ? n_rows : m_rows) : a.act_rows;
  const long long m_tiles = (m_rows + BM - 1) / BM;
  const int n_tiles = (int)((n_rows + BN - 1) / BN);
  const long long total_tiles = m_tiles * n_tiles;
  const int num_kb = a.num_taps * a.kblocks_per_tap;

  if (threadIdx.x == 0) {
    for (int s = 0; s < kStages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int s = 0; s < kAccStages; ++s) {
      mbar_init(&tfull_bar[s], 1);
      mbar_init(&tempty_bar[s], kEpiWarps);
    }
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(smem_u32(tmem_slot)),
                 "r"(kAccStages * BN));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const unsigned tmem_base = *tmem_slot;

  if (warp == 0) {
    // ================= TMA producer =================
    if (lane == 0) {
      asm volatile("prefetch.tensormap [%0];\n" ::"l"(&tmA) : "memory");
      asm volatile("prefetch.tensormap [%0];\n" ::"l"(&tmB) : "memory");
      if (a.tma_store) asm volatile("prefetch.tensormap [%0];\n" ::"l"(&tmC) : "memory");
      int stage = 0;
      unsigned phase = 0;
      const unsigned long long keep = a.l2_stream_out ? l2_policy_evict_last() : 0ull;
      for (long long tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
        long long mt;
        int nt;
        tile_coords<MODE>(tile, m_tiles, n_tiles, a.reverse, a.group_m, mt, nt);
        const int m0 = (int)(mt * BM), n0 = nt * BN;
        if (a.act_base != nullptr && tile + gridDim.x < total_tiles) {
          long long mt2;
          int nt2;
          tile_coords<MODE>(tile + gridDim.x, m_tiles, n_tiles, a.reverse, a.group_m, mt2, nt2);
          // one CTA per activation row block issues the prefetch (the block is shared by the n- / m-tiles)
          const bool mine = a.shift_b ? (mt2 == 0) : (nt2 == 0);
          if (mine) {
            const long long span = a.shift_b ? BN : BM;
            long long r0 = (a.shift_b ? (long long)nt2 * BN : mt2 * BM) - kHalo;
            long long r1 = r0 + span + 2 * kHalo;
            r0 = r0 < 0 ? 0 : r0;
            r1 = r1 > act_rows ? act_rows : r1;
            if (r1 > r0)
              bulk_prefetch_l2(static_cast<const unsigned char*>(a.act_base) + r0 * a.act_ld_bytes,
                               (unsigned)((r1 - r0) * a.act_ld_bytes));
          }
        }
        for (int kb = 0; kb < num_kb; ++kb) {
          const int tap = kb / a.kblocks_per_tap;
          const int d0 = (kb - tap * a.kblocks_per_tap) * BK;
          const int wcol = tap * a.tap_cols + d0;          // column in the weight matrix
          mbar_wait(&empty_bar[stage], phase ^ 1);
          mbar_expect_tx(&full_bar[stage], kStageBytes);
          if (a.shift_b) {
            tma_load_2d(sA + stage * kABytes, &tmA, &full_bar[stage], wcol, m0);
            tma_load_2d(sB + stage * kBBytes, &tmB, &full_bar[stage], d0, n0 + a.ctx[tap]);
          } else if (keep != 0ull) {
            tma_load_2d_hint(sA + stage * kABytes, &tmA, &full_bar[stage], d0, m0 + a.ctx[tap], keep);
            tma_load_2d_hint(sB + stage * kBBytes, &tmB, &full_bar[stage], wcol, n0, keep);
          } else {
            tma_load_2d(sA + stage * kABytes, &tmA, &full_bar[stage], d0, m0 + a.ctx[tap]);
            tma_load_2d(sB + stage * kBBytes, &tmB, &full_bar[stage], wcol, n0);
          }
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ================= MMA issuer =================
    if (lane == 0) {
      // instruction descriptor: D fp32, A/B bf16 (format 1) or fp16 (format 0), both K-major, N, M
      const unsigned fmt = a.fp16 ? 0u : 1u;
      const unsigned idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | ((unsigned)(BN >> 3) << 17) |
                             ((unsigned)(BM >> 4) << 24);
      int stage = 0;
      unsigned phase = 0;
      int it = 0;
      for (long long tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
        const int acc = it & 1;
        const unsigned acc_phase = (unsigned)(it >> 1) & 1u;
        mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
        tc_fence_after();
        const unsigned tmem_d = tmem_base + (unsigned)(acc * BN);
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const unsigned long long adesc = umma_desc(smem_u32(sA + stage * kABytes));
          const unsigned long long bdesc = umma_desc(smem_u32(sB + stage * kBBytes));
#pragma unroll
          for (int k = 0; k < BK / 16; ++k) {
            // advance 16 elements = 32 bytes inside the swizzled row: +2 in the (addr >> 4) field
            umma_f16(tmem_d, adesc + (unsigned long long)(2 * k), bdesc + (unsigned long long)(2 * k), idesc,
                     (kb > 0 || k > 0) ? 1u : 0u);
          }
          umma_commit(&empty_bar[stage]);     // frees the smem slot once these MMAs have read it
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
        umma_commit(&tfull_bar[acc]);         // accumulator ready for the epilogue
      }
    }
  } else {
    // ================= epilogue warps (2..9) =================
    const int quarter = warp & 3;             // TMEM lane quarter this warp may access
    const int colq = (warp - 2) >> 2;         // which kEpiCols of the tile's 256 columns
    const int et = threadIdx.x - 64;          // 0..255
    int staged_nt0 = -1, staged_nt1 = -1;     // n-tile whose epilogue vectors sit in s_vec[0] / s_vec[1]
    bool tma_pending = false;                 // a TMA store of this warp may still be reading its staging buffer
    const unsigned long long store_policy = a.l2_stream_out ? l2_policy_evict_first() : 0ull;
    const CUtensorMap* tmc = a.tma_store ? &tmC : nullptr;
    float pre_b = 0.0f, pre_s = 1.0f, pre_o = 0.0f;   // column (nt * BN + et) of bias / scale / offset, prefetched
    int pre_nt = -1;
    auto prefetch_vec = [&](int nt_) {
      if (MODE != kModeStats && et < BN) {
        const int col = nt_ * BN + et;
        const bool ok = col < n_rows;
        pre_b = (ok && a.bias) ? a.bias[col] : 0.0f;
        pre_s = (ok && a.scale) ? a.scale[col] : 1.0f;
        pre_o = (ok && a.offset) ? a.offset[col] : 0.0f;
      }
      pre_nt = nt_;
    };
    int it = 0;
    for (long long tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
      long long mt;
      int nt;
      tile_coords<MODE>(tile, m_tiles, n_tiles, a.reverse, a.group_m, mt, nt);
      const int col_base = nt * BN;
      const int acc = it & 1;
      const unsigned acc_phase = (unsigned)(it >> 1) & 1u;
      const long long row = mt * BM + quarter * 32 + lane;
      const unsigned taddr0 =
          tmem_base + ((unsigned)(quarter * 32) << 16) + (unsigned)(acc * BN) + (unsigned)(colq * kEpiCols);

      if (MODE == kModeStats) {
        // ---- per-unit running sums over the frames of the tile (stats_pooling.py:228-240) ----
        int* seg = s_seg + acc * BN;
        if (et < BN) {
          const long long fr = (long long)col_base + et;
          seg[et] = (fr < n_rows) ? a.rowseg[fr] : -1;
        }
        const bool unit_ok = row < m_rows;
        const float b = (unit_ok && a.bias) ? a.bias[row] : 0.0f;
        // the sums are of r - c (TcLayer::d_shift), computed as max(acc + (b - c), lo - c): no instruction per frame
        const float ctr = (unit_ok && a.shift) ? a.shift[row] : 0.0f;
        const float bc = b - ctr;
        const float relu_lo = a.relu ? -ctr : -3.402823466e+38f;
        asm volatile("bar.sync 1, 256;\n" ::: "memory");
        mbar_wait(&tfull_bar[acc], acc_phase);
        tc_fence_after();

        const int* sg = seg + colq * kEpiCols;
        float s = 0.0f, s2 = 0.0f;
        int cur = -1;
        auto flush = [&]() {
          if (cur >= 0 && unit_ok) {
            atomicAdd(a.sums + ((long long)cur * 2 + 0) * m_rows + row, s);
            atomicAdd(a.sums + ((long long)cur * 2 + 1) * m_rows + row, s2);
          }
        };
        unsigned r[2][32];
        tmem_ld32_issue(taddr0, r[0]);
#pragma unroll
        for (int c = 0; c < kEpiChunks; ++c) {
          tmem_ld_wait(r[c & 1]);
          if (c + 1 < kEpiChunks) tmem_ld32_issue(taddr0 + (unsigned)((c + 1) * 32), r[(c + 1) & 1]);
          const int* sc = sg + c * 32;
          const int first = sc[0], last = sc[31];
          if (first == last && first >= 0) {   // warp-uniform: the whole chunk lies inside one utterance
            if (first != cur) { flush(); cur = first; s = 0.0f; s2 = 0.0f; }
#pragma unroll
            for (int i = 0; i < 32; ++i) {
              const float t = fmaxf(__uint_as_float(r[c & 1][i]) + bc, relu_lo);
              s += t;
              s2 = fmaf(t, t, s2);
            }
          } else {                             // utterance boundary / halo rows inside the chunk
#pragma unroll
            for (int i = 0; i < 32; ++i) {
              const int u = sc[i];
              if (u >= 0) {
                if (u != cur) { flush(); cur = u; s = 0.0f; s2 = 0.0f; }
                const float t = fmaxf(__uint_as_float(r[c & 1][i]) + bc, relu_lo);
                s += t;
                s2 = fmaf(t, t, s2);
              }
            }
          }
        }
        flush();
      } else {
        // ---- bias / ReLU / BatchNorm per column, rows stored as bf16 or fp32 ----
        float* vb = s_vec + acc * 3 * BN;
        // The per-column vectors of an n-tile are staged once per accumulator stage and reused while the
        // CTA keeps drawing the same n-tile (always, when gridDim.x is a multiple of n_tiles).
        const int have_nt = acc ? staged_nt1 : staged_nt0;
        if (have_nt != nt) {                                 // uniform over all epilogue threads
          if (pre_nt != nt) prefetch_vec(nt);                 // normally issued one tile earlier (see below)
          asm volatile("bar.sync 1, 256;\n" ::: "memory");    // every warp is done reading the old vectors
          if (et < BN) {
            vb[et] = pre_b;
            vb[BN + et] = pre_s;
            vb[2 * BN + et] = pre_o;
          }
          asm volatile("bar.sync 1, 256;\n" ::: "memory");
          if (acc) staged_nt1 = nt; else staged_nt0 = nt;
        }
        {
          // the next tile's per-column vectors: global loads issued now, consumed after this tile's stores
          const long long next = tile + gridDim.x;
          if (next < total_tiles) {
            long long mt2;
            int nt2;
            tile_coords<MODE>(next, m_tiles, n_tiles, a.reverse, a.group_m, mt2, nt2);
            const int have2 = acc ? staged_nt0 : staged_nt1;   // the next tile uses the other accumulator stage
            if (have2 != nt2 && pre_nt != nt2) prefetch_vec(nt2);
          }
        }
        int flags = 0;
        if (row < m_rows) flags = a.rowmap ? a.rowmap[row] : kRowStore;
        if (a.debug & 1) flags = 0;
        const bool plain = __all_sync(0xffffffffu, (flags & kRowFlagMask) == kRowStore);
        float radd = 0.0f;
        if (a.row_add != nullptr && row < m_rows) radd = a.row_add[row];
        mbar_wait(&tfull_bar[acc], acc_phase);
        tc_fence_after();

        const int n_cols = (int)n_rows;
        constexpr bool kBf16 = (MODE == kModeBf16);
        constexpr int kEs = kBf16 ? 2 : 4;                   // output element size
        const long long ld_bytes = a.out_ld * kEs;
        unsigned char* owarp = reinterpret_cast<unsigned char*>(a.out) + (mt * BM + quarter * 32) * ld_bytes;
        unsigned char* stg = s_stg + (warp - 2) * (32 * kStgPitch);
        const bool vec_ok = ((reinterpret_cast<unsigned long long>(a.out) | (unsigned long long)ld_bytes) & 15ull) == 0;
        const float relu_lo = a.relu ? 0.0f : -3.402823466e+38f;
        unsigned r[2][32];                                // TMEM loads run one chunk ahead of the math / stores
        tmem_ld32_issue(taddr0, r[0]);
#pragma unroll
        for (int c = 0; c < kEpiChunks; ++c) {
          tmem_ld_wait(r[c & 1]);
          if (c + 1 < kEpiChunks) tmem_ld32_issue(taddr0 + (unsigned)((c + 1) * 32), r[(c + 1) & 1]);
          const int cc = colq * kEpiCols + c * 32;        // column offset inside the tile
          const int col0 = col_base + cc;
          if (col0 >= n_cols || (a.debug & 2)) continue;  // warp-uniform
          unsigned char* out0 = owarp + (long long)col0 * kEs;
          const int trow = (int)(mt * BM) + quarter * 32;
          if (vec_ok && col0 + 32 <= n_cols)
            store_chunk<kBf16, true>(r[c & 1], vb + cc, relu_lo, radd, stg, lane, flags, plain, out0, ld_bytes, 32, tmc,
                                     col0, trow, tma_pending, store_policy);
          else
            store_chunk<kBf16, false>(r[c & 1], vb + cc, relu_lo, radd, stg, lane, flags, false, out0, ld_bytes,
                                      n_cols - col0, nullptr, 0, 0, tma_pending, 0ull);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty_bar[acc]);
    }
    if (tma_pending && lane == 0) tma_store_wait_read();   // shared memory must outlive the last box
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(tmem_base), "r"(kAccStages * BN));
  }
}

// ---------------------------------------------------------------------------------------------------
// CTA-pair variant (tcgen05 cta_group::2) of the row-storing modes: two CTAs of one cluster (the two SMs of a TPC)
// compute a 256 x 256 tile -- each CTA owns 128 rows of A and of the accumulator and loads only HALF of B (128 of the
// 256 columns); the MMA, issued by the leader CTA alone, reads both halves.  Per CTA a k-block is 16 KB + 16 KB instead
// of 16 KB + 32 KB: a third less operand traffic per output tile, and the ring holds kPairStages = 5 k-blocks in 160 KB,
// which leaves room for double-buffered staging (the boxed store of pass p is still reading its buffer while pass p + 1
// is being written).
//   barriers (same offsets in both CTAs): full[s] lives in the LEADER (2 arrivals: each producer; 64 KB of TMA bytes from
//   both CTAs complete on it), empty[s] and tfull[acc] are signalled in both CTAs by a multicast tcgen05.commit,
//   tempty[acc] lives in the leader (2 x kEpiWarps arrivals, the peer's epilogue warps arrive through the cluster).
// ---------------------------------------------------------------------------------------------------
constexpr int kPairABytes = BM * BK * 2;                 // 16 KB: this CTA's 128 rows
constexpr int kPairBBytes = (BN / 2) * BK * 2;           // 16 KB: this CTA's 128 of the tile's 256 columns
constexpr int kPairStageBytes = kPairABytes + kPairBBytes;
// EW epilogue warps per CTA (8 or 16: EW / 4 warps share a TMEM lane quarter and split the tile's 256 columns).  A thread
// owns one accumulator row and walks TMEM load -> per-column vectors -> staging box -> boxed store; 16 warps double the
// chains in flight and pay for it with one ring stage (4 x 32 KB instead of 5) and 96 registers per thread.  Which one a
// launch gets: pair_epi_warps().
template <int EW> struct PairCfg {
  static constexpr int kStages = EW == 16 ? 4 : 5;
  static constexpr int kThreads = 64 + EW * 32;
  static constexpr int kCols = BN / (EW / 4);              // tile columns per epilogue warp: 128 or 64
  static constexpr int kChunks = kCols / 32;
  static constexpr int kStgBytes = EW * kBoxBytes;         // one 32-row x 128-byte staging box per epilogue warp
  static constexpr int kVecBytes = EW * 3 * kCols * 4;     // per-warp [bias | scale | offset] of the warp's columns
  static constexpr int kSmem = kStages * kPairStageBytes + 1024 + 256 + kVecBytes + kStgBytes;
};
static_assert(PairCfg<8>::kSmem <= 226 * 1024 && PairCfg<16>::kSmem <= 226 * 1024, "pair kernel shared memory");
// Top-k modes store nothing: no staging boxes, only the bias of the per-warp vectors.  What they hold instead: per thread
// a list of CAP 64-bit keys (interleaved by thread, so any per-lane entry index is bank-conflict free) and per warp a
// 16 x 32 float scratch through which a lane walks its candidates of half a chunk.  The ring gets what is left, at most
// the 5 stages of the storing modes.  EW = 8: CAP 8 / 16 / 32 -> 16 / 32 / 64 KB of lists, 5 / 5 / 4 stages;
// EW = 16: 32 / 64 / 128 KB, 4 / 3 / 1 stages.
template <int EW, int CAP> struct TopkCfg {
  static constexpr int kCols = BN / (EW / 4);
  static constexpr int kVecBytes = EW * kCols * 4;
  static constexpr int kScratchBytes = EW * 16 * 32 * 4;
  static constexpr int kListBytes = EW * 32 * CAP * 8;
  static constexpr int kFixed = 1024 + 256 + kVecBytes + kScratchBytes + kListBytes;
  static constexpr int kStages = std::min(5, (226 * 1024 - kFixed) / kPairStageBytes);
  static constexpr int kSmem = kStages * kPairStageBytes + kFixed;
};
static_assert(TopkCfg<8, 32>::kStages == 4 && TopkCfg<16, 32>::kStages >= 1, "top-k pair kernel shared memory");
template <int MODE, int EW>
constexpr int pair_smem() { return topk_cap(MODE) ? TopkCfg<EW, topk_cap(MODE) ? topk_cap(MODE) : 8>::kSmem : PairCfg<EW>::kSmem; }

__device__ __forceinline__ unsigned cluster_ctarank() {
  unsigned r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;\n" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\nbarrier.cluster.wait.acquire.aligned;\n" ::: "memory");
}
__device__ __forceinline__ unsigned mapa_u32(unsigned addr, unsigned rank) {
  unsigned r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;\n" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
// Remote arrive WITHOUT release semantics: what it orders (TMEM reads before the accumulator is overwritten, the TMA
// issue order) is covered by tcgen05.fence / the barrier protocol; a cluster-scope release would also wait for the
// warp's outstanding global stores on every tile.
__device__ __forceinline__ void mbar_arrive_cluster(unsigned cluster_addr) {
  asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];\n" ::"r"(cluster_addr) : "memory");
}
// TMA load whose completion bytes are counted on a barrier that may live in the peer CTA (cluster address)
__device__ __forceinline__ void tma_load_2d_pair(void* smem_dst, const CUtensorMap* map, unsigned bar_cluster_addr, int c0,
                                                 int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], "
      "[%2];\n" ::"r"(smem_u32(smem_dst)),
      "l"(map), "r"(bar_cluster_addr), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void umma_f16_pair(unsigned tmem_d, unsigned long long adesc, unsigned long long bdesc,
                                              unsigned idesc, unsigned accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit_pair(unsigned long long* bar) {   // arrives on `bar` in BOTH CTAs
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;\n" ::"r"(
          smem_u32(bar)),
      "h"((unsigned short)3)
      : "memory");
}

template <int MODE, int EW>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(PairCfg<EW>::kThreads, 1)
tdnn_tc_pair_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                    const __grid_constant__ CUtensorMap tmC, const TcArgs a) {
  static_assert(MODE != kModeStats, "the pair kernel covers the row-storing modes");
  using Cfg = PairCfg<EW>;
  constexpr int kCap = topk_cap(MODE);
  constexpr bool kTopk = kCap > 0;
  using TCfg = TopkCfg<EW, kTopk ? kCap : 8>;
  constexpr int kPairStages = kTopk ? TCfg::kStages : Cfg::kStages;
  constexpr int kPCols = Cfg::kCols, kPChunks = Cfg::kChunks;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  unsigned char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  unsigned char* sA = smem;
  unsigned char* sB = smem + kPairStages * kPairABytes;
  unsigned char* s_stg = smem + kPairStages * kPairStageBytes;          // [EW] boxes of 32 rows x 128 bytes (1024-byte aligned)
  // (top-k: [EW] candidate scratches, then the lists)
  unsigned long long* bars =
      reinterpret_cast<unsigned long long*>(s_stg + (kTopk ? TCfg::kScratchBytes + TCfg::kListBytes : Cfg::kStgBytes));
  unsigned long long* full_bar = bars;                        // [kPairStages]   (used in the leader)
  unsigned long long* empty_bar = bars + kPairStages;         // [kPairStages]
  unsigned long long* tfull_bar = bars + 2 * kPairStages;     // [kAccStages]
  unsigned long long* tempty_bar = tfull_bar + kAccStages;    // [kAccStages]    (used in the leader)
  unsigned* tmem_slot = reinterpret_cast<unsigned*>(tempty_bar + kAccStages);
  float* s_vec = reinterpret_cast<float*>(reinterpret_cast<unsigned char*>(bars) + 256);   // [EW][3][kPCols]

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const unsigned rank = cluster_ctarank();                   // 0 = leader
  const long long cluster_id = blockIdx.x >> 1, num_clusters = gridDim.x >> 1;
  long long m_rows = a.m_rows;
  const long long n_rows = a.n_rows;
  if (a.rows_dev != nullptr) m_rows = min(m_rows, *a.rows_dev);
  constexpr int BM2 = 2 * BM;                                 // rows of a pair tile
  const long long m_tiles = (m_rows + BM2 - 1) / BM2;
  const int n_tiles = (int)((n_rows + BN - 1) / BN);
  const long long total_tiles = m_tiles * n_tiles;
  const int num_kb = a.num_taps * a.kblocks_per_tap;
  // top-k: the cluster runs units cluster_id, cluster_id + num_clusters, ... whole; unit u = split * m_tiles + row block
  // (split-major: the clusters running at the same time sweep the same range of B).  Every unit has unit_tiles n-tiles;
  // those of the last split past the matrix only load zeros (out-of-bounds boxes) and hold no candidates.
  const unsigned unit_tiles = kTopk ? (unsigned)a.topk_unit_tiles : 1u;
  const long long topk_units = kTopk ? m_tiles * (((long long)n_tiles + unit_tiles - 1) / unit_tiles) : 0;
  const long long topk_mine = cluster_id < topk_units ? (topk_units - 1 - cluster_id) / num_clusters + 1 : 0;
  const long long t_begin = kTopk ? 0 : cluster_id;                                    // this cluster's tiles
  const long long t_end = kTopk ? topk_mine * unit_tiles : total_tiles, t_step = kTopk ? 1 : num_clusters;
  auto topk_unit = [&](long long tile_) { return (unsigned)cluster_id + ((unsigned)tile_ / unit_tiles) * (unsigned)num_clusters; };
  auto coords = [&](long long tile_, long long& mt_, int& nt_) {
    if constexpr (kTopk) {
      const unsigned u = topk_unit(tile_), s = u / (unsigned)m_tiles;
      mt_ = u - s * (unsigned)m_tiles;
      nt_ = (int)(s * unit_tiles + (unsigned)tile_ % unit_tiles);
    } else {
      tile_coords<MODE>(tile_, m_tiles, n_tiles, a.reverse, a.group_m, mt_, nt_);
    }
  };

  if (threadIdx.x == 0) {
    for (int s = 0; s < kPairStages; ++s) {
      mbar_init(&full_bar[s], 2);
      mbar_init(&empty_bar[s], 1);
    }
    for (int s = 0; s < kAccStages; ++s) {
      mbar_init(&tfull_bar[s], 1);
      mbar_init(&tempty_bar[s], 2 * EW);
    }
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(smem_u32(tmem_slot)),
                 "r"(kAccStages * BN));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;\n");
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();                                        // both CTAs' barriers exist before any remote arrive
  tc_fence_after();
  const unsigned tmem_base = *tmem_slot;

  if (warp == 0) {
    // ================= TMA producer (both CTAs) =================
    if (lane == 0) {
      asm volatile("prefetch.tensormap [%0];\n" ::"l"(&tmA) : "memory");
      asm volatile("prefetch.tensormap [%0];\n" ::"l"(&tmB) : "memory");
      if (a.tma_store) asm volatile("prefetch.tensormap [%0];\n" ::"l"(&tmC) : "memory");
      int stage = 0;
      unsigned phase = 0;
      for (long long tile = t_begin; tile < t_end; tile += t_step) {
        long long mt;
        int nt;
        coords(tile, mt, nt);
        const int m0 = (int)(mt * BM2) + (int)rank * BM, n0 = nt * BN + (int)rank * (BN / 2);
        if (a.act_base != nullptr && rank == 0 && tile + t_step < t_end) {
          long long mt2;
          int nt2;
          coords(tile + t_step, mt2, nt2);
          if (nt2 == 0) {                                    // one cluster per row block requests it for all its n-tiles
            long long r0 = mt2 * BM2 - kHalo, r1 = r0 + BM2 + 2 * kHalo;
            r0 = r0 < 0 ? 0 : r0;
            r1 = r1 > m_rows ? m_rows : r1;
            if (r1 > r0)
              bulk_prefetch_l2(static_cast<const unsigned char*>(a.act_base) + r0 * a.act_ld_bytes,
                               (unsigned)((r1 - r0) * a.act_ld_bytes));
          }
        }
        for (int kb = 0; kb < num_kb; ++kb) {
          const int tap = kb / a.kblocks_per_tap;
          const int d0 = (kb - tap * a.kblocks_per_tap) * BK;
          const int wcol = tap * a.tap_cols + d0;
          mbar_wait(&empty_bar[stage], phase ^ 1);
          const unsigned full_leader = mapa_u32(smem_u32(&full_bar[stage]), 0);
          // both CTAs' bytes land on the leader's barrier
          if (rank == 0) mbar_expect_tx(&full_bar[stage], 2 * kPairStageBytes);
          else mbar_arrive_cluster(full_leader);
          tma_load_2d_pair(sA + stage * kPairABytes, &tmA, full_leader, d0, m0 + a.ctx[tap]);
          tma_load_2d_pair(sB + stage * kPairBBytes, &tmB, full_leader, wcol, n0);
          if (++stage == kPairStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ================= MMA issuer (leader CTA only) =================
    if (lane == 0 && rank == 0) {
      const unsigned fmt = a.fp16 ? 0u : 1u;
      const unsigned idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | ((unsigned)(BN >> 3) << 17) |
                             ((unsigned)(BM2 >> 4) << 24);
      int stage = 0;
      unsigned phase = 0;
      int it = 0;
      for (long long tile = t_begin; tile < t_end; tile += t_step, ++it) {
        const int acc = it & 1;
        const unsigned acc_phase = (unsigned)(it >> 1) & 1u;
        mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
        tc_fence_after();
        if (a.trace != nullptr && cluster_id == 0 && it < 512) a.trace[4 * it + 0] = clock64();   // accumulator free
        const unsigned tmem_d = tmem_base + (unsigned)(acc * BN);
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          if (kb == num_kb - 1 && a.trace != nullptr && cluster_id == 0 && it < 512)
            a.trace[4 * it + 1] = clock64();                                                       // last operands landed
          const unsigned long long adesc = umma_desc(smem_u32(sA + stage * kPairABytes));
          const unsigned long long bdesc = umma_desc(smem_u32(sB + stage * kPairBBytes));
#pragma unroll
          for (int k = 0; k < BK / 16; ++k)
            umma_f16_pair(tmem_d, adesc + (unsigned long long)(2 * k), bdesc + (unsigned long long)(2 * k), idesc,
                          (kb > 0 || k > 0) ? 1u : 0u);
          umma_commit_pair(&empty_bar[stage]);   // both CTAs' producers may refill the slot
          if (++stage == kPairStages) { stage = 0; phase ^= 1; }
        }
        umma_commit_pair(&tfull_bar[acc]);       // both CTAs' epilogues may read their half of the accumulator
      }
    }
  } else {
    // ================= epilogue warps (2 .. EW + 1), each CTA drains its own 128 rows =================
    const int quarter = warp & 3;
    const int colq = (warp - 2) >> 2;
    bool tma_pending = false;
    const bool lean = a.scale == nullptr && a.offset == nullptr;   // launch-uniform: bias (+ ReLU, + row addend) only
    const unsigned long long store_policy = a.l2_stream_out ? l2_policy_evict_first() : 0ull;
    const CUtensorMap* tmc = a.tma_store ? &tmC : nullptr;
    const unsigned tempty_leader0 = mapa_u32(smem_u32(&tempty_bar[0]), 0), tempty_leader1 = mapa_u32(smem_u32(&tempty_bar[1]), 0);
    // Per-column vectors of the warp's 128 columns live in a region PRIVATE to the warp (no CTA-wide barrier when the
    // n-tile changes -- in PLDA scoring it changes on every tile): lane l owns columns 4l .. 4l+3, the next tile's values
    // are loaded into registers one tile ahead.
    float* wv = s_vec + (warp - 2) * ((kTopk ? 1 : 3) * kPCols);
    // top-k: this thread's list (entry i at s_list[i * kNT + et]: interleaved by thread), its fill, the entry holding its
    // smallest key and that key's value, the bar every later candidate has to pass (-inf while the list is not full)
    constexpr int kNT = EW * 32;
    const int et = threadIdx.x - 64;
    unsigned long long* s_list = reinterpret_cast<unsigned long long*>(s_stg + TCfg::kScratchBytes);
    float* scratch = reinterpret_cast<float*>(s_stg) + (warp - 2) * (16 * 32);
    int tk_cnt = 0, tk_min = 0;
    float tk_bar = -INFINITY;
    auto topk_insert = [&](float x, int col) {
      const int k = a.topk_k;
      const unsigned long long key = top1_key(x, col);
      if (tk_cnt < k) {
        s_list[tk_cnt * kNT + et] = key;
        if (++tk_cnt < k) return;
      } else {
        s_list[tk_min * kNT + et] = key;
      }
      unsigned long long lo = ~0ull;
#pragma unroll 4
      for (int i = 0; i < k; ++i) {
        const unsigned long long e = s_list[i * kNT + et];
        if (e < lo) { lo = e; tk_min = i; }
      }
      tk_bar = top1_key_value(lo);
    };
    constexpr int kVW = kPCols / 32;           // columns per lane: 4 (EW = 8) or 2 (EW = 16)
    int wv_nt = -1, pre_nt = -1;
    float pre_b[kVW], pre_s[kVW], pre_o[kVW];
#pragma unroll
    for (int u = 0; u < kVW; ++u) { pre_b[u] = 0.0f; pre_s[u] = 1.0f; pre_o[u] = 0.0f; }
    auto prefetch_vec = [&](int nt_) {
      const int col = nt_ * BN + colq * kPCols + kVW * lane;
#pragma unroll
      for (int u = 0; u < kVW; ++u) {
        const bool ok = col + u < n_rows;
        pre_b[u] = (ok && a.bias) ? a.bias[col + u] : 0.0f;
        if (!lean) {
          pre_s[u] = (ok && a.scale) ? a.scale[col + u] : 1.0f;
          pre_o[u] = (ok && a.offset) ? a.offset[col + u] : 0.0f;
        }
      }
      pre_nt = nt_;
    };
    int nx_flags = 0;
    float nx_radd = 0.0f;
    auto load_row_meta = [&](long long row_, int& f_, float& ra_) {
      f_ = 0;
      ra_ = 0.0f;
      if (row_ < m_rows) {
        f_ = a.rowmap ? a.rowmap[row_] : kRowStore;
        if (a.row_add != nullptr) ra_ = a.row_add[row_];
      }
    };
    int it = 0;
    for (long long tile = t_begin; tile < t_end; tile += t_step, ++it) {
      long long mt;
      int nt;
      coords(tile, mt, nt);
      const int col_base = nt * BN;
      const int acc = it & 1;
      const unsigned acc_phase = (unsigned)(it >> 1) & 1u;
      const long long row0 = mt * BM2 + (long long)rank * BM;             // first row of this CTA's half
      const long long row = row0 + quarter * 32 + lane;
      const unsigned taddr0 =
          tmem_base + ((unsigned)(quarter * 32) << 16) + (unsigned)(acc * BN) + (unsigned)(colq * kPCols);
      if (kTopk && (unsigned)tile % unit_tiles == 0) {   // a new unit: empty lists
        tk_cnt = 0;
        tk_bar = -INFINITY;
      }

      if (wv_nt != nt) {
        if (pre_nt != nt) prefetch_vec(nt);
        __syncwarp();                            // every lane is done reading the previous tile's vectors
#pragma unroll
        for (int u = 0; u < kVW; ++u) {
          wv[kVW * lane + u] = pre_b[u];
          if (!lean) {
            wv[kPCols + kVW * lane + u] = pre_s[u];
            wv[2 * kPCols + kVW * lane + u] = pre_o[u];
          }
        }
        __syncwarp();
        wv_nt = nt;
      }
      // this tile's row flags / row addend were requested one tile ahead (a global load in front of every tile was 9 % of
      // the stall samples); request the next tile's now
      int flags = nx_flags;
      float radd = nx_radd;
      if (it == 0) load_row_meta(row, flags, radd);
      {
        const long long next = tile + t_step;
        if (next < t_end) {
          long long mt2;
          int nt2;
          coords(next, mt2, nt2);
          if (nt2 != nt && pre_nt != nt2) prefetch_vec(nt2);
          load_row_meta(mt2 * BM2 + (long long)rank * BM + quarter * 32 + lane, nx_flags, nx_radd);
        }
      }
      mbar_wait(&tfull_bar[acc], acc_phase);
      tc_fence_after();
      if (a.trace != nullptr && cluster_id == 0 && rank == 0 && warp == 2 && lane == 0 && it < 512)
        a.trace[4 * it + 2] = clock64();                                                           // accumulator full
      if (a.debug & 1) flags = 0;
      // (the row map carries splice bookkeeping above bit 7: only the store / first / last bits decide the path)
      const bool plain = __all_sync(0xffffffffu, (flags & kRowFlagMask) == kRowStore);

      const int n_cols = (int)n_rows;
      constexpr bool kBf16 = (MODE == kModeBf16);
      constexpr int kEs = kBf16 ? 2 : 4;
      const long long ld_bytes = a.out_ld * kEs;
      unsigned char* owarp = reinterpret_cast<unsigned char*>(a.out) + (row0 + quarter * 32) * ld_bytes;
      unsigned char* stg2 = s_stg + (warp - 2) * kBoxBytes;
      const bool vec_ok = ((reinterpret_cast<unsigned long long>(a.out) | (unsigned long long)ld_bytes) & 15ull) == 0;
      const float relu_lo = a.relu ? 0.0f : -3.402823466e+38f;
      const int epi = lean ? (a.relu ? kEpiLean : kEpiAdd) : kEpiFull;   // launch-uniform
      // EW = 8: TMEM loads run one chunk ahead of the math (two register buffers); EW = 16 has the warps to cover the
      // load latency and 96 registers per thread: one buffer
      constexpr int kRB = EW == 16 ? 1 : 2;
      unsigned r[kRB][32];
      float best_v = -INFINITY;                  // (row_best launches) best entry of this row among the warp's columns
      int best_c = -1;
      tmem_ld32_issue(taddr0, r[0]);
#pragma unroll
      for (int c = 0; c < kPChunks; ++c) {
        tmem_ld_wait(r[c % kRB]);
        if (kRB == 2 && c + 1 < kPChunks) tmem_ld32_issue(taddr0 + (unsigned)((c + 1) * 32), r[(c + 1) % kRB]);
        const int col0 = col_base + colq * kPCols + c * 32;
        if constexpr (kTopk) {
          // the add-only form of the epilogue as below; a value enters the list only if it beats the list's smallest
          // entry (ties lose: every listed column is lower).  A lane with candidates in half a chunk parks the half in its
          // column of the warp's scratch and walks them there, so the warp pays for its busiest lane, not for every
          // column some lane wants to insert.
          const float4* b4 = reinterpret_cast<const float4*>(wv + c * 32);
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            float v[16];
            unsigned cand = 0;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              const float4 bb = b4[4 * h + q];
              v[4 * q + 0] = (__uint_as_float(r[c % kRB][16 * h + 4 * q + 0]) + bb.x) + radd;
              v[4 * q + 1] = (__uint_as_float(r[c % kRB][16 * h + 4 * q + 1]) + bb.y) + radd;
              v[4 * q + 2] = (__uint_as_float(r[c % kRB][16 * h + 4 * q + 2]) + bb.z) + radd;
              v[4 * q + 3] = (__uint_as_float(r[c % kRB][16 * h + 4 * q + 3]) + bb.w) + radd;
            }
#pragma unroll
            for (int j = 0; j < 16; ++j)
              if (col0 + 16 * h + j < n_cols && v[j] > tk_bar) cand |= 1u << j;
            if (cand != 0) {
#pragma unroll
              for (int j = 0; j < 16; ++j) scratch[j * 32 + lane] = v[j];
              while (cand != 0) {
                const int j = __ffs(cand) - 1;
                cand &= cand - 1;
                const float x = scratch[j * 32 + lane];
                if (x > tk_bar) topk_insert(x, col0 + 16 * h + j);
              }
            }
          }
          __syncwarp();                          // converged again before the next .sync.aligned TMEM load / wait
          if (kRB == 1 && c + 1 < kPChunks) tmem_ld32_issue(taddr0 + (unsigned)((c + 1) * 32), r[0]);
          continue;
        }
        if (a.row_best != nullptr) {
          // compact output: nothing is stored, the row keeps its best entry -- the add-only form of the epilogue, columns
          // in ascending order and a strict comparison, so the lowest column wins a tie
          const float4* b4 = reinterpret_cast<const float4*>(wv + c * 32);
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            const float4 bb = b4[q];
            const float v0 = (__uint_as_float(r[c % kRB][4 * q + 0]) + bb.x) + radd;
            const float v1 = (__uint_as_float(r[c % kRB][4 * q + 1]) + bb.y) + radd;
            const float v2 = (__uint_as_float(r[c % kRB][4 * q + 2]) + bb.z) + radd;
            const float v3 = (__uint_as_float(r[c % kRB][4 * q + 3]) + bb.w) + radd;
            const int cq = col0 + 4 * q;
            if (cq + 0 < n_cols && v0 > best_v) { best_v = v0; best_c = cq + 0; }
            if (cq + 1 < n_cols && v1 > best_v) { best_v = v1; best_c = cq + 1; }
            if (cq + 2 < n_cols && v2 > best_v) { best_v = v2; best_c = cq + 2; }
            if (cq + 3 < n_cols && v3 > best_v) { best_v = v3; best_c = cq + 3; }
          }
          if (kRB == 1 && c + 1 < kPChunks) tmem_ld32_issue(taddr0 + (unsigned)((c + 1) * 32), r[0]);
          continue;
        }
        // the 128-byte box this chunk belongs to: the chunk itself (fp32 rows) or a pair of chunks (bf16 rows)
        const int box_col0 = kBf16 ? col_base + colq * kPCols + (c & ~1) * 32 : col0;
        constexpr int kBoxCols = kBoxRow / kEs;
        if (col0 >= n_cols || (a.debug & 2)) {
          if (kRB == 1 && c + 1 < kPChunks) tmem_ld32_issue(taddr0 + (unsigned)((c + 1) * 32), r[0]);
          continue;
        }
        const int trow = (int)row0 + quarter * 32;
        if (vec_ok && box_col0 + kBoxCols <= n_cols) {
          unsigned char* out_box = owarp + (long long)box_col0 * kEs;
          const float* wvc = wv + c * 32;
#define KTF_STORE_BOX(EPI_, HALF_)                                                                                      \
  store_box<kBf16, EPI_, kPCols, HALF_>(r[c % kRB], wvc, relu_lo, radd, stg2, lane, flags, plain, out_box, ld_bytes, tmc, \
                                        box_col0, trow, tma_pending, store_policy, a.debug)
          if ((c & 1) == 0) {
            if (epi == kEpiFull) KTF_STORE_BOX(kEpiFull, 0);
            else if (epi == kEpiAdd) KTF_STORE_BOX(kEpiAdd, 0);
            else KTF_STORE_BOX(kEpiLean, 0);
          } else {
            if (epi == kEpiFull) KTF_STORE_BOX(kEpiFull, 1);
            else if (epi == kEpiAdd) KTF_STORE_BOX(kEpiAdd, 1);
            else KTF_STORE_BOX(kEpiLean, 1);
          }
#undef KTF_STORE_BOX
        } else {
          if (tma_pending) {                     // the ragged path reads back with the generic proxy: no box in flight
            if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;\n" ::: "memory");
            __syncwarp();
            tma_pending = false;
          }
          // (the warp's staging boxes serve as the fp32 staging of the ragged path)
          unsigned char* out0 = owarp + (long long)col0 * kEs;
          store_chunk_ragged<kBf16, kPCols>(r[c % kRB], wv + c * 32, lean, relu_lo, radd, stg2, lane, flags, out0, ld_bytes,
                                            n_cols - col0);
        }
        if (kRB == 1 && c + 1 < kPChunks) tmem_ld32_issue(taddr0 + (unsigned)((c + 1) * 32), r[0]);
      }
      if (a.row_best != nullptr && best_c >= 0 && row < m_rows) atomicMax(a.row_best + row, top1_key(best_v, best_c));
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (rank == 0) mbar_arrive(&tempty_bar[acc]);
        else mbar_arrive_cluster(acc ? tempty_leader1 : tempty_leader0);
        if (a.trace != nullptr && cluster_id == 0 && rank == 0 && warp == 2 && it < 512)
          a.trace[4 * it + 3] = clock64();                                                         // warp 2 drained its part
      }
      if (kTopk && (unsigned)tile % unit_tiles == unit_tiles - 1 && row < m_rows) {   // end of the unit: partial list out
        const int k = a.topk_k;
        const long long list = (long long)(topk_unit(tile) / (unsigned)m_tiles) * (EW / 4) + colq;
        float* os = a.topk_score + (list * m_rows + row) * k;
        long long* oi = a.topk_index + (list * m_rows + row) * k;
        for (int i = 0; i < k; ++i) {
          const unsigned long long key = i < tk_cnt ? s_list[i * kNT + et] : 0ull;
          os[i] = i < tk_cnt ? top1_key_value(key) : -INFINITY;
          oi[i] = i < tk_cnt ? (long long)(0xffffffffu - (unsigned)(key & 0xffffffffull)) : -1LL;
        }
      }
    }
    if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;\n" ::: "memory");   // smem outlives the last boxes
  }

  tc_fence_before();
  __syncthreads();
  cluster_sync_all();                          // the peer's MMAs / remote arrivals are done with this CTA's smem
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;\n" ::"r"(tmem_base), "r"(kAccStages * BN));
  }
}

// ---------------------------------------------------------------------------------------------------
// Layout kernels around the GEMM
// ---------------------------------------------------------------------------------------------------

// Padded-row bookkeeping of a ragged batch: utterance b owns padded rows
// [poffs[b], poffs[b+1]) = kHalo + T_b + kHalo rows.  rowmap: flags per padded row; rowseg: utterance id of
// real rows, -1 - id for halo rows.
__global__ void build_padded_kernel(const long long* __restrict__ offs, long long batch,
                                    long long* __restrict__ poffs, int* __restrict__ rowmap,
                                    int* __restrict__ rowseg) {
  // one CTA per utterance
  const long long b = blockIdx.x;
  const long long r0 = offs[b], T = offs[b + 1] - r0;
  const long long p0 = r0 + 2LL * kHalo * b;
  if (threadIdx.x == 0) {
    poffs[b] = p0;
    if (b == batch - 1) poffs[batch] = p0 + T + 2 * kHalo;
  }
  for (long long i = threadIdx.x; i < T + 2 * kHalo; i += blockDim.x) {
    int f = 0;
    const long long t = i - kHalo;
    const bool real = t >= 0 && t < T;
    if (real) {
      f = kRowStore;
      if (t == 0) f |= kRowFirst;
      if (t == T - 1) f |= kRowLast;
    }
    // bits 8..11 / 12..15: frames available before / after the (clamped) frame, saturated at 15; bits 16..23: 8 + the
    // displacement of the clamped frame (halo rows replicate the edge frames) -- used by splice_rows_kernel.  An empty
    // utterance (T = 0) has no frame to clamp to: its 2 kHalo halo rows carry kRowEmpty and no displacement.
    if (T > 0) {
      const long long tc = min(max(t, 0LL), T - 1);
      f |= (int)min(tc, 15LL) << 8;
      f |= (int)min(T - 1 - tc, 15LL) << 12;
      f |= (int)(tc - t + 8) << 16;
    } else {
      f = kRowEmpty | (8 << 16);
    }
    rowmap[p0 + i] = f;
    rowseg[p0 + i] = real ? (int)b : -1 - (int)b;
  }
}

// Materialised splice ("im2col") for layers whose feature dimension is not a multiple of 64:
// out[p, k*D + d] = x[clamp(t + ctx_k)] for every padded row p (halo rows clamp to the edge frames),
// bf16, row stride ld (a multiple of 8, zero padded).  x is fp32 ragged (rows, D) or bf16 padded-row
// (prow, x_ld).  One thread produces 8 consecutive outputs (one 16-byte store).
template <typename TIn>
__global__ void splice_kernel(const TIn* __restrict__ x, int D, long long x_ld, int x_is_padded,
                              const long long* __restrict__ offs, const long long* __restrict__ poffs,
                              const int* __restrict__ rowseg, long long prow, const long long* __restrict__ prow_dev,
                              int num_taps, const int* __restrict__ ctx_dev, __nv_bfloat16* __restrict__ out,
                              long long ld) {
  __shared__ int s_ctx[KTF_MAX_CONTEXT];
  if (threadIdx.x < KTF_MAX_CONTEXT) s_ctx[threadIdx.x] = threadIdx.x < num_taps ? ctx_dev[threadIdx.x] : 0;
  __syncthreads();
  if (prow_dev != nullptr) prow = min(prow, *prow_dev);   // `prow` from the host is an upper bound
  const int chunks = (int)(ld >> 3);
  const long long total = prow * chunks;
  const int cols = num_taps * D;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const long long p = idx / chunks;
    const int c0 = (int)(idx - p * chunks) << 3;
    const int sgn = rowseg[p];
    const int b = sgn >= 0 ? sgn : -1 - sgn;
    const long long p0 = poffs[b];
    const long long T = poffs[b + 1] - p0 - 2 * kHalo;
    long long t = p - p0 - kHalo;
    t = min(max(t, 0LL), T - 1);
    const long long base = x_is_padded ? (p0 + kHalo) : offs[b];
    __align__(16) __nv_bfloat16 v[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int c = c0 + i;
      float f = 0.0f;
      if (c < cols && T > 0) {                     // an empty utterance has no frame to clamp to: zero rows
        const int k = c / D, d = c - k * D;
        const long long tt = min(max(t + s_ctx[k], 0LL), T - 1);
        f = (float)x[(base + tt) * x_ld + d];
      }
      v[i] = __float2bfloat16_rn(f);
    }
    *reinterpret_cast<uint4*>(out + p * ld + c0) = *reinterpret_cast<const uint4*>(v);
  }
}

// Fast splice for fp32 ragged input with CONSECUTIVE contexts (ctx_k = ctx_0 + k) and an even feature dimension:
// the K taps of frame t are the contiguous span x[(t + ctx_0) D, (t + ctx_0 + K) D) of the utterance, so an output
// row is a converted copy of K D consecutive floats.  One thread per 16-byte output chunk; everything it needs to
// know about its row comes from rowmap / rowseg (two independent loads, no dependent chain through the offsets).
__global__ void __launch_bounds__(256)
splice_rows_kernel(const float* __restrict__ x, int D, const int* __restrict__ rowmap, const int* __restrict__ rowseg,
                   long long prow, const long long* __restrict__ prow_dev, int K, int ctx0,
                   __nv_bfloat16* __restrict__ out, long long ld) {
  if (prow_dev != nullptr) prow = min(prow, *prow_dev);   // `prow` from the host is an upper bound
  const unsigned chunks = (unsigned)(ld >> 3);
  const int cols = K * D;
  const unsigned long long total = (unsigned long long)prow * chunks;
  for (unsigned long long idx = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (unsigned long long)gridDim.x * blockDim.x) {
    long long p;
    if (total < 0xffffffffull) p = (unsigned)idx / chunks; else p = (long long)(idx / chunks);
    const int c0 = (int)(idx - (unsigned long long)p * chunks) << 3;
    const int m = rowmap[p], sg = rowseg[p];
    const int b = sg >= 0 ? sg : -1 - sg;
    const int lo = (m >> 8) & 15, hi = (m >> 12) & 15, delta = ((m >> 16) & 255) - 8;
    const long long srow = p - (long long)kHalo * (2 * b + 1) + delta;   // source row of the (clamped) frame
    const bool inside = (ctx0 >= -lo) && (ctx0 + K - 1 <= hi);
    float f[8];
    if (m & kRowEmpty) {                           // halo row of an empty utterance: nothing to read
#pragma unroll
      for (int i = 0; i < 8; ++i) f[i] = 0.0f;
    } else if (inside) {
      const float* src = x + (srow + ctx0) * D + c0;
      if (c0 + 8 <= cols) {
        const float2* s2 = reinterpret_cast<const float2*>(src);   // D even, c0 % 8 == 0: 8-byte aligned
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float2 v = s2[i];
          f[2 * i] = v.x;
          f[2 * i + 1] = v.y;
        }
      } else {
#pragma unroll
        for (int i = 0; i < 8; ++i) f[i] = (c0 + i < cols) ? src[i] : 0.0f;
      }
    } else {
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int c = c0 + i;
        f[i] = 0.0f;
        if (c < cols) {
          const int k = c / D, d = c - k * D;
          const int o = min(max(ctx0 + k, -lo), hi);
          f[i] = x[(srow + o) * D + d];
        }
      }
    }
    __align__(16) __nv_bfloat16 v[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = __float2bfloat16_rn(f[i]);
    *reinterpret_cast<uint4*>(out + p * ld + c0) = *reinterpret_cast<const uint4*>(v);
  }
}

// Splice for the modes the padded-row layout does not cover -- padding="VALID" and subsampling_factor > 1
// (tdnn.py:224-249): one output row per EVALUATED time step, out[r, k*D + d] = x[in_base + clamp(t_in + ctx_k), d] with
// t_in = start + (r - out_offs[b]) * sub.  Rows map to utterances by binary search over out_offs (batch + 1).  Under
// VALID padding every tap is in range by construction, so the clamp only acts for SAME (edge replication, :244-247).
__global__ void __launch_bounds__(256)
splice_eval_kernel(const float* __restrict__ x, int D, const long long* __restrict__ in_offs,
                   const long long* __restrict__ out_offs, long long batch, long long out_rows, int start, int sub,
                   int num_taps, const int* __restrict__ ctx_dev, __nv_bfloat16* __restrict__ out, long long ld) {
  __shared__ int s_ctx[KTF_MAX_CONTEXT];
  if (threadIdx.x < KTF_MAX_CONTEXT) s_ctx[threadIdx.x] = threadIdx.x < num_taps ? ctx_dev[threadIdx.x] : 0;
  __syncthreads();
  const int chunks = (int)(ld >> 3);
  const long long total = out_rows * chunks;
  const int cols = num_taps * D;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const long long r = idx / chunks;
    const int c0 = (int)(idx - r * chunks) << 3;
    long long lo = 0, hi = batch;
    while (hi - lo > 1) {
      const long long mid = (lo + hi) >> 1;
      if (out_offs[mid] <= r) lo = mid; else hi = mid;
    }
    const long long base = in_offs[lo];
    const long long T = in_offs[lo + 1] - base;
    const long long t = start + (r - out_offs[lo]) * sub;
    __align__(16) __nv_bfloat16 v[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int c = c0 + i;
      float f = 0.0f;
      if (c < cols && T > 0) {
        const int k = c / D, d = c - k * D;
        const long long tt = min(max(t + s_ctx[k], 0LL), T - 1);
        f = x[(base + tt) * D + d];
      }
      v[i] = __float2bfloat16_rn(f);
    }
    *reinterpret_cast<uint4*>(out + r * ld + c0) = *reinterpret_cast<const uint4*>(v);
  }
}


// ---------------------------------------------------------------------------------------------------
// Fused pre-pass of the wav -> x-vector path: VAD gather -> sliding CMVN -> bf16 splice of the first layer.
// Replaces three passes over the same rows -- the tf.gather_nd compaction of models/kaldi/xvector_extractor.py:163-165,
// layers/normalization/cmvn.py:186-250 (center=True, norm_vars=False, padding SAME) and the materialised splice of
// layers/tdnn/tdnn.py:251-258 for a first layer with consecutive contexts -- with one kernel: the kept MFCC rows are
// gathered straight into shared memory through the VAD index list, normalised there, and leave as the spliced bf16
// operand of tdnn1 in the padded-row layout.
//
// grid (batch, ceil(max_frames / tc)), 256 threads.  A CTA owns frames [c0, c1) of the COMPACTED utterance b:
//   1. stage rows [lo, hi) -- every row a window of its frames (and of the +-halo frames its splice taps reach) needs --
//      with 8-byte cp.async through index[] (or contiguously when index == nullptr);
//   2. copy the rows of frames [e0, e1) aside (y), then turn the staged rows into inclusive prefix sums per column:
//      32-row local prefixes, one scan over the block totals, offsets folded in;
//   3. y[t] -= (P[ws + N - 1] - P[ws - 1]) / N with ws = clamp(t - N/2, 0, T - N)   (cmvn.py:172-204; T <= N: the
//      global mean, :214-222);
//   4. emit out[p, k * D + d] = y[clamp(t + ctx0 + k)][d] as bf16, 16 bytes per thread and step.
// The prefix sums are differences of fp32 numbers up to ~N * |x|: their rounding (<= 2^-10 at 10^4) is divided by N again
// in the mean, i.e. ~3e-6 on features of magnitude 20 -- the reference's own fp32 cumsum over the whole utterance
// (cmvn.py:172) is coarser.
constexpr int kPreThreads = 256;
constexpr int kPreWarps = kPreThreads / 32;
constexpr int kPreBlk = 32;

// i / d for 0 <= i < 2^20 and 1 <= d <= 2^10 with one multiply: m = floor(2^32 / d) + 1 (host), exact in that range.
__device__ __forceinline__ unsigned fast_div(unsigned i, unsigned m) { return __umulhi(i, m); }

__global__ void __launch_bounds__(kPreThreads)
gather_cmvn_splice_kernel(const float* __restrict__ feats, int dim, const long long* __restrict__ index,
                          const long long* __restrict__ voffs, int window, int tc, int K, int ctx0,
                          __nv_bfloat16* __restrict__ out, long long ld, unsigned magic_half, unsigned magic_chunks) {
  extern __shared__ __align__(16) float spre[];
  const long long b = blockIdx.x;
  const long long r0 = voffs[b];
  const int T = (int)(voffs[b + 1] - r0);
  const int c0 = blockIdx.y * tc;
  if (T <= 0 || c0 >= T) return;
  const int c1 = min(c0 + tc, T);
  const int halo_l = ctx0 < 0 ? -ctx0 : 0, halo_r = (ctx0 + K - 1) > 0 ? (ctx0 + K - 1) : 0;
  const int e0 = max(c0 - halo_l, 0), e1 = min(c1 + halo_r, T);   // frames whose normalised rows the splice reads
  const int N = window;
  const bool global_stats = T <= N;
  const int lo = global_stats ? 0 : min(max(e0 - N / 2, 0), T - N);
  const int hi = global_stats ? T : min(max(e1 - 1 - N / 2, 0), T - N) + N;
  const int R = hi - lo;
  const int max_rows = tc + 2 * kHalo + N;
  float* sx = spre;                                                             // [R][dim] staged rows
  float* sy = spre + (((size_t)max_rows * dim + 3) & ~(size_t)3);               // [e1 - e0][dim] normalised rows (+ 8 pad)
  float* bsum = sy + (((size_t)(tc + 2 * kHalo) * dim + 8 + 3) & ~(size_t)3);   // [nblk][dim] sums of 32-row blocks
  // [R] source rows, 8-byte aligned: the block sums are rounded up to an even float count
  long long* srow = reinterpret_cast<long long*>(bsum + (((size_t)(max_rows / kPreBlk + 2) * dim + 1) & ~(size_t)1));
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

  // ---- 1. stage (gather): source rows first (independent loads, one latency), then the copies ----------------
  for (int r = tid; r < R; r += kPreThreads) srow[r] = index ? index[r0 + lo + r] : (r0 + lo + r);
  __syncthreads();
  if ((dim & 1) == 0) {
    const unsigned half = (unsigned)dim >> 1;                  // 8-byte pieces: rows start 8-byte aligned
    const unsigned sbase = smem_u32(sx);
    const unsigned total = (unsigned)R * half;
    for (unsigned i = tid; i < total; i += kPreThreads) {
      const unsigned r = fast_div(i, magic_half), h = i - r * half;
      const float* src = feats + srow[r] * dim + 2 * h;
      asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"(sbase + 8u * i), "l"(src) : "memory");
    }
    asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;\n" ::: "memory");
  } else {
    for (int r = warp; r < R; r += kPreWarps) {
      const float* src = feats + srow[r] * dim;
      for (int d = lane; d < dim; d += 32) sx[r * dim + d] = src[d];
    }
  }
  __syncthreads();

  // ---- 2. column sums of 32-row blocks: a warp's first window is then a handful of block sums plus the rows that
  //         stick out on both sides (the arithmetic of cmvn_staged_kernel, vad_cmvn.cu) ----------------------------
  const float* xs = sx - (long long)lo * dim;                  // xs[t * dim + d] = row t of the compacted utterance
  const int nblk = R / kPreBlk;
  for (int k = warp; k < nblk; k += kPreWarps) {
    for (int d = lane; d < dim; d += 32) {
      const float* col = sx + (k * kPreBlk) * dim + d;
      float p0 = 0.0f, p1 = 0.0f, p2 = 0.0f, p3 = 0.0f;
#pragma unroll
      for (int r = 0; r < kPreBlk; r += 4) {
        p0 += col[r * dim]; p1 += col[(r + 1) * dim]; p2 += col[(r + 2) * dim]; p3 += col[(r + 3) * dim];
      }
      bsum[k * dim + d] = (p0 + p1) + (p2 + p3);
    }
  }
  __syncthreads();

  // ---- 3. y[t] = x[t] - mean over the window of t (cmvn.py:172-204; T <= N: the global mean, :214-222) ---------
  {
    const int per = (e1 - e0 + kPreWarps - 1) / kPreWarps;
    const int t0 = e0 + warp * per, t1 = min(t0 + per, e1);
    const int W = global_stats ? T : N, H = N / 2;
    const float inv_n = 1.0f / (float)W;
    for (int d = lane; d < dim && t0 < t1; d += 32) {
      int ws = global_stats ? 0 : min(max(t0 - H, 0), T - N);
      float p0 = 0.0f, p1 = 0.0f, p2 = 0.0f, p3 = 0.0f;
      {
        // rows [ws, ws + W) = leading rows up to the next block boundary, whole blocks, trailing rows
        const int a0 = ws - lo;
        const int kb = (a0 + kPreBlk - 1) / kPreBlk;
        const int ke = min((a0 + W) / kPreBlk, nblk);
        int r_lead_end = ws + W, r_trail = ws + W;               // no whole block inside: everything is "leading"
        if (ke > kb) {
          r_lead_end = lo + kb * kPreBlk;
          r_trail = lo + ke * kPreBlk;
          int k = kb;
          for (; k + 2 <= ke; k += 2) { p0 += bsum[k * dim + d]; p1 += bsum[(k + 1) * dim + d]; }
          if (k < ke) p0 += bsum[k * dim + d];
        }
        for (int r = ws; r < r_lead_end; ++r) p2 += xs[(long long)r * dim + d];
        for (int r = r_trail; r < ws + W; ++r) p3 += xs[(long long)r * dim + d];
      }
      float sacc = (p0 + p1) + (p2 + p3);
      float* yrow = sy + (t0 - e0) * dim + d;
      int tt = t0;
      if (global_stats) {
        for (; tt < t1; ++tt, yrow += dim) *yrow = xs[tt * dim + d] - sacc * inv_n;
      } else {
        // head: frames whose window is still clamped at the start of the utterance
        for (; tt < t1 && tt - H <= ws; ++tt, yrow += dim) *yrow = xs[tt * dim + d] - sacc * inv_n;
        // interior: the window advances by exactly one row per frame
        const int t_mid = min(t1, T - N + H + 1);
        const float* po = xs + ws * dim + d;                     // row leaving the window
        const float* pn = po + N * dim;                          // row entering it
        const float* px = xs + tt * dim + d;
#pragma unroll 4
        for (; tt < t_mid; ++tt) {
          sacc += *pn - *po;
          po += dim; pn += dim;
          *yrow = *px - sacc * inv_n;
          px += dim; yrow += dim;
        }
        // tail: window clamped at the end of the utterance
        for (; tt < t1; ++tt, yrow += dim) *yrow = xs[tt * dim + d] - sacc * inv_n;
      }
    }
  }
  __syncthreads();

  // ---- 4. spliced bf16 rows of frames [c0, c1): the K taps of an interior frame are K * dim CONSECUTIVE floats of y
  const unsigned chunks = (unsigned)(ld >> 3);
  const int cols = K * dim;
  const long long p_first = r0 + 2LL * kHalo * b + kHalo;     // padded row of frame 0
  const unsigned total_chunks = (unsigned)(c1 - c0) * chunks;
  for (unsigned i = tid; i < total_chunks; i += kPreThreads) {
    const unsigned tt = fast_div(i, magic_chunks), q = i - tt * chunks;
    const int t = c0 + (int)tt, col0 = (int)(q << 3);
    const int ta = t + ctx0;
    float f[8];
    if (ta >= 0 && ta + K - 1 <= T - 1) {
      const float* row = sy + (ta - e0) * dim + col0;           // may run up to 7 floats past the taps: masked below
      if ((dim & 1) == 0) {
        const float2* src = reinterpret_cast<const float2*>(row);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const float2 v = src[u];
          f[2 * u] = v.x;
          f[2 * u + 1] = v.y;
        }
      } else {
#pragma unroll
        for (int u = 0; u < 8; ++u) f[u] = row[u];
      }
      if (col0 + 8 > cols) {
#pragma unroll
        for (int u = 0; u < 8; ++u) f[u] = (col0 + u < cols) ? f[u] : 0.0f;
      }
    } else {                                                    // the first / last frames of the utterance
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int c = col0 + u;
        f[u] = 0.0f;
        if (c < cols) {
          const int k = c / dim, d = c - k * dim;
          const int src_t = min(max(ta + k, 0), T - 1);         // edge replication (tdnn.py:244-247)
          f[u] = sy[(src_t - e0) * dim + d];
        }
      }
    }
    __align__(16) __nv_bfloat16 v[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) v[u] = __float2bfloat16_rn(f[u]);
    *reinterpret_cast<uint4*>(out + (p_first + t) * ld + col0) = *reinterpret_cast<const uint4*>(v);
  }
  // halo rows of the operand only feed accumulator rows the GEMM epilogue never stores; keep them finite
  if (c0 == 0 && warp < kHalo)
    for (unsigned q = lane; q < chunks; q += 32)
      *reinterpret_cast<uint4*>(out + (p_first - kHalo + warp) * ld + (q << 3)) = make_uint4(0, 0, 0, 0);
  if (c1 == T && warp >= kPreWarps - kHalo)
    for (unsigned q = lane; q < chunks; q += 32)
      *reinterpret_cast<uint4*>(out + (p_first + T + (warp - (kPreWarps - kHalo))) * ld + (q << 3)) = make_uint4(0, 0, 0, 0);
}

size_t prepass_smem_bytes(int tc, int window, int dim) {
  const size_t a = (((size_t)(tc + 2 * kHalo + window) * dim + 3) & ~(size_t)3);
  const size_t y = (((size_t)(tc + 2 * kHalo) * dim + 8 + 3) & ~(size_t)3);
  const size_t blk = ((size_t)((tc + 2 * kHalo + window) / kPreBlk + 2) * dim + 1) & ~(size_t)1;
  return (a + y + blk) * sizeof(float) + (size_t)(tc + 2 * kHalo + window) * sizeof(long long);
}

// Frames per CTA of the pre-pass: the largest even tc <= 256 (KTF_PREPASS_TC) and >= 32 whose CTA fits 113 KB of shared
// memory, balanced over the longest utterance (998 frames -> 4 x 250) with at most 65535 CTAs per utterance.  A wide
// window or feature dimension takes a smaller tile (D 30: window <= 372 at tc 256, <= 800 at tc 32).  False when even
// tc = 32 does not fit (D 80 at window 300): the caller then runs the separate gather -> CMVN -> splice kernels.
bool prepass_tile(long long max_frames, int window, int dim, int* tc_out, long long* gys_out) {
  static const int tc_target = getenv("KTF_PREPASS_TC") ? std::max(atoi(getenv("KTF_PREPASS_TC")), 32) : 256;
  for (int target = tc_target & ~1; target >= 32; target -= 2) {
    const long long gys = (max_frames + target - 1) / target;
    const int tc = (int)((((max_frames + gys - 1) / gys) + 1) & ~1LL);
    if (gys <= 65535 && prepass_smem_bytes(tc, window, dim) <= 113 * 1024) {
      *tc_out = tc;
      *gys_out = gys;
      return true;
    }
  }
  return false;
}

// (batch, 2, U) sums of d = r - c, r = relu(acc + bias), c = shift (TcLayer::d_shift, 0 if null), over the frames of each
// utterance -> mean || std of y = scale * r + offset (batchnorm.py:81-88 folded in algebraically;
// stats_pooling.py:228-240):
//   mean_y = scale * mean_d + (scale * c + offset),  var_y = scale^2 * (E[d^2] - mean_d^2),  std = sqrt(relu(var_y) + eps)
// (scale * c + offset is 0 up to rounding).  An empty utterance pools to NaN, the mean over zero frames.
__global__ void stats_finalize_tc_kernel(const float* __restrict__ sums, const long long* __restrict__ offs, int U,
                                         const float* __restrict__ scale, const float* __restrict__ offset,
                                         const float* __restrict__ shift, int include_std, float eps,
                                         __nv_bfloat16* __restrict__ out_bf16,
                                         float* __restrict__ out_f32, long long out_ld) {
  const int u = blockIdx.y * blockDim.x + threadIdx.x;
  if (u >= U) return;
  const long long b = blockIdx.x;
  const float n = (float)(offs[b + 1] - offs[b]);
  const float md = sums[(b * 2 + 0) * U + u] / n;
  const float vr = sums[(b * 2 + 1) * U + u] / n - __fmul_rn(md, md);
  const float sc = scale ? scale[u] : 1.0f;
  const float of = offset ? offset[u] : 0.0f;
  float mean = fmaf(sc, md, fmaf(sc, shift ? shift[u] : 0.0f, of));
  float sd = sqrtf(fmaxf(sc * sc * vr, 0.0f) + eps);
  if (!(n > 0.0f)) mean = sd = __int_as_float(0x7fc00000);   // (fmaxf would turn a NaN variance into sqrt(eps))
  if (out_bf16) {
    out_bf16[b * out_ld + u] = __float2bfloat16_rn(mean);
    if (include_std) out_bf16[b * out_ld + U + u] = __float2bfloat16_rn(sd);
  }
  if (out_f32) {
    out_f32[b * out_ld + u] = mean;
    if (include_std) out_f32[b * out_ld + U + u] = sd;
  }
}

// Gathers the real rows of a padded fp32 matrix back into the caller's ragged (rows, dim) layout.
__global__ void unpad_rows_kernel(const float* __restrict__ yp, long long ld, int dim,
                                  const long long* __restrict__ offs, const long long* __restrict__ poffs,
                                  long long batch, float* __restrict__ y) {
  const long long b = blockIdx.x;
  const long long r0 = offs[b], T = offs[b + 1] - r0, p0 = poffs[b] + kHalo;
  for (long long i = threadIdx.x; i < T * dim; i += blockDim.x) {
    const long long t = i / dim;
    const int d = (int)(i - t * dim);
    y[(r0 + t) * dim + d] = yp[(p0 + t) * ld + d];
  }
}

// ---------------------------------------------------------------------------------------------------
// Host side
// ---------------------------------------------------------------------------------------------------

struct TcLayer {
  int D = 0, U = 0, K = 0;
  int ctx[KTF_MAX_CONTEXT] = {0};
  bool implicit = false;            // taps via shifted TMA loads (D % 64 == 0, SAME, no subsampling)
  long long w_ld = 0;               // bf16 weight row stride (elements)
  __nv_bfloat16* d_w = nullptr;     // (U, w_ld)
  int* d_ctx = nullptr;
  // Centre of the pooled sums, per unit: c = -offset / scale, the moving mean BatchNorm subtracts from
  // r = relu(acc + bias) (nullptr without BatchNorm).  The STATS epilogue accumulates r - c and the finaliser adds c
  // back: r can sit far from zero (mean / std of 200 is possible for a unit BatchNorm re-centres), and E[r^2] - E[r]^2
  // formed from fp32 sums of r itself cancels -- 9e-3 relative error in the pooled std at mean / std = 200 over 300
  // frames.  Centred, the sums are of the size of the std.
  float* d_shift = nullptr;
  CUtensorMap tmW_n;                // weights as the B operand (box BK x BN)
  CUtensorMap tmW_m;                // weights as the A operand (box BK x BM), STATS mode
  ktf::Workspace ws;                // scratch of the stand-alone layer call
};

// cuTensorMapEncodeTiled is a driver entry point; it is resolved through the runtime so that the
// library has no link-time dependency on libcuda (it must still load on a box without a driver).
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn == nullptr) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

// 2-D map over a row-major 16-bit matrix (inner = columns); OOB boxes (negative or past-the-end rows /
// columns) are zero filled.  bf16 and fp16 share the map type: TMA only moves the bytes.
int encode_map(CUtensorMap* map, const void* base, unsigned long long inner, unsigned long long rows,
               unsigned long long ld_elems, unsigned box_inner, unsigned box_rows) {
  EncodeTiledFn fn = encode_tiled_fn();
  if (fn == nullptr) {
    ktf::set_error("cuTensorMapEncodeTiled is not available from this driver");
    return KTF_ECUDA;
  }
  cuuint64_t dims[2] = {inner, rows};
  cuuint64_t strides[1] = {ld_elems * 2};
  cuuint32_t box[2] = {box_inner, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    ktf::set_error("cuTensorMapEncodeTiled failed with CUresult %d (inner %llu rows %llu ld %llu)", (int)r, inner,
                   rows, ld_elems);
    return KTF_ECUDA;
  }
  return KTF_OK;
}

// Output map for the TMA-store epilogue: row-major (rows, cols) matrix of 2-byte (bf16) or 4-byte (fp32) elements, boxes
// of 32 rows x 64 bytes with the 64-byte swizzle (the layout store_chunk stages) or 32 rows x 128 bytes with the 128-byte
// swizzle (store_box, pair kernel).  Returns false when the matrix cannot
// be described (unaligned base / pitch): the epilogue then keeps its st.global path.
bool encode_map_out(CUtensorMap* map, const void* base, int elem_bytes, unsigned long long cols, unsigned long long rows,
                    unsigned long long ld_elems, int row_bytes = kRowSeg) {
  EncodeTiledFn fn = encode_tiled_fn();
  if (fn == nullptr || base == nullptr || rows == 0 || cols == 0) return false;
  if ((reinterpret_cast<unsigned long long>(base) & 15ull) != 0 || ((ld_elems * elem_bytes) & 15ull) != 0) return false;
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {ld_elems * elem_bytes};
  cuuint32_t box[2] = {(cuuint32_t)(row_bytes / elem_bytes), 32};
  cuuint32_t estr[2] = {1, 1};
  const CUresult r = fn(map, elem_bytes == 2 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2,
                        const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                        row_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B,
                        CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS;
}

inline long long round_up(long long v, long long m) { return (v + m - 1) / m * m; }

int check_arch() {
  const int arch = ktf_device_arch();                    // the current device's, not the first one's
  if (arch < 100) {
    ktf::set_error("the tcgen05 engine needs an sm_100 device (found sm_%d)", arch);
    return KTF_EINVAL;
  }
  return KTF_OK;
}

int prepare_layer(TcLayer* L, const ktf_affine_cfg& c, const float* w_host) {
  L->D = c.in_dim;
  L->U = c.out_dim;
  L->K = c.num_context;
  for (int k = 0; k < c.num_context; ++k) L->ctx[k] = c.context[k];
  int maxabs = 0;
  for (int k = 0; k < c.num_context; ++k) maxabs = std::max(maxabs, std::abs(c.context[k]));
  L->implicit = (c.in_dim % 64 == 0) && !c.padding_valid && c.subsampling_factor == 1 && maxabs <= kHalo;
  const long long cols = (long long)c.num_context * c.in_dim;
  L->w_ld = round_up(cols, 8);
  std::vector<__nv_bfloat16> wb((size_t)c.out_dim * L->w_ld, __float2bfloat16(0.0f));
  for (int u = 0; u < c.out_dim; ++u)
    for (long long j = 0; j < cols; ++j) wb[(size_t)u * L->w_ld + j] = __float2bfloat16(w_host[(size_t)u * cols + j]);
  int rc;
  if ((rc = ktf::upload(&L->d_w, wb.data(), wb.size())) != KTF_OK) return rc;
  if ((rc = ktf::upload(&L->d_ctx, L->ctx, (size_t)KTF_MAX_CONTEXT)) != KTF_OK) return rc;
  if ((rc = encode_map(&L->tmW_n, L->d_w, (unsigned long long)cols, (unsigned long long)c.out_dim,
                       (unsigned long long)L->w_ld, BK, BN)) != KTF_OK)
    return rc;
  return encode_map(&L->tmW_m, L->d_w, (unsigned long long)cols, (unsigned long long)c.out_dim,
                    (unsigned long long)L->w_ld, BK, BM);
}

void release_layer(TcLayer* L) {
  if (!L) return;
  cudaFree(L->d_w);
  cudaFree(L->d_ctx);
  cudaFree(L->d_shift);
  L->ws.release();
}

int tma_store_enabled() {
  static int on = -1;
  if (on < 0) {
    const char* e = getenv("KTF_TC_TMA_STORE");     // development knob: 0 = st.global epilogue
    on = e ? atoi(e) : 1;
  }
  return on;
}

template <int MODE>
int launch_gemm(const CUtensorMap& tmA, const CUtensorMap& tmB, const TcArgs& args_in, cudaStream_t st) {
  TcArgs args = args_in;
  CUtensorMap tmC = tmA;                                // placeholder when the epilogue does not use it
  args.tma_store = 0;
  if (MODE != kModeStats && tma_store_enabled() && args.out != nullptr) {
    const int es = (MODE == kModeBf16) ? 2 : 4;
    if (encode_map_out(&tmC, args.out, es, (unsigned long long)args.n_rows, (unsigned long long)args.m_rows,
                       (unsigned long long)args.out_ld))
      args.tma_store = 1;
  }
  static unsigned long long attr_done = 0;              // per device (function attributes are per context)
  if (ktf::first_use_on_device(&attr_done))
    KTF_CUDA(cudaFuncSetAttribute(tdnn_tc_kernel<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemTc));
  const long long tiles = ((args.m_rows + BM - 1) / BM) * ((args.n_rows + BN - 1) / BN);
  if (tiles <= 0) return KTF_OK;
  static int dbg = -1;
  if (dbg < 0) {
    const char* e = getenv("KTF_TC_DEBUG");
    dbg = e ? atoi(e) : 0;
  }
  args.debug = dbg;
  const unsigned grid = (unsigned)std::min<long long>(tiles, ktf::num_sms());
  tdnn_tc_kernel<MODE><<<grid, kThreadsTc, kSmemTc, st>>>(tmA, tmB, tmC, args);
  KTF_LAUNCH_OK();
  return KTF_OK;
}

int pair_enabled() {
  static int on = -1;
  if (on < 0) {
    const char* e = getenv("KTF_TC_PAIR");     // development knob: 0 = single-CTA tiles for every launch
    on = e ? atoi(e) : 1;
  }
  return on;
}

// CTA-pair launch of a row-storing mode.  tmB must be encoded with 128-row boxes (each CTA loads half of the tile's 256
// columns); everything else as launch_gemm.
// Epilogue warps per CTA of the pair kernel.  The per-tile trace (KTF_TC_TRACE) shows which side waits: with K <= 256
// (tdnn1) the accumulator is ready long before the 16 epilogue warps are done -- epilogue-bound, 16 warps win (period 5.1 k
// against 5.5 k clocks with 8); from K = 384 up the MMA thread waits for operands (tdnn4: 6.9 k of 7.5 k clocks per tile),
// the epilogue has slack, and what helps is the fifth ring stage that 8 warps leave room for (tdnn4 7.5 k -> 6.4 k clocks,
// tdnn2 / tdnn3 16.1 k -> 14.7 k, PLDA 2.55 -> 2.42 ms).  KTF_TC_PAIR_EPI_WARPS overrides the choice.
int pair_epi_warps(int num_kb) {
  static int ew = -1;
  if (ew < 0) {
    const char* e = getenv("KTF_TC_PAIR_EPI_WARPS");
    ew = e ? atoi(e) : 0;
  }
  if (ew == 8 || ew == 16) return ew;
  return num_kb <= 4 ? 16 : 8;
}

template <int MODE, int EW>
int launch_gemm_pair_ew(const CUtensorMap& tmA, const CUtensorMap& tmB_half, const TcArgs& args_in, cudaStream_t st);

template <int MODE>
int launch_gemm_pair(const CUtensorMap& tmA, const CUtensorMap& tmB_half, const TcArgs& args_in, cudaStream_t st) {
  return pair_epi_warps(args_in.num_taps * args_in.kblocks_per_tap) == 16
             ? launch_gemm_pair_ew<MODE, 16>(tmA, tmB_half, args_in, st)
             : launch_gemm_pair_ew<MODE, 8>(tmA, tmB_half, args_in, st);
}

template <int MODE, int EW>
int launch_gemm_pair_ew(const CUtensorMap& tmA, const CUtensorMap& tmB_half, const TcArgs& args_in, cudaStream_t st) {
  constexpr int kSmemPair = pair_smem<MODE, EW>();
  constexpr int kPairThreads = PairCfg<EW>::kThreads;
  TcArgs args = args_in;
  if (args.row_add != nullptr && (args.scale != nullptr || args.offset != nullptr)) return KTF_EINVAL;
  CUtensorMap tmC = tmA;
  args.tma_store = 0;
  if (tma_store_enabled() && args.out != nullptr) {
    const int es = (MODE == kModeBf16) ? 2 : 4;
    if (encode_map_out(&tmC, args.out, es, (unsigned long long)args.n_rows, (unsigned long long)args.m_rows,
                       (unsigned long long)args.out_ld, kBoxRow))
      args.tma_store = 1;
  }
  static unsigned long long attr_done = 0;
  if (ktf::first_use_on_device(&attr_done))
    KTF_CUDA(cudaFuncSetAttribute(tdnn_tc_pair_kernel<MODE, EW>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemPair));
  long long tiles = ((args.m_rows + 2 * BM - 1) / (2 * BM)) * ((args.n_rows + BN - 1) / BN);
  if (tiles <= 0) return KTF_OK;
  if (topk_cap(MODE))   // work units, not tiles, are what the clusters share out
    tiles = ((args.m_rows + 2 * BM - 1) / (2 * BM)) *
            (((args.n_rows + BN - 1) / BN + args.topk_unit_tiles - 1) / args.topk_unit_tiles);
  static int dbg = -1;
  if (dbg < 0) {
    const char* e = getenv("KTF_TC_DEBUG");
    dbg = e ? atoi(e) : 0;
  }
  args.debug = dbg;
  // clusters that can be co-resident (a TPC with one SM fused off cannot host a pair): a persistent grid larger than
  // that would run its last clusters as a second wave
  static int max_clusters[64] = {0};
  int dev = 0;
  cudaGetDevice(&dev);
  dev &= 63;
  if (max_clusters[dev] == 0) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)ktf::num_sms() & ~1u);
    cfg.blockDim = dim3(kPairThreads);
    cfg.dynamicSmemBytes = kSmemPair;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 2;
    at[0].val.clusterDim.y = 1;
    at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    int n = 0;
    if (cudaOccupancyMaxActiveClusters(&n, tdnn_tc_pair_kernel<MODE, EW>, &cfg) != cudaSuccess || n <= 0) {
      (void)cudaGetLastError();
      n = ktf::num_sms() / 2;
    }
    max_clusters[dev] = n;
    if (getenv("KTF_TC_DEBUG_OCC")) fprintf(stderr, "[ktf] pair kernel: %d co-resident clusters on %d SMs\n", n, ktf::num_sms());
  }
  const unsigned clusters = (unsigned)std::min<long long>(tiles, std::min(max_clusters[dev], ktf::num_sms() / 2));
  // development: KTF_TC_TRACE=file appends, per launch, the clock64 stamps of cluster 0's first 512 tiles
  // (accumulator free / last operands landed / accumulator full / epilogue warp done) -- synchronises, never on by default
  static const char* trace_path = getenv("KTF_TC_TRACE");
  static long long* trace_dev = nullptr;
  if (trace_path != nullptr) {
    if (trace_dev == nullptr) KTF_CUDA(cudaMalloc(&trace_dev, 2048 * sizeof(long long)));
    KTF_CUDA(cudaMemsetAsync(trace_dev, 0, 2048 * sizeof(long long), st));
    args.trace = trace_dev;
  }
  tdnn_tc_pair_kernel<MODE, EW><<<2 * clusters, kPairThreads, kSmemPair, st>>>(tmA, tmB_half, tmC, args);
  KTF_LAUNCH_OK();
  if (trace_path != nullptr) {
    std::vector<long long> h(2048);
    KTF_CUDA(cudaStreamSynchronize(st));
    KTF_CUDA(cudaMemcpy(h.data(), trace_dev, 2048 * sizeof(long long), cudaMemcpyDeviceToHost));
    if (FILE* f = fopen(trace_path, "a")) {
      fprintf(f, "launch mode=%d ew=%d m=%lld n=%lld kb=%d clusters=%u\n", MODE, EW, args.m_rows, args.n_rows,
              args.num_taps * args.kblocks_per_tap, clusters);
      for (int i = 0; i < 512 && h[4 * i] != 0; ++i)
        fprintf(f, "%d %lld %lld %lld %lld\n", i, h[4 * i], h[4 * i + 1], h[4 * i + 2], h[4 * i + 3]);
      fclose(f);
    }
  }
  return KTF_OK;
}

void fill_taps(TcArgs& args, const TcLayer& L, bool a_is_spliced, long long a_cols) {
  if (a_is_spliced) {
    args.num_taps = 1;
    args.ctx[0] = 0;
    args.kblocks_per_tap = (int)((a_cols + BK - 1) / BK);
    args.tap_cols = 0;
  } else {
    args.num_taps = L.K;
    for (int k = 0; k < L.K; ++k) args.ctx[k] = L.ctx[k];
    args.kblocks_per_tap = L.D / BK;
    args.tap_cols = L.D;
  }
}

// One affine layer on padded rows, output stored row-major.  A: bf16 (m_rows, a_ld) padded-row activations
// (implicit taps) or an already spliced matrix.
int run_layer(const TcLayer& L, const ktf_affine* a, const __nv_bfloat16* A, long long a_ld, long long a_cols,
              long long m_rows, const int* rowmap, void* out, long long out_ld, bool out_bf16, bool a_is_spliced,
              cudaStream_t st, int reverse = 0, const long long* rows_dev = nullptr) {
  CUtensorMap tmA;
  int rc = encode_map(&tmA, A, (unsigned long long)a_cols, (unsigned long long)m_rows, (unsigned long long)a_ld, BK, BM);
  if (rc != KTF_OK) return rc;
  TcArgs args{};
  fill_taps(args, L, a_is_spliced, a_cols);
  args.m_rows = m_rows;
  args.n_rows = L.U;
  args.act_base = A;
  args.act_ld_bytes = a_ld * 2;
  args.act_rows = m_rows;
  args.rows_dev = rows_dev;
  args.reverse = reverse;
  args.rowmap = rowmap;
  args.bias = a->d_bias;
  args.scale = a->d_scale;
  args.offset = a->d_offset;
  args.relu = a->cfg.activation == KTF_ACT_RELU;
  args.out = out;
  args.out_ld = out_ld;
  if (pair_enabled())   // CTA-pair tiles: each CTA loads 128 of the 256 weight rows of a tile (tmW_m has 128-row boxes)
    return out_bf16 ? launch_gemm_pair<kModeBf16>(tmA, L.tmW_m, args, st) : launch_gemm_pair<kModeF32>(tmA, L.tmW_m, args, st);
  return out_bf16 ? launch_gemm<kModeBf16>(tmA, L.tmW_n, args, st) : launch_gemm<kModeF32>(tmA, L.tmW_n, args, st);
}

// The layer that feeds StatsPooling: operands swapped (M = units, N = frames), epilogue accumulates
// per-utterance sum / sum of squares of relu(acc + bias) into sums (batch, 2, U) (pre-zeroed).
int run_layer_stats(const TcLayer& L, const ktf_affine* a, const __nv_bfloat16* X, long long x_ld, long long x_cols,
                    long long frames, const int* rowseg, float* sums, bool x_is_spliced, cudaStream_t st,
                    int reverse = 0, const long long* rows_dev = nullptr) {
  CUtensorMap tmX;
  int rc = encode_map(&tmX, X, (unsigned long long)x_cols, (unsigned long long)frames, (unsigned long long)x_ld, BK, BN);
  if (rc != KTF_OK) return rc;
  TcArgs args{};
  fill_taps(args, L, x_is_spliced, x_cols);
  args.shift_b = 1;
  args.m_rows = L.U;
  args.n_rows = frames;
  args.act_base = X;
  args.act_ld_bytes = x_ld * 2;
  args.act_rows = frames;
  args.rows_dev = rows_dev;
  args.reverse = reverse;
  args.rowseg = rowseg;
  args.bias = a->d_bias;
  args.shift = L.d_shift;       // the sums are centred on the BatchNorm moving mean
  args.relu = a->cfg.activation == KTF_ACT_RELU;
  args.sums = sums;
  return launch_gemm<kModeStats>(L.tmW_m, tmX, args, st);
}

unsigned blocks_for(long long items, int threads) {
  return (unsigned)std::min<long long>((items + threads - 1) / threads, (long long)ktf::num_sms() * 16);
}

}  // namespace

namespace ktf {

int affine_tc_prepare(ktf_affine* a, const float* weights_host, const float* bn_scale_host,
                      const float* bn_offset_host) {
  int rc = check_arch();
  if (rc != KTF_OK) return rc;
  TcLayer* L = new TcLayer();
  rc = prepare_layer(L, a->cfg, weights_host);
  if (rc == KTF_OK && bn_scale_host && bn_offset_host) {
    std::vector<float> c(a->cfg.out_dim);
    for (int u = 0; u < a->cfg.out_dim; ++u)
      c[u] = bn_scale_host[u] != 0.0f ? -bn_offset_host[u] / bn_scale_host[u] : 0.0f;
    rc = ktf::upload(&L->d_shift, c.data(), c.size());
  }
  if (rc != KTF_OK) {
    release_layer(L);
    delete L;
    return rc;
  }
  a->tc = L;
  return KTF_OK;
}

void affine_tc_release(ktf_affine* a) {
  if (a && a->tc) {
    release_layer(static_cast<TcLayer*>(a->tc));
    delete static_cast<TcLayer*>(a->tc);
    a->tc = nullptr;
  }
}

// Stand-alone layer call (fp32 in / fp32 out): splice to bf16 once, then the tensor-core GEMM.
// Only SAME padding without subsampling is offered on this engine (the x-vector networks use nothing else).

// Materialises the spliced bf16 operand of a layer fed by fp32 ragged features.
static int launch_splice_f32(const TcLayer& L, const float* x, const long long* offs, const long long* poffs,
                      const int* rowmap, const int* rowseg, long long prow, const long long* prow_dev,
                      __nv_bfloat16* out, long long ld, cudaStream_t st) {
  bool consecutive = (L.D % 2) == 0;
  for (int k = 1; k < L.K; ++k) consecutive = consecutive && (L.ctx[k] == L.ctx[0] + k);
  bool small = true;                       // contexts inside the halo (the edge distances saturate at 15)
  for (int k = 0; k < L.K; ++k) small = small && L.ctx[k] >= -kHalo && L.ctx[k] <= kHalo;
  if (consecutive && small) {
    splice_rows_kernel<<<blocks_for(prow * (ld >> 3), 256), 256, 0, st>>>(x, L.D, rowmap, rowseg, prow, prow_dev, L.K,
                                                                           L.ctx[0], out, ld);
  } else {
    splice_kernel<float><<<blocks_for(prow * (ld >> 3), 256), 256, 0, st>>>(x, L.D, L.D, 0, offs, poffs, rowseg, prow,
                                                                            prow_dev, L.K, L.d_ctx, out, ld);
  }
  KTF_LAUNCH_OK();
  return KTF_OK;
}

int affine_tc_forward(const ktf_affine* a, const float* x_dev, const int64_t* in_offsets_dev,
                      const int64_t* out_offsets_dev, int64_t batch, int64_t total_in_rows,
                      int64_t total_out_rows, float* y_dev, float* stats_dev, cudaStream_t st) {
  TcLayer& L = *static_cast<TcLayer*>(a->tc);
  const long long cols = (long long)L.K * L.D, ld = round_up(cols, 8);
  int rc;
  if (a->cfg.padding_valid || a->cfg.subsampling_factor != 1) {
    // padding="VALID" / subsampling (tdnn.py:224-249): splice the evaluated time steps only, one plain GEMM over them
    ktf::Carver cv;
    const size_t o_spliced = cv.take((size_t)total_out_rows * ld * sizeof(__nv_bfloat16));
    const size_t o_y = cv.take(y_dev ? 0 : (size_t)total_out_rows * L.U * sizeof(float));
    if ((rc = L.ws.ensure(cv.off)) != KTF_OK) return rc;
    char* base = static_cast<char*>(L.ws.ptr);
    __nv_bfloat16* spliced = reinterpret_cast<__nv_bfloat16*>(base + o_spliced);
    float* y = y_dev ? y_dev : reinterpret_cast<float*>(base + o_y);
    const int start = (a->cfg.padding_valid && a->cfg.context[0] < 0) ? -a->cfg.context[0] : 0;
    splice_eval_kernel<<<blocks_for(total_out_rows * (ld >> 3), 256), 256, 0, st>>>(
        x_dev, L.D, (const long long*)in_offsets_dev, (const long long*)out_offsets_dev, batch, total_out_rows, start,
        a->cfg.subsampling_factor, L.K, L.d_ctx, spliced, ld);
    KTF_LAUNCH_OK();
    if ((rc = run_layer(L, a, spliced, ld, cols, total_out_rows, nullptr, y, L.U, /*out_bf16=*/false, /*spliced=*/true,
                        st)) != KTF_OK)
      return rc;
    if (stats_dev) return ktf::stats_sums_f32(y, out_offsets_dev, batch, L.U, stats_dev, st);
    return KTF_OK;
  }
  KTF_CHECK_ARG(total_in_rows == total_out_rows, "row count mismatch");
  // total_in_rows may be an upper bound of in_offsets_dev[batch] (VAD-compacted batches): the padded-row count is
  // read back on the device (poffs[batch]) by the splice and the GEMM
  const long long prow = total_in_rows + 2LL * kHalo * batch;
  ktf::Carver cv;
  const size_t o_poffs = cv.take((batch + 1) * sizeof(long long));
  const size_t o_rowmap = cv.take(prow * sizeof(int));
  const size_t o_rowseg = cv.take(prow * sizeof(int));
  const size_t o_spliced = cv.take((size_t)prow * ld * sizeof(__nv_bfloat16));
  const size_t o_yp = cv.take((size_t)prow * L.U * sizeof(float));
  const size_t o_y = cv.take(y_dev ? 0 : (size_t)total_out_rows * L.U * sizeof(float));
  rc = L.ws.ensure(cv.off);
  if (rc != KTF_OK) return rc;
  char* base = static_cast<char*>(L.ws.ptr);
  long long* poffs = reinterpret_cast<long long*>(base + o_poffs);
  int* rowmap = reinterpret_cast<int*>(base + o_rowmap);
  int* rowseg = reinterpret_cast<int*>(base + o_rowseg);
  __nv_bfloat16* spliced = reinterpret_cast<__nv_bfloat16*>(base + o_spliced);
  float* yp = reinterpret_cast<float*>(base + o_yp);
  float* y = y_dev ? y_dev : reinterpret_cast<float*>(base + o_y);

  build_padded_kernel<<<(unsigned)batch, 128, 0, st>>>((const long long*)in_offsets_dev, batch, poffs, rowmap, rowseg);
  KTF_LAUNCH_OK();
  if ((rc = launch_splice_f32(L, x_dev, (const long long*)in_offsets_dev, poffs, rowmap, rowseg, prow, poffs + batch,
                              spliced, ld, st)) != KTF_OK)
    return rc;
  rc = run_layer(L, a, spliced, ld, cols, prow, rowmap, yp, L.U, /*out_bf16=*/false, /*spliced=*/true, st, 0,
                 poffs + batch);
  if (rc != KTF_OK) return rc;
  unpad_rows_kernel<<<(unsigned)batch, 256, 0, st>>>(yp, L.U, L.U, (const long long*)in_offsets_dev, poffs, batch, y);
  KTF_LAUNCH_OK();
  if (stats_dev) {
    rc = ktf::stats_sums_f32(y, in_offsets_dev, batch, L.U, stats_dev, st);
    if (rc != KTF_OK) return rc;
  }
  return KTF_OK;
}

// C[i, j] = sum_k A[i, k] * B[j, k] + row_add[i] + col_add[j], A (m, K) and B (n, K) row-major 16-bit
// (bf16 or fp16), C fp32 with row stride ldc.  K and both leading dimensions must be multiples of 8.
int tc_gemm_nt(const void* A, long long m, long long lda, const void* B, long long n, long long ldb, long long K,
               int fp16, const float* row_add, const float* col_add, void* C, long long ldc, int c_bf16,
               cudaStream_t st, unsigned long long* row_best) {
  int rc = check_arch();
  if (rc != KTF_OK) return rc;
  CUtensorMap tmA, tmB;
  if ((rc = encode_map(&tmA, A, (unsigned long long)K, (unsigned long long)m, (unsigned long long)lda, BK, BM)) != KTF_OK)
    return rc;
  if ((rc = encode_map(&tmB, B, (unsigned long long)K, (unsigned long long)n, (unsigned long long)ldb, BK, BN)) != KTF_OK)
    return rc;
  TcArgs args{};
  args.num_taps = 1;
  args.kblocks_per_tap = (int)((K + BK - 1) / BK);
  args.fp16 = fp16;
  args.m_rows = m;
  args.n_rows = n;
  args.bias = col_add;
  args.row_add = row_add;
  args.out = C;
  args.out_ld = ldc;
  args.row_best = row_best;
  // streaming output (PLDA: the score matrix), operands re-read by every tile: see TcArgs::l2_stream_out
  args.l2_stream_out = ((double)m * (double)n * (c_bf16 ? 2.0 : 4.0) > 64e6) ? 1 : 0;
  if (const char* e = getenv("KTF_TC_L2_HINTS")) args.l2_stream_out = atoi(e);
  args.group_m = (n + BN - 1) / BN > 8 ? 32 : 0;     // (measured at 50 000^2: 1 -> 2.77, 8 -> 2.61, 16 -> 2.54, 32 -> 2.47-2.51, 64 -> 2.65 ms)
  if (const char* e = getenv("KTF_TC_GROUP_M")) args.group_m = atoi(e);
  if (pair_enabled() || row_best != nullptr) {    // (the best-entry epilogue exists in the pair kernel only)
    CUtensorMap tmBh;
    if ((rc = encode_map(&tmBh, B, (unsigned long long)K, (unsigned long long)n, (unsigned long long)ldb, BK, BN / 2)) != KTF_OK)
      return rc;
    return c_bf16 ? launch_gemm_pair<kModeBf16>(tmA, tmBh, args, st) : launch_gemm_pair<kModeF32>(tmA, tmBh, args, st);
  }
  return c_bf16 ? launch_gemm<kModeBf16>(tmA, tmB, args, st) : launch_gemm<kModeF32>(tmA, tmB, args, st);
}

}  // namespace ktf

namespace {

// Work units of the top-k walk: how many n-ranges (splits) a 256-row block is cut into.  Few splits keep the lists
// long-lived (a list fills up once per unit, and every unit writes one partial list per row and column quarter); enough
// of them give the clusters balanced waves.  Chosen by the modelled time: waves x (tiles per unit + one tile for filling
// and writing out the lists).  50 000 x 50 000: 196 row blocks x 3 splits of 66 n-tiles = 588 units, 7.9 waves of 74.
struct TopkPlan {
  int ew;             // epilogue warps per CTA
  int unit_tiles;     // n-tiles per unit
  int splits;
};

TopkPlan topk_plan(long long m, long long n, long long K) {
  TopkPlan pl{pair_epi_warps((int)((K + BK - 1) / BK)), 1, 0};
  const long long m_tiles = (m + 2 * BM - 1) / (2 * BM), n_tiles = (n + BN - 1) / BN;
  const long long clusters = std::max(1, ktf::num_sms() / 2);
  double best = 0.0;
  for (long long s = 1; s <= std::min<long long>(n_tiles, 16); ++s) {
    const long long len = (n_tiles + s - 1) / s, splits = (n_tiles + len - 1) / len;
    if (splits != s) continue;                     // the same cut as a smaller s
    const double cost = (double)((m_tiles * splits + clusters - 1) / clusters) * (double)(len + 1);
    if (pl.splits == 0 || cost < best) {
      best = cost;
      pl.unit_tiles = (int)len;
      pl.splits = (int)splits;
    }
  }
  return pl;
}

}  // namespace

namespace ktf {

int tc_topk_lists(long long m, long long n, long long K) {
  if (m <= 0 || n <= 0) return 0;
  const TopkPlan pl = topk_plan(m, n, K);
  return pl.splits * (pl.ew / 4);
}

int tc_gemm_topk(const void* A, long long m, long long lda, const void* B, long long n, long long ldb, long long K,
                 int fp16, const float* row_add, const float* col_add, int k, float* part_score, long long* part_index,
                 cudaStream_t st) {
  int rc = check_arch();
  if (rc != KTF_OK) return rc;
  if (m <= 0 || n <= 0) return KTF_OK;
  if (k < 1 || k > 32) {
    ktf::set_error("tc_gemm_topk: k = %d outside 1..32", k);
    return KTF_EINVAL;
  }
  CUtensorMap tmA, tmBh;
  if ((rc = encode_map(&tmA, A, (unsigned long long)K, (unsigned long long)m, (unsigned long long)lda, BK, BM)) != KTF_OK)
    return rc;
  if ((rc = encode_map(&tmBh, B, (unsigned long long)K, (unsigned long long)n, (unsigned long long)ldb, BK, BN / 2)) != KTF_OK)
    return rc;
  const TopkPlan pl = topk_plan(m, n, K);
  TcArgs args{};
  args.num_taps = 1;
  args.kblocks_per_tap = (int)((K + BK - 1) / BK);
  args.fp16 = fp16;
  args.m_rows = m;
  args.n_rows = n;
  args.bias = col_add;
  args.row_add = row_add;
  args.topk_k = k;
  args.topk_unit_tiles = pl.unit_tiles;
  args.topk_score = part_score;
  args.topk_index = part_index;
#define KTF_TOPK_LAUNCH(MODE_)                                                         \
  (pl.ew == 16 ? launch_gemm_pair_ew<MODE_, 16>(tmA, tmBh, args, st)                   \
               : launch_gemm_pair_ew<MODE_, 8>(tmA, tmBh, args, st))
  rc = k <= 8 ? KTF_TOPK_LAUNCH(kModeTopk8) : k <= 16 ? KTF_TOPK_LAUNCH(kModeTopk16) : KTF_TOPK_LAUNCH(kModeTopk32);
#undef KTF_TOPK_LAUNCH
  return rc;
}

}  // namespace ktf

// ---------------------------------------------------------------------------------------------------
// Whole-stack API: [affine(+ReLU+BN)] x n1 -> StatsPooling(reduce-all) -> [affine(+ReLU+BN)] x n2
// with bf16 activations that never leave the padded-row layout between layers.
// ---------------------------------------------------------------------------------------------------

struct ktf_tdnn_stack {
  std::vector<ktf_affine*> layers;       // borrowed handles (must be KTF_PREC_BF16)
  int stats_after = -1;                  // index of the layer followed by stats pooling (-1 = none)
  int include_std = 1;
  float stats_eps = 1e-10f;
  ktf::Workspace ws;                     // activations, padded-row maps, statistics (grow-only)
};

extern "C" {

int ktf_tdnn_stack_create(ktf_affine* const* layers, int32_t num_layers, int32_t stats_after_layer,
                          int32_t include_std, float stats_epsilon, ktf_tdnn_stack** out) {
  KTF_CHECK_ARG(layers && out && num_layers > 0, "ktf_tdnn_stack_create: bad arguments");
  KTF_CHECK_ARG(stats_after_layer >= -1 && stats_after_layer < num_layers, "stats_after_layer out of range");
  int rc = check_arch();
  if (rc != KTF_OK) return rc;
  int dim = -1;
  for (int i = 0; i < num_layers; ++i) {
    KTF_CHECK_ARG(layers[i] && layers[i]->tc, "layer %d was not created with KTF_PREC_BF16", i);
    const ktf_affine_cfg& c = layers[i]->cfg;
    KTF_CHECK_ARG(!c.padding_valid && c.subsampling_factor == 1,
                  "layer %d: the tcgen05 stack supports padding=SAME, subsampling_factor=1", i);
    KTF_CHECK_ARG(dim < 0 || c.in_dim == dim, "layer %d expects in_dim %d, previous layer produces %d", i, c.in_dim,
                  dim);
    dim = c.out_dim;
    if (i == stats_after_layer) dim = include_std ? 2 * dim : dim;
    if (i > stats_after_layer && stats_after_layer >= 0)
      KTF_CHECK_ARG(c.num_context == 1 && c.context[0] == 0, "layer %d (after stats pooling) must have context [0]", i);
  }
  ktf_tdnn_stack* s = new ktf_tdnn_stack();
  s->layers.assign(layers, layers + num_layers);
  s->stats_after = stats_after_layer;
  s->include_std = include_std;
  s->stats_eps = stats_epsilon;
  *out = s;
  return KTF_OK;
}

void ktf_tdnn_stack_destroy(ktf_tdnn_stack* s) {
  if (!s) return;
  s->ws.release();
  delete s;
}

int32_t ktf_tdnn_stack_out_dim(const ktf_tdnn_stack* s) {
  if (!s) return 0;
  int dim = s->layers.back()->cfg.out_dim;
  if (s->stats_after == (int)s->layers.size() - 1) dim = s->include_std ? 2 * dim : dim;
  return dim;
}

}  // extern "C"

// Shared body of ktf_tdnn_stack_forward (pre = nullptr) and ktf_tdnn_stack_forward_vad (fused pre-pass).
struct StackPre {
  const long long* index;   // kept-row indices into feats (or nullptr = rows are already compacted)
  long long max_frames;     // upper bound on the longest compacted utterance
  int cmvn_window;
};

static int stack_forward_impl(ktf_tdnn_stack* s, const float* feats_dev, const int64_t* offsets_dev, int64_t batch,
                              int64_t total_rows, float* out_dev, const StackPre* pre, cudaStream_t st) {
  if (batch <= 0 || total_rows <= 0) return KTF_OK;
  const long long prow = total_rows + 2LL * kHalo * batch;
  const int nl = (int)s->layers.size();
  const long long* offs = (const long long*)offsets_dev;

  // ---- workspace plan: per-frame activation ping-pong sized for the widest STORED matrix -------------
  long long max_ld = 8, final_frame_dim = 0;
  int stats_U = 0;
  for (int i = 0; i < nl; ++i) {
    const ktf_affine_cfg& c = s->layers[i]->cfg;
    const TcLayer& L = *static_cast<const TcLayer*>(s->layers[i]->tc);
    const bool per_frame_in = (s->stats_after < 0) || (i <= s->stats_after);
    if (per_frame_in && (i == 0 || !L.implicit)) max_ld = std::max(max_ld, round_up((long long)c.num_context * c.in_dim, 8));
    const bool stored_bf16 = per_frame_in && i != s->stats_after && i != nl - 1;
    if (stored_bf16) max_ld = std::max(max_ld, round_up(c.out_dim, 8));
    if (i == s->stats_after) stats_U = c.out_dim;
    if (i == nl - 1 && per_frame_in && i != s->stats_after) final_frame_dim = c.out_dim;
  }
  const int pooled_dim = s->include_std ? 2 * stats_U : stats_U;
  const long long p_ld = round_up(std::max(pooled_dim, 8), 8);
  long long post_ld = 8;                                    // widest bf16 activation after pooling
  for (int i = s->stats_after + 1; i < nl - 1 && s->stats_after >= 0; ++i)
    post_ld = std::max(post_ld, round_up(s->layers[i]->cfg.out_dim, 8));

  ktf::Carver cv;
  const size_t o_poffs = cv.take((batch + 1) * sizeof(long long));
  const size_t o_rowmap = cv.take(prow * sizeof(int));
  const size_t o_rowseg = cv.take(prow * sizeof(int));
  const size_t o_buf0 = cv.take((size_t)prow * max_ld * sizeof(__nv_bfloat16));
  const size_t o_buf1 = cv.take((size_t)prow * max_ld * sizeof(__nv_bfloat16));
  const size_t o_sums = cv.take((size_t)batch * 2 * std::max(stats_U, 1) * sizeof(float));
  const size_t o_pooled = cv.take((size_t)batch * p_ld * sizeof(__nv_bfloat16));
  const size_t o_post0 = cv.take((size_t)batch * post_ld * sizeof(__nv_bfloat16));
  const size_t o_post1 = cv.take((size_t)batch * post_ld * sizeof(__nv_bfloat16));
  const size_t o_yp = cv.take((size_t)prow * final_frame_dim * sizeof(float));
  int rc = s->ws.ensure(cv.off);
  if (rc != KTF_OK) return rc;
  char* base = static_cast<char*>(s->ws.ptr);
  long long* poffs = reinterpret_cast<long long*>(base + o_poffs);
  int* rowmap = reinterpret_cast<int*>(base + o_rowmap);
  int* rowseg = reinterpret_cast<int*>(base + o_rowseg);
  __nv_bfloat16* buf[2] = {reinterpret_cast<__nv_bfloat16*>(base + o_buf0),
                           reinterpret_cast<__nv_bfloat16*>(base + o_buf1)};
  float* sums = reinterpret_cast<float*>(base + o_sums);
  __nv_bfloat16* pooled = reinterpret_cast<__nv_bfloat16*>(base + o_pooled);
  __nv_bfloat16* post[2] = {reinterpret_cast<__nv_bfloat16*>(base + o_post0),
                            reinterpret_cast<__nv_bfloat16*>(base + o_post1)};
  float* yp = reinterpret_cast<float*>(base + o_yp);

  build_padded_kernel<<<(unsigned)batch, 128, 0, st>>>(offs, batch, poffs, rowmap, rowseg);
  KTF_LAUNCH_OK();
  // `total_rows` may be an upper bound of offsets_dev[batch]: the per-frame kernels read the actual padded-row count
  // (poffs[batch], written by the kernel above) on the device, so a VAD-compacted batch needs no host round trip
  const long long* prow_dev = poffs + batch;

  const __nv_bfloat16* cur = nullptr;   // current activations (bf16) and their geometry
  long long cur_ld = 0;
  bool per_frame = true;                // false once stats pooling collapsed the time axis
  int which = 0, pwhich = 0;

  for (int i = 0; i < nl; ++i) {
    const ktf_affine* a = s->layers[i];
    const TcLayer& L = *static_cast<const TcLayer*>(a->tc);
    const long long cols = (long long)L.K * L.D;
    const bool last = (i == nl - 1);

    if (!per_frame) {
      // pooled rows: a plain (batch x K) GEMM, context [0]
      if (last) return run_layer(L, a, cur, cur_ld, L.D, batch, nullptr, out_dev, L.U, false, true, st);
      __nv_bfloat16* y = post[pwhich];
      const long long y_ld = round_up(L.U, 8);
      if ((rc = run_layer(L, a, cur, cur_ld, L.D, batch, nullptr, y, y_ld, true, true, st)) != KTF_OK) return rc;
      cur = y;
      cur_ld = y_ld;
      pwhich ^= 1;
      continue;
    }

    // ---- operand of a per-frame layer: implicit taps on the padded activations, or a materialised splice
    const __nv_bfloat16* A = cur;
    long long a_ld = cur_ld, a_cols = L.D;
    bool spliced = false;
    if (i == 0 || !L.implicit) {
      __nv_bfloat16* sp = buf[which];
      const long long ld = round_up(cols, 8);
      const unsigned grid = blocks_for(prow * (ld >> 3), 256);
      if (i == 0 && pre != nullptr) {
        // VAD gather + sliding CMVN + splice in one pass (the rows never exist as a gathered / normalised fp32 matrix)
        int tc = 0;
        long long gys = 0;
        KTF_CHECK_ARG(prepass_tile(pre->max_frames, pre->cmvn_window, L.D, &tc, &gys),
                      "CMVN window %d x dim %d does not fit the fused pre-pass (see ktf_tdnn_stack_vad_prepass_fits)",
                      pre->cmvn_window, L.D);
        const size_t smem = prepass_smem_bytes(tc, pre->cmvn_window, L.D);
        static unsigned long long attr_set = 0;
        if (ktf::first_use_on_device(&attr_set))
          KTF_CUDA(cudaFuncSetAttribute(gather_cmvn_splice_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 113 * 1024));
        const unsigned half = (unsigned)std::max(L.D / 2, 1), chunks = (unsigned)(ld >> 3);
        gather_cmvn_splice_kernel<<<dim3((unsigned)batch, (unsigned)gys), kPreThreads, smem, st>>>(
            feats_dev, L.D, pre->index, offs, pre->cmvn_window, tc, L.K, L.ctx[0], sp, ld,
            (unsigned)(0x100000000ull / half) + 1u, (unsigned)(0x100000000ull / chunks) + 1u);
        KTF_LAUNCH_OK();
      } else if (i == 0) {
        if ((rc = ktf::launch_splice_f32(L, feats_dev, offs, poffs, rowmap, rowseg, prow, prow_dev, sp, ld, st)) != KTF_OK)
          return rc;
      } else {
        splice_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>(cur, L.D, cur_ld, 1, offs, poffs, rowseg, prow, prow_dev,
                                                           L.K, L.d_ctx, sp, ld);
        KTF_LAUNCH_OK();
      }
      A = sp;
      a_ld = ld;
      a_cols = cols;
      spliced = true;
      which ^= 1;
    }

    if (i == s->stats_after) {
      // fused StatsPooling: the activation of this layer is never stored
      KTF_CUDA(cudaMemsetAsync(sums, 0, (size_t)batch * 2 * L.U * sizeof(float), st));
      if ((rc = run_layer_stats(L, a, A, a_ld, a_cols, prow, rowseg, sums, spliced, st, i & 1, prow_dev)) != KTF_OK)
        return rc;
      dim3 grid((unsigned)batch, (unsigned)((L.U + 127) / 128));
      stats_finalize_tc_kernel<<<grid, 128, 0, st>>>(sums, offs, L.U, a->d_scale, a->d_offset, L.d_shift,
                                                     s->include_std, s->stats_eps, last ? nullptr : pooled,
                                                     last ? out_dev : nullptr,
                                                     last ? (long long)pooled_dim : p_ld);
      KTF_LAUNCH_OK();
      cur = pooled;
      cur_ld = p_ld;
      per_frame = false;
      continue;
    }
    if (last) {
      // per-frame fp32 output, un-padded into the caller's ragged layout
      if ((rc = run_layer(L, a, A, a_ld, a_cols, prow, rowmap, yp, L.U, false, spliced, st, 0, prow_dev)) != KTF_OK)
        return rc;
      unpad_rows_kernel<<<(unsigned)batch, 256, 0, st>>>(yp, L.U, L.U, offs, poffs, batch, out_dev);
      KTF_LAUNCH_OK();
      return KTF_OK;
    }
    __nv_bfloat16* y = buf[which];
    const long long y_ld = round_up(L.U, 8);
    // serpentine: odd layers walk the row blocks backwards, starting on the rows the previous layer wrote
    // last (still L2 resident) instead of the ones it wrote first (long evicted when activations > L2)
    if ((rc = run_layer(L, a, A, a_ld, a_cols, prow, rowmap, y, y_ld, true, spliced, st, i & 1, prow_dev)) != KTF_OK)
      return rc;
    cur = y;
    cur_ld = y_ld;
    which ^= 1;
  }
  return KTF_OK;
}

// The pre-pass emits the first layer's splice: its contexts must be consecutive and within the +-kHalo padding.
static bool prepass_contexts_ok(const ktf_tdnn_stack* s) {
  const TcLayer& L0 = *static_cast<const TcLayer*>(s->layers[0]->tc);
  bool ok = true;
  for (int k = 1; k < L0.K; ++k) ok = ok && (L0.ctx[k] == L0.ctx[0] + k);
  for (int k = 0; k < L0.K; ++k) ok = ok && L0.ctx[k] >= -kHalo && L0.ctx[k] <= kHalo;
  return ok;
}

extern "C" {

int ktf_tdnn_stack_forward(ktf_tdnn_stack* s, const float* feats_dev, const int64_t* offsets_dev,
                           int64_t batch, int64_t total_rows, float* out_dev, void* stream) {
  KTF_CHECK_ARG(s && feats_dev && offsets_dev && out_dev, "ktf_tdnn_stack_forward: null argument");
  return stack_forward_impl(s, feats_dev, offsets_dev, batch, total_rows, out_dev, nullptr, (cudaStream_t)stream);
}

int ktf_tdnn_stack_forward_vad(ktf_tdnn_stack* s, const float* feats_dev, const int64_t* index_dev,
                               const int64_t* offsets_dev, int64_t batch, int64_t total_rows, int64_t max_frames,
                               int32_t cmvn_window, float* out_dev, void* stream) {
  KTF_CHECK_ARG(s && feats_dev && offsets_dev && out_dev, "ktf_tdnn_stack_forward_vad: null argument");
  KTF_CHECK_ARG(cmvn_window > 0 && max_frames > 0, "`window` and `min_window` must be > 0");
  KTF_CHECK_ARG(prepass_contexts_ok(s),
                "the fused VAD / CMVN pre-pass needs a first layer with consecutive contexts within +-%d", kHalo);
  StackPre pre{(const long long*)index_dev, (long long)max_frames, cmvn_window};
  return stack_forward_impl(s, feats_dev, offsets_dev, batch, total_rows, out_dev, &pre, (cudaStream_t)stream);
}

int32_t ktf_tdnn_stack_vad_prepass_fits(const ktf_tdnn_stack* s, int32_t cmvn_window, int64_t max_frames) {
  if (!s || cmvn_window <= 0 || max_frames <= 0 || !prepass_contexts_ok(s)) return 0;
  int tc = 0;
  long long gys = 0;
  return prepass_tile(max_frames, cmvn_window, static_cast<const TcLayer*>(s->layers[0]->tc)->D, &tc, &gys) ? 1 : 0;
}

}  // extern "C"

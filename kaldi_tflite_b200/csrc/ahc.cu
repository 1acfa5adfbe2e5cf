// Average-linkage agglomerative clustering of the diarization back-end: Kaldi's single-pass AgglomerativeClusterer
// (agglomerative-cluster) for a batch of recordings, one CTA per recording (ktf_ahc_cluster in include/ktf_b200.h).
//
// Kaldi keeps a priority queue of (avg, lower id, higher id) and pops stale entries lazily.  Here every active slot
// (cluster) caches the smallest key of its eligible pairs, and a block-wide min over the caches is the queue's next valid
// entry.  After merging i and j into m, a slot whose cached partner was i or j rescans its row; every other slot
// compares its cache with its one new pair (k, m).  The other pairs' avg did not change, so every cache stays the exact
// minimum of its row and the merge order is Kaldi's, tie rules included, with no reducibility argument.
//
// Storage: the cost sums W live symmetric in a global scratch copy of the group's matrix (rows are read coalesced by the
// rescans and the merge update); the per-slot caches (8 bytes) and id / size words (4 bytes) are in shared memory, 12
// bytes per point, 192 KB at KTF_AHC_MAX_POINTS.
#include <float.h>
#include <math.h>

#include <algorithm>
#include <vector>

#include "common.cuh"

namespace {

constexpr int kAhcThreads = 512;
constexpr int kAhcWarps = kAhcThreads / 32;
constexpr unsigned long long kNoPair = ~0ull;        // no eligible pair
constexpr unsigned long long kRescan = ~0ull - 1;    // the slot's row has to be rescanned (never a real key)
constexpr int kRescanList = 32;                      // rows rescanned by the whole CTA per merge; more go one per warp

// One recording, in the order the CTAs take them (the largest first).
struct AhcGroup {
  long long s_off;      // its matrix in the packed scores (and in the W scratch)
  long long p_off;      // its first point (labels; 4 ints per point of id scratch)
  long long m_off;      // its first merge row
  int n;
  int min_clusters;
  float threshold;
  int index;            // its position in the caller's order (cluster_counts)
};

// Order key of an eligible pair: the float bits made unsigned-ordered (-0 taken as +0), then the lower and the higher
// cluster id (< 2^15: ids stay below 2 KTF_AHC_MAX_POINTS - 1).
__device__ __forceinline__ unsigned long long pair_key(float avg, unsigned a, unsigned b, float threshold) {
  if (!(avg <= threshold)) return kNoPair;
  const unsigned bits = avg == 0.0f ? 0u : __float_as_uint(avg);
  const unsigned ord = (bits & 0x80000000u) ? ~bits : (bits | 0x80000000u);
  return ((unsigned long long)ord << 32) | ((unsigned long long)min(a, b) << 15) | (unsigned long long)max(a, b);
}
__device__ __forceinline__ float key_avg(unsigned long long key) {
  const unsigned ord = (unsigned)(key >> 32);
  return __uint_as_float((ord & 0x80000000u) ? (ord & 0x7fffffffu) : ~ord);
}
__device__ __forceinline__ unsigned key_lo(unsigned long long key) { return (unsigned)(key >> 15) & 0x7fffu; }
__device__ __forceinline__ unsigned key_hi(unsigned long long key) { return (unsigned)key & 0x7fffu; }

__device__ __forceinline__ unsigned long long warp_min(unsigned long long v) {
  for (int o = 16; o > 0; o >>= 1) v = min(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// The smallest pair key of slot k's row over the active slots t != k, from the threads whose positions are
// t = first, first + stride, ...  (not reduced).
__device__ __forceinline__ unsigned long long row_min(const float* __restrict__ Wk, const unsigned* info, int n, int k,
                                                      int first, int stride, float threshold) {
  const unsigned ik = info[k], id_k = ik >> 16, sz_k = ik & 0xffffu;
  unsigned long long m = kNoPair;
#pragma unroll 4
  for (int t = first; t < n; t += stride) {
    const unsigned it = info[t];
    if ((it & 0xffffu) == 0u || t == k) continue;
    const float avg = __fdiv_rn(Wk[t], __int2float_rn((int)(sz_k * (it & 0xffffu))));
    m = min(m, pair_key(avg, id_k, it >> 16, threshold));
  }
  return m;
}

__global__ void __launch_bounds__(kAhcThreads) ahc_kernel(const float* __restrict__ scores, const AhcGroup* __restrict__ groups,
                                                         float* __restrict__ w_all, int* __restrict__ ids_all,
                                                         int* __restrict__ labels, int* __restrict__ merge_ids,
                                                         float* __restrict__ merge_costs, int* __restrict__ counts) {
  extern __shared__ __align__(16) unsigned long long ahc_smem[];
  __shared__ float s_tile[kAhcWarps][8][33];            // per-warp stripe of the transposed copy
  __shared__ unsigned long long s_red[kAhcWarps];
  __shared__ int s_res[kRescanList];
  __shared__ int s_nres, s_sa, s_sb, s_szm;
  const AhcGroup G = groups[blockIdx.x];
  const int n = G.n, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (n == 0) {
    if (tid == 0) counts[G.index] = 0;
    return;
  }
  unsigned long long* best = ahc_smem;                                   // [n] cached key of every slot's row
  unsigned* info = reinterpret_cast<unsigned*>(ahc_smem + n);            // [n] id << 16 | size (size 0: inactive slot)
  const float* S = scores + G.s_off;
  float* W = w_all + G.s_off;
  int* parent = ids_all + 4 * G.p_off;                                   // [2n] cluster id -> the id it merged into
  int* slot_of = parent + 2 * n;                                         // [2n] active cluster id -> slot
  int* mids = merge_ids != nullptr ? merge_ids + 2 * G.m_off : nullptr;
  float* mcost = merge_costs != nullptr ? merge_costs + G.m_off : nullptr;
  const float thr = G.threshold;

  for (int i = tid; i < n - 1; i += kAhcThreads) {
    if (mids != nullptr) mids[2 * i] = mids[2 * i + 1] = -1;
    if (mcost != nullptr) mcost[i] = __int_as_float(0x7fffffff);
  }
  for (int s = tid; s < n; s += kAhcThreads) {
    info[s] = ((unsigned)s << 16) | 1u;
    best[s] = kRescan;
    parent[s] = s;
    slot_of[s] = s;
  }
  // W = -S, symmetric from the upper triangle: warps take 32 x 32 tiles (bi <= bj) and write each 8-row stripe
  // straight and, through shared memory, transposed (a lane writes 8 consecutive floats of one of 4 rows)
  const int nb = (n + 31) / 32;
  for (long long t = warp; t < (long long)nb * nb; t += kAhcWarps) {
    const int bi = (int)(t / nb), bj = (int)(t % nb);
    if (bi > bj) continue;
    for (int r0 = 0; r0 < 32; r0 += 8) {
      const int col = bj * 32 + lane;
#pragma unroll
      for (int rr = 0; rr < 8; ++rr) {
        const int row = bi * 32 + r0 + rr;
        float v = 0.0f;
        if (row < n && col < n && row < col) {
          v = -S[(long long)row * n + col];
          W[(long long)row * n + col] = v;
        } else if (row < n && row == col) {
          W[(long long)row * n + col] = 0.0f;                            // (never read)
        }
        s_tile[warp][rr][lane] = v;
      }
      __syncwarp();
      const int rr = lane & 7, trow0 = bi * 32 + r0 + rr;
      for (int c = lane >> 3; c < 32; c += 4) {
        const int trow = bj * 32 + c;
        if (trow < n && trow0 < trow) W[(long long)trow * n + trow0] = s_tile[warp][rr][c];
      }
      __syncwarp();
    }
  }
  __syncthreads();

  // rows flagged kRescan: one warp per row
  auto rescan_flagged = [&]() {
    for (int b = warp * 32; b < n; b += kAhcThreads) {
      unsigned ball = __ballot_sync(0xffffffffu, b + lane < n && best[b + lane] == kRescan);
      while (ball != 0u) {
        const int k = b + __ffs(ball) - 1;
        ball &= ball - 1;
        const unsigned long long m = warp_min(row_min(W + (long long)k * n, info, n, k, lane, 32, thr));
        __syncwarp();
        if (lane == 0) best[k] = m;
      }
    }
  };
  rescan_flagged();
  __syncthreads();

  int clusters = n;
  for (int step = 0; clusters > G.min_clusters; ++step) {
    // the queue's next entry: the smallest cached key of the active slots
    unsigned long long m = kNoPair;
    for (int s = tid; s < n; s += kAhcThreads)
      if (info[s] & 0xffffu) m = min(m, best[s]);
    m = warp_min(m);
    if (lane == 0) s_red[warp] = m;
    __syncthreads();
    unsigned long long key = s_red[0];
    for (int w = 1; w < kAhcWarps; ++w) key = min(key, s_red[w]);
    if (key == kNoPair) break;                                           // (CTA-uniform)
    const unsigned lo = key_lo(key), hi = key_hi(key), new_id = (unsigned)(n + step);
    if (tid == 0) {
      const int sa = slot_of[lo], sb = slot_of[hi];
      if (mids != nullptr) {
        mids[2 * step] = (int)lo;
        mids[2 * step + 1] = (int)hi;
      }
      if (mcost != nullptr) mcost[step] = key_avg(key);
      parent[lo] = parent[hi] = parent[new_id] = (int)new_id;
      slot_of[new_id] = sa;
      s_sa = sa;
      s_sb = sb;
      s_szm = (int)((info[sa] & 0xffffu) + (info[sb] & 0xffffu));
      s_nres = 0;
    }
    __syncthreads();
    const int sa = s_sa, sb = s_sb, szm = s_szm;
    // W(k, m) = W(k, i) + W(k, j) into row and column sa; each slot's cache takes its new pair, or is rescanned when
    // its cached partner was i or j
    float* Wa = W + (long long)sa * n;
    const float* Wb = W + (long long)sb * n;
    unsigned long long mrow = kNoPair;
    for (int k = tid; k < n; k += kAhcThreads) {
      const unsigned ik = info[k];
      if ((ik & 0xffffu) == 0u || k == sa || k == sb) continue;
      const float w = __fadd_rn(Wa[k], Wb[k]);
      Wa[k] = w;
      W[(long long)k * n + sa] = w;
      const unsigned id_k = ik >> 16;
      const unsigned long long nk = pair_key(__fdiv_rn(w, __int2float_rn(szm * (int)(ik & 0xffffu))), id_k, new_id, thr);
      mrow = min(mrow, nk);
      const unsigned long long pb = best[k];
      if (pb != kNoPair) {
        const unsigned partner = key_lo(pb) == id_k ? key_hi(pb) : key_lo(pb);
        if (partner == lo || partner == hi) {
          const int at = atomicAdd(&s_nres, 1);
          if (at < kRescanList) s_res[at] = k;
          best[k] = kRescan;
          continue;
        }
      }
      best[k] = min(pb, nk);
    }
    mrow = warp_min(mrow);
    if (lane == 0) s_red[warp] = mrow;                                   // (every thread read the key before s_sa)
    __syncthreads();
    if (tid == 0) {
      unsigned long long r = s_red[0];
      for (int w = 1; w < kAhcWarps; ++w) r = min(r, s_red[w]);
      best[sa] = r;
      info[sa] = (new_id << 16) | (unsigned)szm;
      info[sb] = 0u;
    }
    __syncthreads();
    // the first kRescanList flagged rows with the whole CTA, any others one warp per row
    const int nres = min(s_nres, kRescanList);
    for (int i = 0; i < nres; ++i) {
      const int k = s_res[i];
      const unsigned long long r = warp_min(row_min(W + (long long)k * n, info, n, k, tid, kAhcThreads, thr));
      if (lane == 0) s_red[warp] = r;
      __syncthreads();
      if (tid == 0) {
        unsigned long long b = s_red[0];
        for (int w = 1; w < kAhcWarps; ++w) b = min(b, s_red[w]);
        best[k] = b;
      }
      __syncthreads();
    }
    if (s_nres > kRescanList) {                                          // (CTA-uniform)
      rescan_flagged();
      __syncthreads();
    }
    --clusters;
  }
  if (tid == 0) counts[G.index] = clusters;

  // labels: every point's root (pointer jumping over the parent ids), then the roots' ranks in id order
  const int num_ids = n + (n - clusters);
  for (;;) {
    int changed = 0;
    for (int x = tid; x < num_ids; x += kAhcThreads) {
      const int p = parent[x], pp = parent[p];
      if (pp != p) {
        parent[x] = pp;
        changed = 1;
      }
    }
    if (!__syncthreads_or(changed)) break;
  }
  int* rank = slot_of;                                                   // (slot_of is no longer needed)
  for (int x = tid; x < num_ids; x += kAhcThreads) rank[x] = 0;
  __syncthreads();
  for (int s = tid; s < n; s += kAhcThreads)
    if (info[s] & 0xffffu) rank[info[s] >> 16] = 1;
  __syncthreads();
  // exclusive prefix count of the root flags: thread t owns ids [t per, (t + 1) per)
  const int per = (num_ids + kAhcThreads - 1) / kAhcThreads, x0 = min(tid * per, num_ids), x1 = min(x0 + per, num_ids);
  int local = 0;
  for (int x = x0; x < x1; ++x) local += rank[x];
  int incl = local;
  for (int o = 1; o < 32; o <<= 1) {
    const int v = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += v;
  }
  __shared__ int s_wsum[kAhcWarps];
  if (lane == 31) s_wsum[warp] = incl;
  __syncthreads();
  int run = incl - local;
  for (int w = 0; w < warp; ++w) run += s_wsum[w];
  for (int x = x0; x < x1; ++x) {
    const int f = rank[x];
    rank[x] = run;
    run += f;
  }
  __syncthreads();
  for (int p = tid; p < n; p += kAhcThreads) labels[G.p_off + p] = rank[parent[p]] + 1;
}

}  // namespace

extern "C" int ktf_ahc_cluster(const float* scores_dev, const int64_t* offsets_host, int32_t num_groups, float threshold,
                               const int32_t* num_clusters_host, int32_t* labels_dev, int32_t* merge_ids_dev,
                               float* merge_costs_dev, int32_t* cluster_counts_dev, void* stream) {
  KTF_CHECK_ARG(num_groups >= 0, "ktf_ahc_cluster: num_groups = %d, must be >= 0", num_groups);
  if (num_groups == 0) return KTF_OK;
  KTF_CHECK_ARG(offsets_host && cluster_counts_dev, "ktf_ahc_cluster: null argument");
  std::vector<AhcGroup> groups((size_t)num_groups);
  long long s_off = 0, m_off = 0, max_n = 0;
  for (int32_t g = 0; g < num_groups; ++g) {
    const long long n = offsets_host[g + 1] - offsets_host[g];
    KTF_CHECK_ARG(n >= 0, "ktf_ahc_cluster: group %d has a negative length", g);
    KTF_CHECK_ARG(n <= KTF_AHC_MAX_POINTS, "ktf_ahc_cluster: group %d has %lld points, more than KTF_AHC_MAX_POINTS (%d)",
                  g, n, KTF_AHC_MAX_POINTS);
    KTF_CHECK_ARG(num_clusters_host == nullptr || num_clusters_host[g] >= 1,
                  "ktf_ahc_cluster: num_clusters[%d] = %d, must be >= 1", g, num_clusters_host ? num_clusters_host[g] : 0);
    groups[g] = AhcGroup{s_off, offsets_host[g] - offsets_host[0], m_off, (int)n,
                         num_clusters_host ? num_clusters_host[g] : 1, num_clusters_host ? FLT_MAX : threshold, g};
    s_off += n * n;
    m_off += std::max(n - 1, 0LL);
    max_n = std::max(max_n, n);
  }
  const long long points = offsets_host[num_groups] - offsets_host[0];
  if (points > 0) KTF_CHECK_ARG(scores_dev && labels_dev, "ktf_ahc_cluster: null argument");
  std::stable_sort(groups.begin(), groups.end(), [](const AhcGroup& a, const AhcGroup& b) { return a.n > b.n; });
  cudaStream_t st = (cudaStream_t)stream;
  ktf::Scratch scratch(st);            // released on every exit path
  const size_t table_bytes = ((size_t)num_groups * sizeof(AhcGroup) + 255) & ~(size_t)255;
  const size_t w_bytes = ((size_t)s_off * sizeof(float) + 255) & ~(size_t)255;
  char* base = nullptr;
  KTF_CUDA(scratch.take(&base, table_bytes + w_bytes + (size_t)points * 4 * sizeof(int) + 256));
  AhcGroup* table = reinterpret_cast<AhcGroup*>(base);
  float* w = reinterpret_cast<float*>(base + table_bytes);
  int* ids = reinterpret_cast<int*>(base + table_bytes + w_bytes);
  // pageable source: cudaMemcpyAsync returns once it is staged (no device synchronisation), so `groups` may die
  KTF_CUDA(cudaMemcpyAsync(table, groups.data(), (size_t)num_groups * sizeof(AhcGroup), cudaMemcpyHostToDevice, st));
  const size_t smem = (size_t)max_n * (sizeof(unsigned long long) + sizeof(unsigned));
  static unsigned long long attr_done = 0;
  if (ktf::first_use_on_device(&attr_done))
    KTF_CUDA(cudaFuncSetAttribute(ahc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)(KTF_AHC_MAX_POINTS * (sizeof(unsigned long long) + sizeof(unsigned)))));
  ahc_kernel<<<(unsigned)num_groups, kAhcThreads, smem, st>>>(scores_dev, table, w, ids, labels_dev, merge_ids_dev,
                                                              merge_costs_dev, cluster_counts_dev);
  KTF_LAUNCH_OK();
  return KTF_OK;
}

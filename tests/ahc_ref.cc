// Compiled reference of the diarization back-end's clustering: Kaldi's single-pass AgglomerativeClusterer
// (ivector/agglomerative-clustering.cc) restated in C++, the contract of tests/ahc_oracle.py, fast enough for recordings
// of KTF_AHC_MAX_POINTS segments.  It keeps Kaldi's priority queue with lazy deletion (not the GPU kernel's per-row
// cached minima), so it stays independent of the kernel it checks.  tests/ahc_testlib.py compiles it with
// -ffp-contract=off and without -ffast-math: every float operation is one IEEE float32 operation.
#include <cfloat>
#include <cstdint>
#include <queue>
#include <vector>

namespace {

// A queue entry (avg, lower id, higher id); ids stay below 2 * 16384 - 1, so 16 bits hold them.
struct Entry {
  float avg;
  uint16_t lo, hi;
};

// The priority queue's order: smallest (avg, lo, hi) first, field by field, so -0 and +0 are the same avg.
struct Later {
  bool operator()(const Entry& x, const Entry& y) const {
    if (x.avg != y.avg) return x.avg > y.avg;
    if (x.lo != y.lo) return x.lo > y.lo;
    return x.hi > y.hi;
  }
};

}  // namespace

// Clusters the n x n row-major scores S (only the upper triangle is read): cost(a, b) = -S[min][max]; pairs with
// avg <= thr enter the queue (NaN never does); merging stops at min_clusters clusters or an empty queue.  Writes the
// labels (n: the final clusters in increasing id order are 1 .. C) and the merges (lower id, higher id) to merge_ids
// (2 per merge) and their avg to merge_costs (n - 1 entries of room each), and returns the number of merges, or -1
// when n is out of range.
extern "C" int ahc_ref(const float* S, int n, float thr, int min_clusters, int* labels, int* merge_ids,
                       float* merge_costs) {
  if (n < 0 || n > 32768) return -1;
  const size_t nn = (size_t)n;
  std::vector<float> W(nn * nn);                     // by slot: slot s holds cluster id[s]
  for (size_t i = 0; i < nn; ++i)
    for (size_t j = i + 1; j < nn; ++j) W[i * nn + j] = W[j * nn + i] = -S[i * nn + j];
  std::vector<int> id(nn), size(nn, 1), slot(2 * nn, -1), parent(2 * nn);
  std::vector<char> alive(nn, 1);
  std::vector<Entry> init;
  init.reserve(nn * (nn - (n > 0)) / 2);
  for (int i = 0; i < n; ++i) {
    id[i] = slot[i] = parent[i] = i;
    for (int j = i + 1; j < n; ++j)
      if (W[i * nn + j] <= thr) init.push_back(Entry{W[i * nn + j], (uint16_t)i, (uint16_t)j});
  }
  std::priority_queue<Entry, std::vector<Entry>, Later> queue(Later(), std::move(init));
  int clusters = n, merges = 0;
  while (clusters > min_clusters && !queue.empty()) {
    const Entry e = queue.top();
    queue.pop();
    const int si = slot[e.lo], sj = slot[e.hi];
    if (si < 0 || sj < 0) continue;                  // a cluster of the entry has been merged: stale
    const int m = n + merges;
    merge_ids[2 * merges] = e.lo;
    merge_ids[2 * merges + 1] = e.hi;
    merge_costs[merges] = e.avg;
    ++merges;
    slot[e.lo] = slot[e.hi] = -1;
    parent[e.lo] = parent[e.hi] = parent[m] = m;
    alive[sj] = 0;
    const int size_m = size[si] + size[sj];
    for (size_t k = 0; k < nn; ++k) {
      if (!alive[k] || (int)k == si) continue;
      const float w = W[(size_t)si * nn + k] + W[(size_t)sj * nn + k];
      W[(size_t)si * nn + k] = W[k * nn + si] = w;
      const float avg = w / (float)(size[k] * size_m);
      if (avg <= thr) queue.push(Entry{avg, (uint16_t)id[k], (uint16_t)m});
    }
    id[si] = m;
    size[si] = size_m;
    slot[m] = si;
    --clusters;
  }
  // labels: every point's root, then the roots' ranks in id order
  std::vector<int> rank(nn + merges, 0);
  for (int x = n + merges - 1; x >= 0; --x) parent[x] = parent[parent[x]];   // parents have higher ids: one pass
  for (int s = 0; s < n; ++s)
    if (alive[s]) rank[id[s]] = 1;
  for (int x = 0, r = 0; x < n + merges; ++x)
    if (rank[x]) rank[x] = ++r;
  for (int p = 0; p < n; ++p) labels[p] = rank[parent[p]];
  return merges;
}

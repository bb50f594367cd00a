// Lockstep agglomeration of erickson_SVD (splitp/phylogenetics.py:99-171) for many replicates at once.
//
// Every replicate keeps its clusters as ids: leaves 0 .. n-1, the cluster merged at step t gets id n + t.  The current
// clusters are held in ascending id order, which is erickson_SVD's list order (the remaining clusters keep their order, the
// merged one is appended), so `combinations` over that list enumerates pairs (a < b) of list positions lexicographically.
// A candidate split joins clusters x and y against all others; its score does not change while x and y exist, so it is
// scored once and kept in a per-replicate cache keyed by (x, y).  A step therefore scores only the pairs with the cluster
// merged last: C(n, 2) candidates at step 0 (agglomerate_init_kernel), m - 2 after a step with m clusters.
//
// Candidates are written in the orientation erickson_SVD scores (score_canonical): the side holding taxon `first` (the
// taxon with the smallest name) is side A.  The step kernel (one CTA per replicate) stores the step's scores in the cache,
// finds the first minimum over all current pairs in combinations order -- (score, pair index) compared lexicographically,
// so the reduction order cannot change the pick -- records the joined side and its score, merges, and writes the next
// step's candidates.  A NaN score is ordered as +inf: subflattening scores are NaN only for an all-zero subflattening.
#include "common.cuh"

#include <limits.h>
#include <math.h>

using namespace spb;

namespace {

constexpr int kAThreads = 256;

// Per-replicate state: cluster masks [2n - 1], score cache [2n - 1][2n - 1] (entry [x][y], x < y), current order [n] (ids).
__host__ __device__ inline int64_t rep_bytes(int n) {
  const int64_t nid = 2 * n - 1;
  return ((8 * nid + 8 * nid * nid + 4 * (int64_t)n) + 15) / 16 * 16;
}

struct RepState {
  uint64_t* masks;
  double* cache;
  int* order;
};

__device__ __forceinline__ RepState rep_state(unsigned char* ws, int n, int64_t r) {
  const int64_t nid = 2 * n - 1;
  unsigned char* base = ws + r * rep_bytes(n);
  return RepState{reinterpret_cast<uint64_t*>(base), reinterpret_cast<double*>(base + 8 * nid),
                  reinterpret_cast<int*>(base + 8 * nid + 8 * nid * nid)};
}

__device__ __forceinline__ void write_candidate(uint64_t joined, uint64_t full, int first, uint64_t* ma, uint64_t* mb, int64_t i) {
  const uint64_t rest = full & ~joined;
  const bool joined_first = (joined >> first) & 1ull;
  ma[i] = joined_first ? joined : rest;
  mb[i] = joined_first ? rest : joined;
}

__global__ void agglomerate_init_kernel(int n, int64_t reps, int first, uint64_t* __restrict__ ma, uint64_t* __restrict__ mb,
                                        unsigned char* ws) {
  const uint64_t full = (n == 64) ? ~0ull : ((1ull << n) - 1ull);
  const int64_t npairs = (int64_t)n * (n - 1) / 2;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < reps * npairs; g += stride) {
    const int64_t r = g / npairs;
    int rem = (int)(g - r * npairs), i = 0;
    while (rem >= n - 1 - i) { rem -= n - 1 - i; ++i; }  // combinations order: (0,1), (0,2), ..., (1,2), ...
    const int j = i + 1 + rem;
    write_candidate((1ull << i) | (1ull << j), full, first, ma, mb, g);
  }
  for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < reps * n; g += stride) {
    const int64_t r = g / n;
    const int i = (int)(g - r * n);
    const RepState st = rep_state(ws, n, r);
    st.masks[i] = 1ull << i;
    st.order[i] = i;
  }
}

__device__ __forceinline__ bool before(double v, int p, double w, int q) { return v < w || (v == w && p < q); }

__global__ void __launch_bounds__(kAThreads) agglomerate_step_kernel(int n, int step, int first, const double* __restrict__ scores,
                                                                     int64_t per_table, uint64_t* __restrict__ ma,
                                                                     uint64_t* __restrict__ mb, unsigned char* ws, uint64_t* chosen,
                                                                     double* chosen_scores) {
  __shared__ int s_order[SPB_MAX_TAXA];
  __shared__ double s_best[kAThreads / 32];
  __shared__ int s_idx[kAThreads / 32];
  __shared__ uint64_t s_joined;
  const int64_t r = blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31;
  const int m = n - step;  // current clusters
  const int nid = 2 * n - 1;
  const RepState st = rep_state(ws, n, r);
  if (tid < m) s_order[tid] = st.order[tid];
  __syncthreads();
  // this step's scores into the cache
  const double* sc = scores + r * per_table;
  if (step == 0) {
    for (int p = tid; p < per_table; p += kAThreads) {
      int rem = p, i = 0;
      while (rem >= n - 1 - i) { rem -= n - 1 - i; ++i; }
      st.cache[i * nid + i + 1 + rem] = sc[p];
    }
  } else {
    const int y = s_order[m - 1];  // the cluster merged last: largest id, last in the order
    for (int q = tid; q < m - 1; q += kAThreads) st.cache[s_order[q] * nid + y] = sc[q];
  }
  __syncthreads();
  // first minimum over the pairs (a < b) of list positions; p = index of (a, b) in combinations order
  double best = INFINITY;
  int bidx = INT_MAX;
  for (int e = tid; e < m * m; e += kAThreads) {
    const int a = e / m, b = e - a * m;
    if (a >= b) continue;
    double v = st.cache[s_order[a] * nid + s_order[b]];
    if (v != v) v = INFINITY;
    const int p = a * (2 * m - a - 1) / 2 + (b - a - 1);
    if (before(v, p, best, bidx)) { best = v; bidx = p; }
  }
  for (int o = 16; o > 0; o >>= 1) {
    const double ov = __shfl_xor_sync(0xFFFFFFFFu, best, o);
    const int op = __shfl_xor_sync(0xFFFFFFFFu, bidx, o);
    if (before(ov, op, best, bidx)) { best = ov; bidx = op; }
  }
  if (lane == 0) { s_best[tid >> 5] = best; s_idx[tid >> 5] = bidx; }
  __syncthreads();
  if (tid == 0) {
    for (int w = 1; w < kAThreads / 32; ++w)
      if (before(s_best[w], s_idx[w], best, bidx)) { best = s_best[w]; bidx = s_idx[w]; }
    int a = 0, rem = bidx;
    while (rem >= m - 1 - a) { rem -= m - 1 - a; ++a; }
    const int b = a + 1 + rem;
    const int x = s_order[a], y = s_order[b];
    const uint64_t joined = st.masks[x] | st.masks[y];
    chosen[r * (n - 2) + step] = joined;
    chosen_scores[r * (n - 2) + step] = st.cache[x * nid + y];
    st.masks[n + step] = joined;
    int w = 0;
    for (int i = 0; i < m; ++i)
      if (i != a && i != b) s_order[w++] = s_order[i];
    s_order[w] = n + step;
    s_joined = joined;
  }
  __syncthreads();
  if (tid < m - 1) st.order[tid] = s_order[tid];
  if (step + 1 < n - 2) {  // the next step's candidates: every remaining cluster with the merged one
    const uint64_t full = (n == 64) ? ~0ull : ((1ull << n) - 1ull);
    const uint64_t joined = s_joined;
    for (int q = tid; q < m - 2; q += kAThreads)
      write_candidate(st.masks[s_order[q]] | joined, full, first, ma, mb, r * (m - 2) + q);
  }
}

}  // namespace

extern "C" int64_t spb_agglomerate_ws_bytes(int n_taxa, int64_t reps) {
  if (n_taxa < 3 || n_taxa > SPB_MAX_TAXA || reps < 0) return 0;
  return reps * rep_bytes(n_taxa);
}

extern "C" int spb_agglomerate_init(int n_taxa, int64_t reps, int first_taxon, uint64_t* d_ma, uint64_t* d_mb, void* d_ws,
                                    void* stream) {
  SPB_REQUIRE(n_taxa >= 3 && n_taxa <= SPB_MAX_TAXA && first_taxon >= 0 && first_taxon < n_taxa && reps >= 0 &&
                  reps <= 0x7FFFFFFF,
              "spb_agglomerate_init: bad arguments");
  if (reps == 0) return SPB_OK;
  SPB_REQUIRE(d_ma && d_mb && d_ws, "spb_agglomerate_init: NULL buffer");
  const int64_t work = reps * n_taxa * (n_taxa - 1) / 2;
  int64_t grid = (work + 255) / 256;
  if (grid > (int64_t)sm_count() * 8) grid = (int64_t)sm_count() * 8;
  agglomerate_init_kernel<<<(unsigned)grid, 256, 0, (cudaStream_t)stream>>>(n_taxa, reps, first_taxon, d_ma, d_mb,
                                                                           (unsigned char*)d_ws);
  SPB_LAUNCH_CHECK();
  return SPB_OK;
}

extern "C" int spb_agglomerate_step(int n_taxa, int64_t reps, int step, int first_taxon, const double* d_scores, uint64_t* d_ma,
                                    uint64_t* d_mb, void* d_ws, uint64_t* d_chosen, double* d_chosen_scores, void* stream) {
  SPB_REQUIRE(n_taxa >= 3 && n_taxa <= SPB_MAX_TAXA && step >= 0 && step < n_taxa - 2 && first_taxon >= 0 &&
                  first_taxon < n_taxa && reps >= 0 && reps <= 0x7FFFFFFF,
              "spb_agglomerate_step: bad arguments");
  if (reps == 0) return SPB_OK;
  SPB_REQUIRE(d_scores && d_ma && d_mb && d_ws && d_chosen && d_chosen_scores, "spb_agglomerate_step: NULL buffer");
  const int64_t per_table = step == 0 ? (int64_t)n_taxa * (n_taxa - 1) / 2 : n_taxa - step - 1;
  agglomerate_step_kernel<<<(unsigned)reps, kAThreads, 0, (cudaStream_t)stream>>>(n_taxa, step, first_taxon, d_scores, per_table,
                                                                                 d_ma, d_mb, (unsigned char*)d_ws, d_chosen,
                                                                                 d_chosen_scores);
  SPB_LAUNCH_CHECK();
  return SPB_OK;
}

// Quartet split scores: the joint count table of every listed quartet, read from the bit planes, and the three 2|2
// flattenings of each table scored in one call (replaces the reference's per-quartet loop
// Alignment.sub_alignment([a, b, c, d]) -> flattening(split, sub, FlatFormat.reduced) -> split_score, three times).
//
// spb_quartet_tables: a CTA owns kQPerCta quartets and a run of 64-word tiles of the sites.  For every tile the low / high
// planes of the quartets' taxa go to shared memory; thread (quartet, ab-state x y) forms ab = [x_a = x][x_b = y][usable] once
// per word and keeps 16 counters popc(ab & [x_c = z] & [x_d = w]).  The counters are uint32 (a CTA's site run is far below
// 2^32 sites) and are flushed with one 64-bit atomic per non-zero counter per CTA, as pair_kernel flushes its raw row, so the
// tables are exact integers and do not depend on the schedule.  Work: Q x 256 AND + POPC per 32-site word.
//
// Flattening scores: for each (quartet, pairing) the 16 x 16 count flattening is a re-indexing of the table; its fp64 Gram
// (rows = the side holding the quartet's first taxon) goes to spb_score_gram_small (k = 16: the warp Householder + 9-section
// path of pairs.cu).  Beside it the number of non-empty rows and columns is kept: at most 4 of either scores exactly 0.0 (at
// most 4 singular values), an all-zero table NaN, as split_score gives for the reduced flattening.
//
// Rank-1 divergence: one warp per quartet computes the row and column sums of each pairing's flattening exactly as integers,
// then sum v log(v / (r c)) over the non-zero cells of the probability flattening (counts / usable sites) with a fixed
// per-lane order and a fixed butterfly: the result does not depend on the launch configuration.
#include "common.cuh"

using namespace spb;

namespace {

constexpr int kQThreads = 256;
constexpr int kQPerCta = kQThreads / 16;  // 16 ab-states per quartet
constexpr int kQSlots = kQPerCta * 4;     // taxon rows staged per tile
constexpr int kQW = 64;                   // plane words per tile (2048 sites)
constexpr int64_t kQMinTilesPerChunk = 8;  // a site chunk costs one flush of its CTA's counters: keep chunks at least this long

// mask of the sites where a taxon with planes (lo, hi) is in state s (A=0 C=1 G=2 T=3: lo = bit 0, hi = bit 1)
__device__ __forceinline__ uint32_t state_mask(uint2 p, int s) {
  return ((s & 1) ? p.x : ~p.x) & ((s & 2) ? p.y : ~p.y);
}

__global__ void __launch_bounds__(kQThreads) quartet_tables_kernel(const uint32_t* __restrict__ planes, const uint32_t* __restrict__ valid,
                                                                   int n, int64_t Wp, int64_t word_begin, int64_t word_end,
                                                                   const uint8_t* __restrict__ quartets, int64_t Q, int64_t chunk_tiles,
                                                                   unsigned long long* __restrict__ tables) {
  __shared__ uint2 s_pl[kQSlots][kQW];  // {lo, hi} of each staged taxon row
  __shared__ uint32_t s_valid[kQW];
  __shared__ int s_tax[kQSlots];
  const int tid = threadIdx.x;
  const int ql = tid >> 4, x = (tid >> 2) & 3, y = tid & 3;
  const int64_t q = (int64_t)blockIdx.x * kQPerCta + ql;
  if (tid < kQSlots) {  // a quartet past the end or with a taxon out of range stages taxon 0 and is not counted
    const int64_t qq = (int64_t)blockIdx.x * kQPerCta + (tid >> 2);
    const int t = qq < Q ? (int)quartets[qq * 4 + (tid & 3)] : 0;
    s_tax[tid] = t < n ? t : -1;
  }
  __syncthreads();
  const int sa = ql * 4;
  const bool active = q < Q && s_tax[sa] >= 0 && s_tax[sa + 1] >= 0 && s_tax[sa + 2] >= 0 && s_tax[sa + 3] >= 0;
  uint32_t cnt[16];
#pragma unroll
  for (int e = 0; e < 16; ++e) cnt[e] = 0;
  const int64_t tile0 = word_begin / kQW, tile1 = (word_end + kQW - 1) / kQW;
  const int64_t t_lo = tile0 + (int64_t)blockIdx.y * chunk_tiles;
  const int64_t t_hi = t_lo + chunk_tiles < tile1 ? t_lo + chunk_tiles : tile1;
  for (int64_t tile = t_lo; tile < t_hi; ++tile) {
    const int64_t wbase = tile * kQW;
    __syncthreads();
    for (int idx = tid; idx < kQSlots * kQW; idx += kQThreads) {
      const int s = idx / kQW, w = idx - s * kQW;
      const int64_t gw = wbase + w;
      const int t = s_tax[s];
      uint2 p = make_uint2(0u, 0u);
      if (t >= 0 && gw >= word_begin && gw < word_end) {
        p.x = __ldg(planes + ((int64_t)t * 2) * Wp + gw);
        p.y = __ldg(planes + ((int64_t)t * 2 + 1) * Wp + gw);
      }
      s_pl[s][w] = p;
    }
    if (tid < kQW) {
      const int64_t gw = wbase + tid;
      s_valid[tid] = (gw >= word_begin && gw < word_end) ? __ldg(valid + gw) : 0u;
    }
    __syncthreads();
    if (!active) continue;
#pragma unroll 4
    for (int w = 0; w < kQW; ++w) {
      const uint32_t ab = state_mask(s_pl[sa][w], x) & state_mask(s_pl[sa + 1][w], y) & s_valid[w];
      const uint2 c = s_pl[sa + 2][w], d = s_pl[sa + 3][w];
#pragma unroll
      for (int z = 0; z < 4; ++z) {
        const uint32_t abc = ab & state_mask(c, z);
#pragma unroll
        for (int v = 0; v < 4; ++v) cnt[z * 4 + v] += __popc(abc & state_mask(d, v));
      }
    }
  }
  if (!active) return;
  unsigned long long* row = tables + q * 256 + (x * 4 + y) * 16;  // cell 64 x_a + 16 x_b + 4 x_c + x_d
#pragma unroll
  for (int e = 0; e < 16; ++e)
    if (cnt[e]) atomicAdd(row + e, (unsigned long long)cnt[e]);
}

// cell of the table holding entry (r, c) of the flattening of pairing p: p = 0 {a,b}|{c,d}, 1 {a,c}|{b,d}, 2 {a,d}|{b,c};
// r = 4 x_a + x_(partner of a), c = 4 x_(first other) + x_(second other)
__device__ __forceinline__ int pairing_cell(int p, int r, int c) {
  const int xa = r >> 2, xp = r & 3, xu = c >> 2, xv = c & 3;
  if (p == 0) return 64 * xa + 16 * xp + 4 * xu + xv;
  if (p == 1) return 64 * xa + 16 * xu + 4 * xp + xv;
  return 64 * xa + 16 * xu + 4 * xv + xp;
}

// one CTA per quartet at a time: the table to shared memory, then thread (r, r') forms G_p[r][r'] of the three pairings in a
// fixed order, and the non-empty rows / columns of each pairing are counted
__global__ void __launch_bounds__(256) quartet_gram_kernel(const unsigned long long* __restrict__ tables, int64_t Q, double* __restrict__ G,
                                                           int32_t* __restrict__ used) {
  __shared__ double s_t[256];
  __shared__ int s_nz[2][3][16];  // [rows / columns][pairing][index]
  const int tid = threadIdx.x, r = tid >> 4, r2 = tid & 15;
  for (int64_t q = blockIdx.x; q < Q; q += gridDim.x) {
    __syncthreads();
    s_t[tid] = (double)tables[q * 256 + tid];
    __syncthreads();
#pragma unroll
    for (int p = 0; p < 3; ++p) {
      double g = 0.0;
#pragma unroll
      for (int c = 0; c < 16; ++c) g = fma(s_t[pairing_cell(p, r, c)], s_t[pairing_cell(p, r2, c)], g);
      G[((q * 3 + p) * 16 + r) * 16 + r2] = g;
    }
    if (tid < 96) {  // 2 x 3 x 16 lines: any non-zero cell in row (or column) i of pairing p
      const int kind = tid / 48, p = (tid / 16) % 3, i = tid & 15;
      int nz = 0;
      for (int j = 0; j < 16; ++j) nz |= s_t[kind ? pairing_cell(p, j, i) : pairing_cell(p, i, j)] != 0.0;
      s_nz[kind][p][i] = nz;
    }
    __syncthreads();
    if (tid < 3) {
      int rows = 0, cols = 0;
      for (int i = 0; i < 16; ++i) { rows += s_nz[0][tid][i]; cols += s_nz[1][tid][i]; }
      used[q * 3 + tid] = rows < cols ? rows : cols;
    }
  }
}

// the reduced flattening's rule: no non-empty line -> NaN (empty matrix), at most 4 on the short side -> 0.0
__global__ void quartet_fix_kernel(const int32_t* __restrict__ used, int64_t num, double* __restrict__ scores) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= num) return;
  const int u = used[i];
  if (u == 0) scores[i] = nan("");
  else if (u <= 4) scores[i] = 0.0;
}

constexpr int kMWarps = 8;

__global__ void __launch_bounds__(32 * kMWarps) quartet_mi_kernel(const unsigned long long* __restrict__ tables, int64_t Q,
                                                                  double* __restrict__ out) {
  __shared__ unsigned long long s_t[kMWarps][256];
  __shared__ unsigned long long s_sum[kMWarps][32];  // row sums 0..15, column sums 16..31 of the current pairing
  const int lane = threadIdx.x & 31, wi = threadIdx.x >> 5;
  unsigned long long* t = s_t[wi];
  unsigned long long* sums = s_sum[wi];
  const int64_t nwarps = (int64_t)gridDim.x * kMWarps;
  for (int64_t q = (int64_t)blockIdx.x * kMWarps + wi; q < Q; q += nwarps) {
    __syncwarp();
    unsigned long long part = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const unsigned long long v = tables[q * 256 + k * 32 + lane];
      t[k * 32 + lane] = v;
      part += v;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
    const double N = (double)part;  // usable sites
    __syncwarp();
#pragma unroll 1
    for (int p = 0; p < 3; ++p) {
      unsigned long long s = 0;
      for (int j = 0; j < 16; ++j) s += t[lane < 16 ? pairing_cell(p, lane, j) : pairing_cell(p, j, lane - 16)];
      sums[lane] = s;
      __syncwarp();
      double acc = 0.0;
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const int e = k * 32 + lane, r = e >> 4, c = e & 15;
        const unsigned long long v = t[pairing_cell(p, r, c)];
        if (v) {
          const double f = (double)v / N, rc = ((double)sums[16 + c] / N) * ((double)sums[r] / N);
          acc += f * log(f / rc);
        }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
      if (lane == 0) out[q * 3 + p] = acc;  // an empty table has no non-zero cell: 0.0
      __syncwarp();
    }
  }
}

}  // namespace

extern "C" int spb_quartet_tables(const uint32_t* d_planes, const uint32_t* d_valid, int n_taxa, int64_t plane_words, int64_t word_begin,
                                  int64_t word_end, const uint8_t* d_quartets, int64_t num, uint64_t* d_tables, void* stream) {
  SPB_REQUIRE(n_taxa >= 4 && n_taxa <= SPB_MAX_TAXA, "spb_quartet_tables: n_taxa must be 4..%d (got %d)", SPB_MAX_TAXA, n_taxa);
  SPB_REQUIRE(num >= 0 && word_begin >= 0 && word_begin <= word_end && word_end <= plane_words,
              "spb_quartet_tables: bad range (num=%lld, words [%lld, %lld) of %lld)", (long long)num, (long long)word_begin,
              (long long)word_end, (long long)plane_words);
  if (num == 0 || word_begin == word_end) return SPB_OK;
  SPB_REQUIRE(d_planes && d_valid && d_quartets && d_tables, "spb_quartet_tables: NULL buffer");
  const int64_t qblocks = (num + kQPerCta - 1) / kQPerCta;
  SPB_REQUIRE(qblocks <= 0x7FFFFFFF, "spb_quartet_tables: too many quartets (%lld)", (long long)num);
  const int64_t tiles = (word_end + kQW - 1) / kQW - word_begin / kQW;
  // site chunks: enough CTAs for several waves, but no chunk under kQMinTilesPerChunk tiles
  int64_t chunks = (8 * (int64_t)sm_count() + qblocks - 1) / qblocks;
  const int64_t most = (tiles + kQMinTilesPerChunk - 1) / kQMinTilesPerChunk;
  if (chunks > most) chunks = most;
  if (chunks > 65535) chunks = 65535;
  if (chunks < 1) chunks = 1;
  const int64_t chunk_tiles = (tiles + chunks - 1) / chunks;
  chunks = (tiles + chunk_tiles - 1) / chunk_tiles;
  SPB_REQUIRE(chunk_tiles * kQW * 32 < (1ll << 32), "spb_quartet_tables: too many sites for 32-bit counters");
  quartet_tables_kernel<<<dim3((unsigned)qblocks, (unsigned)chunks), kQThreads, 0, (cudaStream_t)stream>>>(
      d_planes, d_valid, n_taxa, plane_words, word_begin, word_end, d_quartets, num, chunk_tiles, (unsigned long long*)d_tables);
  SPB_LAUNCH_CHECK();
  return SPB_OK;
}

extern "C" int64_t spb_quartet_flattening_ws(int64_t num) { return num * 3 * 256 + (num * 3 + 1) / 2; }

extern "C" int spb_quartet_flattening_scores(const uint64_t* d_tables, int64_t num, double* d_ws, double* d_scores, void* stream) {
  SPB_REQUIRE(num >= 0 && num <= INT64_MAX / 1024, "spb_quartet_flattening_scores: bad size (num=%lld)", (long long)num);
  if (num == 0) return SPB_OK;
  SPB_REQUIRE(d_tables && d_ws && d_scores, "spb_quartet_flattening_scores: NULL buffer");
  cudaStream_t st = (cudaStream_t)stream;
  double* G = d_ws;
  int32_t* used = reinterpret_cast<int32_t*>(d_ws + num * 3 * 256);
  int64_t grid = (int64_t)sm_count() * 8;
  if (grid > num) grid = num;
  quartet_gram_kernel<<<(unsigned)grid, 256, 0, st>>>((const unsigned long long*)d_tables, num, G, used);
  SPB_LAUNCH_CHECK();
  int rc = spb_score_gram_small(G, 16, 16, num * 3, d_scores, nullptr, stream);
  if (rc) return rc;
  quartet_fix_kernel<<<(unsigned)((num * 3 + 255) / 256), 256, 0, st>>>(used, num * 3, d_scores);
  SPB_LAUNCH_CHECK();
  return SPB_OK;
}

extern "C" int spb_quartet_mi_scores(const uint64_t* d_tables, int64_t num, double* d_scores, void* stream) {
  SPB_REQUIRE(num >= 0, "spb_quartet_mi_scores: bad size (num=%lld)", (long long)num);
  if (num == 0) return SPB_OK;
  SPB_REQUIRE(d_tables && d_scores, "spb_quartet_mi_scores: NULL buffer");
  int64_t grid = (int64_t)sm_count() * 8;
  const int64_t need = (num + kMWarps - 1) / kMWarps;
  if (grid > need) grid = need;
  quartet_mi_kernel<<<(unsigned)grid, 32 * kMWarps, 0, (cudaStream_t)stream>>>((const unsigned long long*)d_tables, num, d_scores);
  SPB_LAUNCH_CHECK();
  return SPB_OK;
}

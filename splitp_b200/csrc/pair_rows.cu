// Joint pair tables of many count rows over one sorted pattern list (spb_pair_tables_count_rows): the pair tables of a
// table and of all its bootstrap replicates from their count rows, in one launch.
//
// Row r's table is N_r[i][j][x][y] = sum_p counts[r][p] [digit i of key p = x][digit j of key p = y].  The work items are
// the combinations (row r, taxon pair i <= j), R n (n + 1) / 2 of them in row-major order; CTA (t, c) takes the kRTile
// combinations of tile t over the patterns of chunk c.  A thread owns kRCombos combinations and their 16 cells each, as
// uint32 counters in shared memory at [combination][cell][thread] (no atomics, no bank conflicts: a thread only touches
// its own column).  The patterns are staged in shared memory, keys once for the whole CTA and counts of the rows the tile
// spans, and every thread adds each pattern's count of its row to the cell its two digits select.  A warp's combinations
// are consecutive, so they mostly share a row and skip a zero count together.  At the end the CTA adds its non-zero
// counters to N with fp64 atomics, to (i, j) and to the mirrored (j, i).
//
// Exactness: a row sums to less than 2^32, so no counter overflows, and every partial and total is an integer below 2^53:
// the fp64 atomic sums are exact whatever their order.  The result is therefore bitwise the same on every run and equals
// what spb_pair_tables_weighted / spb_pair_tables_wide give for the values (double) counts[r][p].
#include "common.cuh"

using namespace spb;

namespace {

constexpr int kRThreads = 256;
constexpr int kRCombos = 4;                       // (row, pair) combinations per thread
constexpr int kRTile = kRThreads * kRCombos;      // combinations per CTA
constexpr int64_t kRChunkMin = 1024;              // patterns per chunk at least
constexpr int kRStageMax = 256;                   // patterns staged in shared memory at once
constexpr size_t kRCountStageBytes = 32 << 10;    // shared memory of the staged count rows at most (above the 32-pattern floor)

__global__ void __launch_bounds__(kRThreads, 2) pair_rows_kernel(const unsigned long long* __restrict__ keys, int key_words,
                                                                const uint32_t* __restrict__ counts, int64_t R, int64_t P,
                                                                int n, int stage, int64_t chunk, double* __restrict__ N) {
  extern __shared__ __align__(16) uint32_t s_mem[];
  uint32_t* s_acc = s_mem;                                                            // [kRCombos][16][kRThreads]
  unsigned long long* s_key = reinterpret_cast<unsigned long long*>(s_acc + kRCombos * 16 * kRThreads);  // [stage][2]
  uint32_t* s_cnt = reinterpret_cast<uint32_t*>(s_key + 2 * stage);                   // [rows the tile spans][stage]
  const int tid = threadIdx.x;
  const int npairs = n * (n + 1) / 2;
  const int64_t total = R * npairs;
  const int64_t c0 = (int64_t)blockIdx.x * kRTile;
  const int64_t r0 = c0 / npairs;
  const int64_t c_last = (c0 + kRTile < total ? c0 + kRTile : total) - 1;
  const int nrows = (int)(c_last / npairs - r0 + 1);
  int rl[kRCombos], si[kRCombos], sj[kRCombos];  // row within the tile (-1: past the end), digit shifts of i and j
#pragma unroll
  for (int k = 0; k < kRCombos; ++k) {
    const int64_t c = c0 + k * kRThreads + tid;
    rl[k] = -1;
    si[k] = sj[k] = 0;
    if (c < total) {
      const int64_t r = c / npairs;
      int q = (int)(c - r * npairs), i = 0;
      while (q >= n - i) { q -= n - i; ++i; }  // row i of the upper triangle (diagonal included) holds j = i .. n - 1
      rl[k] = (int)(r - r0);
      si[k] = 2 * (n - 1 - i);
      sj[k] = 2 * (n - 1 - (i + q));
    }
#pragma unroll
    for (int e = 0; e < 16; ++e) s_acc[(k * 16 + e) * kRThreads + tid] = 0u;
  }
  const int64_t p_begin = (int64_t)blockIdx.y * chunk;
  const int64_t p_end = p_begin + chunk < P ? p_begin + chunk : P;
  for (int64_t s0 = p_begin; s0 < p_end; s0 += stage) {
    const int len = (int)(p_end - s0 < stage ? p_end - s0 : stage);
    __syncthreads();
    for (int e = tid; e < len; e += kRThreads) {
      unsigned long long lo, hi = 0;
      if (key_words == 2) {
        const ulonglong2 k = __ldg(reinterpret_cast<const ulonglong2*>(keys) + s0 + e);
        lo = k.x;
        hi = k.y;
      } else {
        lo = __ldg(keys + s0 + e);
      }
      s_key[2 * e] = lo;
      s_key[2 * e + 1] = hi;
    }
    for (int e = tid; e < nrows * len; e += kRThreads) {
      const int r = e / len, p = e - r * len;
      s_cnt[r * stage + p] = __ldg(counts + (r0 + r) * P + s0 + p);
    }
    __syncthreads();
    for (int p = 0; p < len; ++p) {
      const unsigned long long lo = s_key[2 * p], hi = s_key[2 * p + 1];
#pragma unroll
      for (int k = 0; k < kRCombos; ++k) {
        if (rl[k] < 0) continue;
        const uint32_t v = s_cnt[rl[k] * stage + p];
        if (v == 0u) continue;
        const int x = (int)(((si[k] < 64 ? lo : hi) >> (si[k] & 63)) & 3ull);
        const int y = (int)(((sj[k] < 64 ? lo : hi) >> (sj[k] & 63)) & 3ull);
        s_acc[(k * 16 + x * 4 + y) * kRThreads + tid] += v;
      }
    }
  }
  // flush: the thread reads only its own counters, so no barrier is needed
#pragma unroll
  for (int k = 0; k < kRCombos; ++k) {
    if (rl[k] < 0) continue;
    const int64_t r = r0 + rl[k];
    const int i = n - 1 - si[k] / 2, j = n - 1 - sj[k] / 2;
    double* Nij = N + ((r * n + i) * n + j) * 16;
    double* Nji = N + ((r * n + j) * n + i) * 16;
#pragma unroll
    for (int e = 0; e < 16; ++e) {
      const uint32_t v = s_acc[(k * 16 + e) * kRThreads + tid];
      if (v == 0u) continue;
      atomicAdd(Nij + e, (double)v);
      if (i != j) atomicAdd(Nji + (e & 3) * 4 + (e >> 2), (double)v);
    }
  }
}

}  // namespace

extern "C" int spb_pair_tables_count_rows(const uint64_t* d_keys, const uint32_t* d_counts, int64_t rows, int64_t num, int n_taxa,
                                          double* d_N, void* stream) {
  SPB_REQUIRE(n_taxa >= 2 && n_taxa <= SPB_MAX_TAXA, "spb_pair_tables_count_rows: n_taxa must be 2..%d (got %d)", SPB_MAX_TAXA, n_taxa);
  SPB_REQUIRE(rows >= 0 && num >= 0 && num <= INT64_MAX / (rows > 0 ? rows : 1), "spb_pair_tables_count_rows: bad sizes (rows=%lld, num=%lld)",
              (long long)rows, (long long)num);
  if (rows == 0) return SPB_OK;
  SPB_REQUIRE(d_N, "spb_pair_tables_count_rows: NULL buffer");
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t cells = rows * n_taxa * n_taxa * 16;
  SPB_CUDA(cudaMemsetAsync(d_N, 0, (size_t)cells * sizeof(double), st));
  if (num == 0) return SPB_OK;
  SPB_REQUIRE(d_keys && d_counts, "spb_pair_tables_count_rows: NULL buffer");
  const int key_words = n_taxa > 31 ? 2 : 1;
  SPB_REQUIRE(key_words == 1 || (reinterpret_cast<uintptr_t>(d_keys) & 15) == 0,
              "spb_pair_tables_count_rows: the 128-bit key array must be 16-byte aligned");
  const int npairs = n_taxa * (n_taxa + 1) / 2;
  const int64_t tiles = (rows * npairs + kRTile - 1) / kRTile;
  const int64_t span = (kRTile + npairs - 1) / npairs + 1;  // rows a tile of consecutive combinations touches at most
  const int rows_span = (int)(span < rows ? span : rows);
  int stage = kRStageMax;
  while (stage > 32 && (size_t)rows_span * stage * 4 > kRCountStageBytes) stage >>= 1;
  const size_t smem = (size_t)kRCombos * 16 * kRThreads * 4 + (size_t)stage * 16 + (size_t)rows_span * stage * 4;
  // chunks: enough CTAs for two per SM, but no chunk under kRChunkMin patterns (each chunk costs a flush of its counters)
  int64_t chunks = (2 * (int64_t)sm_count() + tiles - 1) / tiles;
  const int64_t most = (num + kRChunkMin - 1) / kRChunkMin;
  if (chunks > most) chunks = most;
  if (chunks < 1) chunks = 1;
  const int64_t chunk = (num + chunks - 1) / chunks;
  chunks = (num + chunk - 1) / chunk;
  SPB_REQUIRE(tiles <= 0x7FFFFFFF, "spb_pair_tables_count_rows: too many rows (%lld)", (long long)rows);
  SPB_CUDA(cudaFuncSetAttribute(pair_rows_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  pair_rows_kernel<<<dim3((unsigned)tiles, (unsigned)chunks), kRThreads, smem, st>>>((const unsigned long long*)d_keys, key_words,
                                                                                    d_counts, rows, num, n_taxa, stage, chunk, d_N);
  SPB_LAUNCH_CHECK();
  return SPB_OK;
}

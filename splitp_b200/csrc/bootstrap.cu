// Nonparametric bootstrap of a pattern table: replicate b is a multinomial draw of the N usable sites over the P patterns
// (sites with the same pattern are exchangeable, so drawing sites and drawing patterns with probability count / N is the
// same thing).  Draw s of replicate b, with the table in its sorted key order:
//   u = fmix(seed + gamma (b 2^40 + s + 1))     SplitMix64 output (the plain SplitMix64 sequence from `seed` when b = 0)
//   j = floor(u N / 2^64)                       high word of the 128-bit product
//   p : prefix[p] <= j < prefix[p + 1]          prefix = exclusive cumulative counts
// Every draw is a function of (seed, b, s) alone, so a replicate does not depend on which launch produced it.
//
//   bootstrap_counts_kernel   grid (draw blocks, replicates).  The block first copies every (16 << shift)-th prefix entry into
//                             shared memory (shift = 0 while that index fits kCoarseMax entries: 15 KB for the 60,203 patterns
//                             of 12 taxa x 10^6 sites), searches it, narrows a wider stride by binary search over 64-byte
//                             lines of the prefix and finishes inside one line.  Equal patterns of a warp's 32 draws are
//                             added by one integer atomic (__match_any_sync): constant sites hold a large share of the draws
//                             and same-address atomics serialise in one L2 slice.  Integer sums make the counts exact.
//   compaction                three passes over tiles of kTile patterns: non-zeros per (replicate, tile); one exclusive scan
//                             of all of them in (replicate, tile) order; ordered write of keys (or pattern indices), counts
//                             and replicate offsets.
#include "common.cuh"

namespace spb {
namespace {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr int kLine = 16;            // uint32 prefix entries per 64-byte line
constexpr int64_t kCoarseMax = 8192;  // shared coarse index: at most 32 KB
constexpr int kDrawsPerThread = 64;   // draws per thread: amortises the block's copy of the coarse index
constexpr int kTile = 4 * kThreads;   // patterns per compaction tile
constexpr int kScanThreads = 1024;
constexpr uint64_t kGamma = 0x9E3779B97F4A7C15ull;

__device__ __forceinline__ uint64_t fmix(uint64_t z) {
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}

int coarse_shift(int64_t P) {
  int shift = 0;
  while ((P + ((int64_t)kLine << shift) - 1) / ((int64_t)kLine << shift) > kCoarseMax) ++shift;
  return shift;
}

// number of prefix entries of line `line` (entries [kLine line, min(kLine line + kLine, P))) that are <= j
__device__ __forceinline__ int line_rank(const uint32_t* __restrict__ prefix, int64_t P, int64_t line, uint32_t j) {
  const int64_t q0 = line * kLine;
  int r = 0;
  if (q0 + kLine <= P) {
    const uint4* v = reinterpret_cast<const uint4*>(prefix + q0);
#pragma unroll
    for (int w = 0; w < kLine / 4; ++w) {
      const uint4 x = __ldg(v + w);
      r += (x.x <= j) + (x.y <= j) + (x.z <= j) + (x.w <= j);
    }
  } else {
    for (int64_t q = q0; q < P; ++q) r += __ldg(prefix + q) <= j;
  }
  return r;
}

__global__ void __launch_bounds__(kThreads) bootstrap_counts_kernel(const uint32_t* __restrict__ prefix, int64_t P, uint64_t N,
                                                                    uint64_t seed, int64_t rep_first, int shift, int64_t ncoarse,
                                                                    uint32_t* __restrict__ out) {
  extern __shared__ uint32_t coarse[];  // coarse[i] = prefix[(kLine << shift) i]
  const int64_t stride = (int64_t)kLine << shift;
  for (int64_t i = threadIdx.x; i < ncoarse; i += kThreads) coarse[i] = __ldg(prefix + i * stride);
  __syncthreads();
  const uint64_t rep = (uint64_t)(rep_first + blockIdx.y);
  uint32_t* cnt = out + (int64_t)blockIdx.y * P;
  const uint64_t base = seed + kGamma * (rep << 40);  // mod 2^64: u = fmix(base + gamma (s + 1))
  const int lane = threadIdx.x & 31;
  const uint64_t step = (uint64_t)gridDim.x * kThreads;
  // s0 is the same for the 32 lanes, so every lane runs every iteration and the warp votes stay full
  for (uint64_t s0 = ((uint64_t)blockIdx.x * kWarps + (threadIdx.x >> 5)) * 32; s0 < N; s0 += step) {
    const uint64_t s = s0 + lane;
    const bool valid = s < N;
    uint32_t p = 0xFFFFFFFFu;
    if (valid) {
      const uint32_t j = (uint32_t)__umul64hi(fmix(base + kGamma * (s + 1)), N);
      int64_t lo = 0, hi = ncoarse;  // largest i with coarse[i] <= j (coarse[0] = 0)
      while (hi - lo > 1) {
        const int64_t mid = (lo + hi) >> 1;
        if (coarse[mid] <= j) lo = mid; else hi = mid;
      }
      int64_t l0 = lo << shift;  // lines [l0, l1) hold the answer; the first entry of line l0 is <= j
      int64_t l1 = l0 + ((int64_t)1 << shift);
      const int64_t lines = (P + kLine - 1) / kLine;
      if (l1 > lines) l1 = lines;
      while (l1 - l0 > 1) {
        const int64_t mid = (l0 + l1) >> 1;
        if (__ldg(prefix + mid * kLine) <= j) l0 = mid; else l1 = mid;
      }
      p = (uint32_t)(l0 * kLine + line_rank(prefix, P, l0, j) - 1);
    }
    const unsigned peers = __match_any_sync(0xFFFFFFFFu, p);
    if (valid && lane == __ffs(peers) - 1) atomicAdd(cnt + p, (uint32_t)__popc(peers));
  }
}

__global__ void __launch_bounds__(kThreads) compact_count_kernel(const uint32_t* __restrict__ counts, int64_t P, int64_t* __restrict__ tile_nnz) {
  __shared__ int sh[kWarps];
  const int64_t q0 = (int64_t)blockIdx.x * kTile;
  const uint32_t* c = counts + (int64_t)blockIdx.y * P;
  int k = 0;
  for (int i = threadIdx.x; i < kTile; i += kThreads) k += (q0 + i < P && c[q0 + i] != 0u);
  for (int o = 16; o; o >>= 1) k += __shfl_down_sync(0xFFFFFFFFu, k, o);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = k;
  __syncthreads();
  if (threadIdx.x == 0) {
    int t = 0;
    for (int w = 0; w < kWarps; ++w) t += sh[w];
    tile_nnz[(int64_t)blockIdx.y * gridDim.x + blockIdx.x] = t;
  }
}

// exclusive scan of m values in place (one block; every thread scans a contiguous run); offsets[r] = first value of
// replicate r's tiles, offsets[reps] = total
__global__ void __launch_bounds__(kScanThreads) compact_scan_kernel(int64_t* __restrict__ v, int64_t m, int64_t tiles, int64_t reps,
                                                                    int64_t* __restrict__ offsets) {
  __shared__ int64_t sh[kScanThreads / 32];
  const int64_t run = (m + kScanThreads - 1) / kScanThreads;
  const int64_t b = threadIdx.x * run, e = b + run < m ? b + run : m;
  int64_t own = 0;
  for (int64_t i = b; i < e; ++i) own += v[i];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  int64_t x = own;  // inclusive warp scan
  for (int o = 1; o < 32; o <<= 1) {
    const int64_t y = __shfl_up_sync(0xFFFFFFFFu, x, o);
    if (lane >= o) x += y;
  }
  if (lane == 31) sh[w] = x;
  __syncthreads();
  if (w == 0) {
    int64_t t = lane < kScanThreads / 32 ? sh[lane] : 0;
    for (int o = 1; o < 32; o <<= 1) {
      const int64_t y = __shfl_up_sync(0xFFFFFFFFu, t, o);
      if (lane >= o) t += y;
    }
    if (lane < kScanThreads / 32) sh[lane] = t;
  }
  __syncthreads();
  int64_t acc = x - own + (w ? sh[w - 1] : 0);
  for (int64_t i = b; i < e; ++i) {
    const int64_t t = v[i];
    v[i] = acc;
    acc += t;
  }
  __syncthreads();
  for (int64_t r = threadIdx.x; r < reps; r += kScanThreads) offsets[r] = v[r * tiles];
  if (threadIdx.x == kScanThreads - 1) offsets[reps] = acc;
}

template <int W>
__global__ void __launch_bounds__(kThreads) compact_write_kernel(const uint32_t* __restrict__ counts, const uint64_t* __restrict__ keys,
                                                                 int64_t P, const int64_t* __restrict__ tile_off, int64_t cap,
                                                                 uint64_t* __restrict__ out_keys, uint32_t* __restrict__ out_counts) {
  __shared__ int sh[kWarps];
  const int64_t q = (int64_t)blockIdx.x * kTile + 4 * threadIdx.x;  // four consecutive patterns per thread
  const uint32_t* c = counts + (int64_t)blockIdx.y * P;
  uint32_t v[4];
  int k = 0;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    v[i] = q + i < P ? c[q + i] : 0u;
    k += v[i] != 0u;
  }
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  int x = k;
  for (int o = 1; o < 32; o <<= 1) {
    const int y = __shfl_up_sync(0xFFFFFFFFu, x, o);
    if (lane >= o) x += y;
  }
  if (lane == 31) sh[w] = x;
  __syncthreads();
  int before = x - k;
  for (int i = 0; i < w; ++i) before += sh[i];
  int64_t pos = tile_off[(int64_t)blockIdx.y * gridDim.x + blockIdx.x] + before;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    if (v[i] != 0u && pos < cap) {
      if (W == 0) out_keys[pos] = (uint64_t)(q + i);  // the pattern's index instead of its key
#pragma unroll
      for (int t = 0; t < W; ++t) out_keys[pos * W + t] = keys[(q + i) * W + t];
      out_counts[pos] = v[i];
    }
    pos += v[i] != 0u;
  }
}

}  // namespace
}  // namespace spb

using namespace spb;

extern "C" int spb_bootstrap_counts(const uint32_t* d_prefix, int64_t P, int64_t N, uint64_t seed, int64_t rep_first, int64_t reps,
                                    uint32_t* d_counts, void* stream) {
  SPB_REQUIRE(P >= 1, "spb_bootstrap_counts: the table has no pattern (P = %lld)", (long long)P);
  SPB_REQUIRE(N >= 1 && N <= (int64_t)0xFFFFFFFFll, "spb_bootstrap_counts: N = %lld usable sites, need 1 .. 2^32 - 1", (long long)N);
  SPB_REQUIRE(rep_first >= 0 && reps >= 0 && rep_first + reps <= ((int64_t)1 << 24),
              "spb_bootstrap_counts: replicates [%lld, %lld) outside [0, 2^24)", (long long)rep_first, (long long)(rep_first + reps));
  if (reps == 0) return SPB_OK;
  SPB_REQUIRE(d_prefix && d_counts, "spb_bootstrap_counts: NULL buffer");
  SPB_REQUIRE((reinterpret_cast<uintptr_t>(d_prefix) & 15) == 0, "spb_bootstrap_counts: the prefix must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  SPB_CUDA(cudaMemsetAsync(d_counts, 0, (size_t)reps * P * sizeof(uint32_t), st));
  const int shift = coarse_shift(P);
  const int64_t ncoarse = (P + ((int64_t)kLine << shift) - 1) / ((int64_t)kLine << shift);
  const int64_t per_block = (int64_t)kThreads * kDrawsPerThread;
  const unsigned blocks = (unsigned)((N + per_block - 1) / per_block);
  for (int64_t r0 = 0; r0 < reps; r0 += 65535) {
    const unsigned ry = (unsigned)(reps - r0 < 65535 ? reps - r0 : 65535);
    bootstrap_counts_kernel<<<dim3(blocks, ry), kThreads, (size_t)ncoarse * sizeof(uint32_t), st>>>(
        d_prefix, P, (uint64_t)N, seed, rep_first + r0, shift, ncoarse, d_counts + r0 * P);
    SPB_LAUNCH_CHECK();
  }
  return SPB_OK;
}

extern "C" int64_t spb_bootstrap_compact_ws(int64_t P, int64_t reps) {
  if (P < 1 || reps < 1) return 1;
  return reps * ((P + kTile - 1) / kTile);
}

extern "C" int spb_bootstrap_compact(const uint32_t* d_counts, const uint64_t* d_keys, int key_words, int64_t P, int64_t reps,
                                     uint64_t* d_out_keys, uint32_t* d_out_counts, int64_t cap, int64_t* d_offsets, int64_t* d_ws,
                                     void* stream) {
  SPB_REQUIRE(key_words >= 0 && key_words <= 2, "spb_bootstrap_compact: key_words must be 0, 1 or 2 (got %d)", key_words);
  SPB_REQUIRE(P >= 1 && reps >= 0 && cap >= 0, "spb_bootstrap_compact: bad sizes P=%lld reps=%lld cap=%lld", (long long)P,
              (long long)reps, (long long)cap);
  SPB_REQUIRE(reps <= 65535, "spb_bootstrap_compact: at most 65535 replicates per call");
  SPB_REQUIRE(d_offsets, "spb_bootstrap_compact: NULL offsets");
  cudaStream_t st = (cudaStream_t)stream;
  if (reps == 0) {
    SPB_CUDA(cudaMemsetAsync(d_offsets, 0, sizeof(int64_t), st));
    return SPB_OK;
  }
  SPB_REQUIRE(d_counts && (d_keys || key_words == 0) && d_out_keys && d_out_counts && d_ws, "spb_bootstrap_compact: NULL buffer");
  const int64_t tiles = (P + kTile - 1) / kTile;
  SPB_REQUIRE(tiles <= 0x7FFFFFFF, "spb_bootstrap_compact: too many patterns");
  const dim3 grid((unsigned)tiles, (unsigned)reps);
  compact_count_kernel<<<grid, kThreads, 0, st>>>(d_counts, P, d_ws);
  SPB_LAUNCH_CHECK();
  compact_scan_kernel<<<1, kScanThreads, 0, st>>>(d_ws, tiles * reps, tiles, reps, d_offsets);
  SPB_LAUNCH_CHECK();
  if (key_words == 0)
    compact_write_kernel<0><<<grid, kThreads, 0, st>>>(d_counts, d_keys, P, d_ws, cap, d_out_keys, d_out_counts);
  else if (key_words == 1)
    compact_write_kernel<1><<<grid, kThreads, 0, st>>>(d_counts, d_keys, P, d_ws, cap, d_out_keys, d_out_counts);
  else
    compact_write_kernel<2><<<grid, kThreads, 0, st>>>(d_counts, d_keys, P, d_ws, cap, d_out_keys, d_out_counts);
  SPB_LAUNCH_CHECK();
  return SPB_OK;
}

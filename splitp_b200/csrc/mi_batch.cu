// Rank-1 divergence (mutual information) of MANY splits of one pattern list in one call:
//   D(split) = sum over non-zero patterns p of v_p log(v_p / (r c)),  r, c = the sums of v over the patterns that share
//   p's digits on side 0 / side 1
// (reference: splitp/phylogenetics.py:136-140 and 364-373, one split at a time; spb_table_marginals + spb_mi_table are the
// per-split form).  Every split must place every taxon on exactly one side, so every pattern is its own flattening cell.
//
// The side key of a pattern is its key with the other side's digits zeroed (key AND mask): no digit packing, and the same
// code serves uint64 and 128-bit keys.  A side that is not empty leaves zero digits in every masked key, so a masked key is
// never all ones, the EMPTY marker of the tables.
//   pass 1  mi_sums_kernel: a thread loads one pattern and inserts it into both side tables of kGroup splits (grid y =
//           split groups); counts are added as uint64 integers (exact, order independent), f64 values with fp64 atomics.
//           A table has at least twice as many slots as keys, so a probe always ends.
//   pass 2  mi_terms_kernel: block (chunk, group) looks both sums of every pattern of its chunk up and leaves one partial
//           per split; mi_total_kernel adds a split's partials in chunk order.  Chunks are a function of the pattern count
//           only, so a score's summation order does not depend on the device or on the other splits of the call.
#include "key128.cuh"

namespace spb {
namespace {

constexpr int kThreads = 256;
constexpr int kGroup = 8;               // splits per thread
constexpr int64_t kChunkMin = 2048;     // patterns per pass-2 chunk at least ...
constexpr int64_t kChunksMax = 256;     // ... and at most this many chunks per split

__host__ __device__ __forceinline__ void mi_plan(int64_t num, int64_t* chunk, int64_t* nchunks) {
  int64_t c = (num + kChunkMin - 1) / kChunkMin;
  if (c > kChunksMax) c = kChunksMax;
  if (c < 1) c = 1;
  *chunk = (num + c - 1) / c;
  if (*chunk < 1) *chunk = 1;
  *nchunks = (num + *chunk - 1) / *chunk;
  if (*nchunks < 1) *nchunks = 1;
}

// chunks of any pattern count up to num: mi_plan(m) makes at most min(ceil(m / kChunkMin), kChunksMax) chunks
int64_t mi_chunks_max(int64_t num) {
  int64_t c = (num + kChunkMin - 1) / kChunkMin;
  return c > kChunksMax ? kChunksMax : (c < 1 ? 1 : c);
}

template <int W>
struct MiKey;
template <>
struct MiKey<1> {
  unsigned long long k;
  __device__ __forceinline__ static MiKey load(const unsigned long long* keys, int64_t i) { return MiKey{__ldg(keys + i)}; }
  __device__ __forceinline__ MiKey masked(const uint64_t (&m)[2]) const { return MiKey{k & m[0]}; }
  __device__ __forceinline__ uint64_t hash() const { return mix64(k); }
};
template <>
struct MiKey<2> {
  Key128 k;
  __device__ __forceinline__ static MiKey load(const unsigned long long* keys, int64_t i) {
    const ulonglong2 v = __ldg(reinterpret_cast<const ulonglong2*>(keys) + i);
    return MiKey{Key128{v.x, v.y}};
  }
  __device__ __forceinline__ MiKey masked(const uint64_t (&m)[2]) const { return MiKey{Key128{k.lo & m[0], k.hi & m[1]}}; }
  __device__ __forceinline__ uint64_t hash() const { return hash128(k); }
};

// slot of `key` in the table of cap slots at slot `base`, inserting it if absent
__device__ __forceinline__ int64_t slot_insert(unsigned long long* tkeys, int64_t base, int64_t cap, MiKey<1> key) {
  const uint64_t m = (uint64_t)cap - 1;
  uint64_t h = key.hash() & m;
  for (uint64_t probe = 0; probe <= m; ++probe) {
    unsigned long long* p = tkeys + base + h;
    unsigned long long cur = *p;  // a stale EMPTY only sends the thread to the CAS, which reads the slot atomically
    if (cur == kAll) cur = atomicCAS(p, kAll, key.k);
    if (cur == kAll || cur == key.k) return base + (int64_t)h;
    h = (h + 1) & m;
  }
  return -1;
}

__device__ __forceinline__ int64_t slot_insert(unsigned long long* tkeys, int64_t base, int64_t cap, MiKey<2> key) {
  const uint64_t m = (uint64_t)cap - 1;
  uint64_t h = key.hash() & m;
  for (uint64_t probe = 0; probe <= m; ++probe) {
    unsigned long long* p = tkeys + 2 * (base + h);
    // A plain 16-byte read may be torn while another thread fills the slot, but a slot only ever goes from EMPTY (both
    // words all ones) to its key: a read with no all-ones word is the settled key.  Anything else takes the 128-bit CAS.
    Key128 cur = load_key(tkeys, base + h);
    if (cur.lo == kAll || cur.hi == kAll) cur = cas128(p, Key128{kAll, kAll}, key.k);
    if (is_empty(cur) || same(cur, key.k)) return base + (int64_t)h;
    h = (h + 1) & m;
  }
  return -1;
}

// slot of a key that pass 1 inserted (the tables are complete: plain reads)
__device__ __forceinline__ int64_t slot_find(const unsigned long long* tkeys, int64_t base, int64_t cap, MiKey<1> key) {
  const uint64_t m = (uint64_t)cap - 1;
  uint64_t h = key.hash() & m;
  for (uint64_t probe = 0; probe <= m; ++probe) {
    const unsigned long long cur = tkeys[base + h];
    if (cur == key.k) return base + (int64_t)h;
    if (cur == kAll) break;
    h = (h + 1) & m;
  }
  return -1;
}

__device__ __forceinline__ int64_t slot_find(const unsigned long long* tkeys, int64_t base, int64_t cap, MiKey<2> key) {
  const uint64_t m = (uint64_t)cap - 1;
  uint64_t h = key.hash() & m;
  for (uint64_t probe = 0; probe <= m; ++probe) {
    const Key128 cur = load_key(tkeys, base + h);
    if (same(cur, key.k)) return base + (int64_t)h;
    if (is_empty(cur)) break;
    h = (h + 1) & m;
  }
  return -1;
}

template <bool COUNTS>
__device__ __forceinline__ double raw_at(const void* vals, int64_t i) {
  return COUNTS ? (double)__ldg((const uint32_t*)vals + i) : __ldg((const double*)vals + i);
}

template <int W, bool COUNTS>
__global__ void __launch_bounds__(kThreads) mi_sums_kernel(const unsigned long long* __restrict__ keys, const void* __restrict__ vals,
                                                           int64_t num, const spb_mi_split* __restrict__ splits, int64_t n_splits,
                                                           unsigned long long* tkeys, unsigned long long* sums) {
  const int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x;
  if (i >= num) return;
  const double raw = raw_at<COUNTS>(vals, i);
  if (raw == 0.0) return;
  const MiKey<W> key = MiKey<W>::load(keys, i);
  const int64_t s0 = (int64_t)blockIdx.y * kGroup;
  const int ng = (int)(n_splits - s0 < kGroup ? n_splits - s0 : kGroup);
  for (int g = 0; g < ng; ++g) {
    const spb_mi_split& sp = splits[s0 + g];
#pragma unroll
    for (int side = 0; side < 2; ++side) {
      const int64_t slot = slot_insert(tkeys, sp.slot[side], sp.cap[side], key.masked(sp.mask[side]));
      if (slot < 0) continue;  // unreachable with cap >= 2 x keys
      if (COUNTS) atomicAdd(sums + slot, (unsigned long long)raw);
      else atomicAdd(reinterpret_cast<double*>(sums) + slot, raw);
    }
  }
}

// fixed-order tree: the result depends on the inputs only, not on scheduling
__device__ __forceinline__ double block_sum(double v, double* sh) {
  for (int o = 16; o; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  __syncthreads();
  if (l == 0) sh[w] = v;
  __syncthreads();
  if (w == 0) {
    v = l < (int)(blockDim.x >> 5) ? sh[l] : 0.0;
    for (int o = 16; o; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  }
  return v;  // valid in thread 0
}

// counts -> probabilities (fasta.py:66-70), as spb_mi_table
__device__ __forceinline__ double mi_value(double raw, double divisor) { return divisor > 0.0 ? raw / divisor : raw; }

// acc + the pattern's term v log(v / (r c)), from its value v and the raw sums c / r of its side-0 / side-1 key.  Every
// kernel of this file adds its terms through here, so they round alike.
__device__ __forceinline__ double mi_add_term(double acc, double v, double c, double r, double divisor) {
  if (divisor > 0.0) { c /= divisor; r /= divisor; }
  return acc + v * log(v / (r * c));
}

template <bool COUNTS>
__device__ __forceinline__ double side_sum(const unsigned long long* sums, int64_t slot) {
  if (slot < 0) return 0.0;
  return COUNTS ? (double)sums[slot] : __longlong_as_double((long long)sums[slot]);
}

template <int W, bool COUNTS>
__global__ void __launch_bounds__(kThreads) mi_terms_kernel(const unsigned long long* __restrict__ keys, const void* __restrict__ vals,
                                                            int64_t num, double divisor, const spb_mi_split* __restrict__ splits,
                                                            int64_t n_splits, const unsigned long long* __restrict__ tkeys,
                                                            const unsigned long long* __restrict__ sums, int64_t chunk,
                                                            double* __restrict__ partials) {
  __shared__ spb_mi_split sp[kGroup];
  __shared__ double sh[kThreads / 32];
  const int64_t s0 = (int64_t)blockIdx.y * kGroup;
  const int ng = (int)(n_splits - s0 < kGroup ? n_splits - s0 : kGroup);
  if (threadIdx.x < ng) sp[threadIdx.x] = splits[s0 + threadIdx.x];
  __syncthreads();
  double acc[kGroup];
#pragma unroll
  for (int g = 0; g < kGroup; ++g) acc[g] = 0.0;
  const int64_t begin = (int64_t)blockIdx.x * chunk;
  const int64_t end = begin + chunk < num ? begin + chunk : num;
  for (int64_t i = begin + threadIdx.x; i < end; i += kThreads) {
    const double raw = raw_at<COUNTS>(vals, i);
    if (raw == 0.0) continue;
    const MiKey<W> key = MiKey<W>::load(keys, i);
    const double v = mi_value(raw, divisor);
#pragma unroll
    for (int g = 0; g < kGroup; ++g) {
      if (g < ng) {
        const double c = side_sum<COUNTS>(sums, slot_find(tkeys, sp[g].slot[0], sp[g].cap[0], key.masked(sp[g].mask[0])));
        const double r = side_sum<COUNTS>(sums, slot_find(tkeys, sp[g].slot[1], sp[g].cap[1], key.masked(sp[g].mask[1])));
        acc[g] = mi_add_term(acc[g], v, c, r, divisor);
      }
    }
  }
#pragma unroll
  for (int g = 0; g < kGroup; ++g) {
    const double t = block_sum(acc[g], sh);
    if (threadIdx.x == 0 && g < ng) partials[(s0 + g) * (int64_t)gridDim.x + blockIdx.x] = t;
  }
}

// a score from its chunk partials, in chunk order
__device__ __forceinline__ double chunk_total(const double* partials, int64_t nchunks) {
  double acc = 0.0;
  for (int64_t q = 0; q < nchunks; ++q) acc += partials[q];
  return acc;
}

__global__ void mi_total_kernel(const double* __restrict__ partials, int64_t nchunks, int64_t n_splits, double* __restrict__ out) {
  const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_splits) return;
  out[s] = chunk_total(partials + s * nchunks, nchunks);
}

template <int W, bool COUNTS>
int launch(const uint64_t* d_keys, const void* d_vals, int64_t num, double divisor, const spb_mi_split* d_splits, int64_t n_splits,
           int64_t slots, uint64_t* d_ws, double* d_out, cudaStream_t st) {
  int64_t chunk, nchunks;
  mi_plan(num, &chunk, &nchunks);
  unsigned long long* tkeys = (unsigned long long*)d_ws;
  unsigned long long* sums = tkeys + slots * W;
  double* partials = reinterpret_cast<double*>(sums + slots);
  SPB_CUDA(cudaMemsetAsync(tkeys, 0xFF, (size_t)slots * W * sizeof(uint64_t), st));
  SPB_CUDA(cudaMemsetAsync(sums, 0, (size_t)slots * sizeof(uint64_t), st));
  const unsigned groups = (unsigned)((n_splits + kGroup - 1) / kGroup);
  const unsigned long long* k = (const unsigned long long*)d_keys;
  mi_sums_kernel<W, COUNTS><<<dim3((unsigned)((num + kThreads - 1) / kThreads), groups), kThreads, 0, st>>>(k, d_vals, num, d_splits,
                                                                                                          n_splits, tkeys, sums);
  SPB_LAUNCH_CHECK();
  mi_terms_kernel<W, COUNTS><<<dim3((unsigned)nchunks, groups), kThreads, 0, st>>>(k, d_vals, num, divisor, d_splits, n_splits, tkeys,
                                                                                   sums, chunk, partials);
  SPB_LAUNCH_CHECK();
  mi_total_kernel<<<(unsigned)((n_splits + kThreads - 1) / kThreads), kThreads, 0, st>>>(partials, nchunks, n_splits, d_out);
  SPB_LAUNCH_CHECK();
  return SPB_OK;
}

// ---- count rows over one pattern list ----
// slot pass: inserts every key into both side tables of every split and records its slot in each, relative to the side's
// first slot: slot_of[(s 2 + side) num + p].  The layout depends on the keys only, so every count row over them shares it.
template <int W>
__global__ void __launch_bounds__(kThreads) mi_slots_kernel(const unsigned long long* __restrict__ keys, int64_t num,
                                                            const spb_mi_split* __restrict__ splits, int64_t n_splits,
                                                            unsigned long long* tkeys, uint32_t* __restrict__ slot_of) {
  const int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x;
  if (i >= num) return;
  const MiKey<W> key = MiKey<W>::load(keys, i);
  const int64_t s0 = (int64_t)blockIdx.y * kGroup;
  const int ng = (int)(n_splits - s0 < kGroup ? n_splits - s0 : kGroup);
  for (int g = 0; g < ng; ++g) {
    const spb_mi_split& sp = splits[s0 + g];
#pragma unroll
    for (int side = 0; side < 2; ++side) {
      const int64_t slot = slot_insert(tkeys, sp.slot[side], sp.cap[side], key.masked(sp.mask[side]));
      slot_of[((s0 + g) * 2 + side) * num + i] = (uint32_t)(slot - sp.slot[side]);  // slot >= 0 with cap >= 2 x keys
    }
  }
}

// row pass 1: block (patterns, split group, row) adds the row's counts into the row's side sums at the recorded slots
__global__ void __launch_bounds__(kThreads) mi_row_sums_kernel(const uint32_t* __restrict__ counts, int64_t num,
                                                               const spb_mi_split* __restrict__ splits, int64_t n_splits,
                                                               int64_t slots, const uint32_t* __restrict__ slot_of,
                                                               unsigned long long* __restrict__ sums) {
  const int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x;
  if (i >= num) return;
  const uint32_t c = __ldg(counts + (int64_t)blockIdx.z * num + i);
  if (c == 0u) return;
  unsigned long long* rs = sums + (int64_t)blockIdx.z * slots;
  const int64_t s0 = (int64_t)blockIdx.y * kGroup;
  const int ng = (int)(n_splits - s0 < kGroup ? n_splits - s0 : kGroup);
  for (int g = 0; g < ng; ++g) {
    const spb_mi_split& sp = splits[s0 + g];
#pragma unroll
    for (int side = 0; side < 2; ++side)
      atomicAdd(rs + sp.slot[side] + __ldg(slot_of + ((s0 + g) * 2 + side) * num + i), (unsigned long long)c);
  }
}

// row pass 2: mi_terms_kernel over the row's non-zero patterns (index[offsets[r] ..]) in table order, chunked by
// mi_plan(non-zeros): block (chunk, group, row) leaves one partial per split, at partials[(r n_splits + s) cmax + chunk]
__global__ void __launch_bounds__(kThreads) mi_row_terms_kernel(const uint32_t* __restrict__ counts, int64_t num,
                                                                const unsigned long long* __restrict__ index,
                                                                const int64_t* __restrict__ offsets, double divisor,
                                                                const spb_mi_split* __restrict__ splits, int64_t n_splits,
                                                                int64_t slots, const uint32_t* __restrict__ slot_of,
                                                                const unsigned long long* __restrict__ sums, int64_t cmax,
                                                                double* __restrict__ partials) {
  __shared__ spb_mi_split sp[kGroup];
  __shared__ double sh[kThreads / 32];
  const int64_t r = blockIdx.z;
  const int64_t o0 = offsets[r], nnz = offsets[r + 1] - o0;
  int64_t chunk, nchunks;
  mi_plan(nnz, &chunk, &nchunks);
  if ((int64_t)blockIdx.x >= nchunks) return;  // the whole block
  const int64_t s0 = (int64_t)blockIdx.y * kGroup;
  const int ng = (int)(n_splits - s0 < kGroup ? n_splits - s0 : kGroup);
  if (threadIdx.x < ng) sp[threadIdx.x] = splits[s0 + threadIdx.x];
  __syncthreads();
  const uint32_t* row = counts + r * num;
  const unsigned long long* rs = sums + r * slots;
  double acc[kGroup];
#pragma unroll
  for (int g = 0; g < kGroup; ++g) acc[g] = 0.0;
  const int64_t begin = (int64_t)blockIdx.x * chunk;
  const int64_t end = begin + chunk < nnz ? begin + chunk : nnz;
  for (int64_t i = begin + threadIdx.x; i < end; i += kThreads) {
    const int64_t p = (int64_t)__ldg(index + o0 + i);
    const double raw = (double)__ldg(row + p);
    if (raw == 0.0) continue;
    const double v = mi_value(raw, divisor);
#pragma unroll
    for (int g = 0; g < kGroup; ++g) {
      if (g < ng) {
        const uint32_t* so = slot_of + (s0 + g) * 2 * num + p;
        const double c = (double)rs[sp[g].slot[0] + __ldg(so)];
        const double rr = (double)rs[sp[g].slot[1] + __ldg(so + num)];
        acc[g] = mi_add_term(acc[g], v, c, rr, divisor);
      }
    }
  }
#pragma unroll
  for (int g = 0; g < kGroup; ++g) {
    const double t = block_sum(acc[g], sh);
    if (threadIdx.x == 0 && g < ng) partials[(r * n_splits + s0 + g) * cmax + blockIdx.x] = t;
  }
}

__global__ void mi_row_total_kernel(const double* __restrict__ partials, const int64_t* __restrict__ offsets, int64_t rows,
                                    int64_t n_splits, int64_t cmax, double* __restrict__ out) {
  const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= rows * n_splits) return;
  const int64_t r = j / n_splits;
  int64_t chunk, nchunks;
  mi_plan(offsets[r + 1] - offsets[r], &chunk, &nchunks);
  out[j] = chunk_total(partials + j * cmax, nchunks);
}

}  // namespace
}  // namespace spb

using namespace spb;

extern "C" int64_t spb_mi_side_cap(int64_t num, int side_len) {
  int64_t distinct = num < 1 ? 1 : num;
  if (side_len >= 0 && side_len < 31 && (1ll << (2 * side_len)) < distinct) distinct = 1ll << (2 * side_len);
  int64_t cap = 2;
  while (cap < 2 * distinct) cap *= 2;
  return cap;
}

extern "C" int64_t spb_mi_scores_ws(int64_t num, int key_words, int64_t slots, int64_t n_splits) {
  if (num < 0 || slots < 0 || n_splits < 0 || (key_words != 1 && key_words != 2)) return 0;
  int64_t chunk, nchunks;
  mi_plan(num, &chunk, &nchunks);
  return slots * (key_words + 1) + n_splits * nchunks;
}

extern "C" int spb_mi_scores(const uint64_t* d_keys, int key_words, const void* d_vals, int val_kind, double divisor, int64_t num,
                             const spb_mi_split* d_splits, int64_t n_splits, int64_t slots, uint64_t* d_ws, double* d_out,
                             void* stream) {
  SPB_REQUIRE(key_words == 1 || key_words == 2, "spb_mi_scores: key_words must be 1 or 2 (got %d)", key_words);
  SPB_REQUIRE(val_kind == SPB_VAL_U32 || val_kind == SPB_VAL_F64, "spb_mi_scores: bad value kind");
  SPB_REQUIRE(num >= 0 && n_splits >= 0 && slots >= 0, "spb_mi_scores: negative size");
  SPB_REQUIRE(n_splits <= (int64_t)65535 * kGroup, "spb_mi_scores: at most %lld splits per call", (long long)65535 * kGroup);
  if (n_splits == 0) return SPB_OK;
  SPB_REQUIRE(d_out, "spb_mi_scores: NULL output");
  cudaStream_t st = (cudaStream_t)stream;
  if (num == 0) {
    SPB_CUDA(cudaMemsetAsync(d_out, 0, (size_t)n_splits * sizeof(double), st));
    return SPB_OK;
  }
  SPB_REQUIRE(d_keys && d_vals && d_splits && d_ws && slots > 0, "spb_mi_scores: NULL buffer");
  SPB_REQUIRE(key_words == 1 || (reinterpret_cast<uintptr_t>(d_keys) & 15) == 0, "spb_mi_scores: 128-bit keys must be 16-byte aligned");
  SPB_REQUIRE((reinterpret_cast<uintptr_t>(d_ws) & 15) == 0, "spb_mi_scores: the workspace must be 16-byte aligned");
  const bool counts = val_kind == SPB_VAL_U32;
  if (key_words == 1)
    return counts ? launch<1, true>(d_keys, d_vals, num, divisor, d_splits, n_splits, slots, d_ws, d_out, st)
                  : launch<1, false>(d_keys, d_vals, num, divisor, d_splits, n_splits, slots, d_ws, d_out, st);
  return counts ? launch<2, true>(d_keys, d_vals, num, divisor, d_splits, n_splits, slots, d_ws, d_out, st)
                : launch<2, false>(d_keys, d_vals, num, divisor, d_splits, n_splits, slots, d_ws, d_out, st);
}

extern "C" int spb_mi_row_slots(const uint64_t* d_keys, int key_words, int64_t num, const spb_mi_split* d_splits, int64_t n_splits,
                                int64_t slots, uint64_t* d_tkeys, uint32_t* d_slot_of, void* stream) {
  SPB_REQUIRE(key_words == 1 || key_words == 2, "spb_mi_row_slots: key_words must be 1 or 2 (got %d)", key_words);
  SPB_REQUIRE(num >= 0 && n_splits >= 0 && slots >= 0, "spb_mi_row_slots: negative size");
  SPB_REQUIRE(n_splits <= (int64_t)65535 * kGroup, "spb_mi_row_slots: at most %lld splits per call", (long long)65535 * kGroup);
  if (num == 0 || n_splits == 0) return SPB_OK;
  SPB_REQUIRE(d_keys && d_splits && d_tkeys && d_slot_of && slots > 0, "spb_mi_row_slots: NULL buffer");
  SPB_REQUIRE(key_words == 1 || (reinterpret_cast<uintptr_t>(d_keys) & 15) == 0, "spb_mi_row_slots: 128-bit keys must be 16-byte aligned");
  SPB_REQUIRE((reinterpret_cast<uintptr_t>(d_tkeys) & 15) == 0, "spb_mi_row_slots: the side tables must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  SPB_CUDA(cudaMemsetAsync(d_tkeys, 0xFF, (size_t)slots * key_words * sizeof(uint64_t), st));
  const dim3 grid((unsigned)((num + kThreads - 1) / kThreads), (unsigned)((n_splits + kGroup - 1) / kGroup));
  const unsigned long long* k = (const unsigned long long*)d_keys;
  unsigned long long* t = (unsigned long long*)d_tkeys;
  if (key_words == 1) mi_slots_kernel<1><<<grid, kThreads, 0, st>>>(k, num, d_splits, n_splits, t, d_slot_of);
  else mi_slots_kernel<2><<<grid, kThreads, 0, st>>>(k, num, d_splits, n_splits, t, d_slot_of);
  SPB_LAUNCH_CHECK();
  return SPB_OK;
}

extern "C" int64_t spb_mi_rows_ws(int64_t num, int64_t rows, int64_t slots, int64_t n_splits) {
  if (num < 0 || rows < 0 || slots < 0 || n_splits < 0) return 0;
  return rows * (slots + n_splits * mi_chunks_max(num));
}

extern "C" int spb_mi_row_scores(const uint32_t* d_counts, int64_t num, const uint64_t* d_index, const int64_t* d_offsets, int64_t rows,
                                 double divisor, const spb_mi_split* d_splits, int64_t n_splits, int64_t slots,
                                 const uint32_t* d_slot_of, uint64_t* d_ws, double* d_out, void* stream) {
  SPB_REQUIRE(num >= 0 && rows >= 0 && n_splits >= 0 && slots >= 0, "spb_mi_row_scores: negative size");
  SPB_REQUIRE(n_splits <= (int64_t)65535 * kGroup, "spb_mi_row_scores: at most %lld splits per call", (long long)65535 * kGroup);
  SPB_REQUIRE(rows <= 65535, "spb_mi_row_scores: at most 65535 rows per call");
  if (n_splits == 0 || rows == 0) return SPB_OK;
  SPB_REQUIRE(d_out, "spb_mi_row_scores: NULL output");
  cudaStream_t st = (cudaStream_t)stream;
  if (num == 0) {
    SPB_CUDA(cudaMemsetAsync(d_out, 0, (size_t)rows * n_splits * sizeof(double), st));
    return SPB_OK;
  }
  SPB_REQUIRE(d_counts && d_index && d_offsets && d_splits && d_slot_of && d_ws && slots > 0, "spb_mi_row_scores: NULL buffer");
  const int64_t cmax = mi_chunks_max(num);
  unsigned long long* sums = (unsigned long long*)d_ws;
  double* partials = reinterpret_cast<double*>(sums + rows * slots);
  SPB_CUDA(cudaMemsetAsync(sums, 0, (size_t)rows * slots * sizeof(uint64_t), st));
  const unsigned groups = (unsigned)((n_splits + kGroup - 1) / kGroup);
  mi_row_sums_kernel<<<dim3((unsigned)((num + kThreads - 1) / kThreads), groups, (unsigned)rows), kThreads, 0, st>>>(
      d_counts, num, d_splits, n_splits, slots, d_slot_of, sums);
  SPB_LAUNCH_CHECK();
  mi_row_terms_kernel<<<dim3((unsigned)cmax, groups, (unsigned)rows), kThreads, 0, st>>>(
      d_counts, num, (const unsigned long long*)d_index, d_offsets, divisor, d_splits, n_splits, slots, d_slot_of, sums, cmax, partials);
  SPB_LAUNCH_CHECK();
  mi_row_total_kernel<<<(unsigned)((rows * n_splits + kThreads - 1) / kThreads), kThreads, 0, st>>>(partials, d_offsets, rows, n_splits,
                                                                                                    cmax, d_out);
  SPB_LAUNCH_CHECK();
  return SPB_OK;
}

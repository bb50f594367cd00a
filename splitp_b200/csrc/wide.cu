// Wide pattern keys (up to 64 taxa): BASELINE config 4 (64-taxon alignment, pattern compression + thin reduced
// flattenings).  A pattern key is the 128-bit base-4 number of the site pattern, taxon 0 most significant (the
// significance of `__index_of`, splitp/constructions.py:166-171), stored as two uint64 words {lo, hi}.
//
//   spb_pack_wide        chars -> one 128-bit key per site (16 bytes per site = N*n/4 bytes at 64 taxa) + validity
//                        mask (splitp/parsers/fasta.py:54-57)
//   spb_count_hash_wide  pattern compression (fasta.py:48-63) into an open-addressing table with 128-bit keys
//                        (atom.cas.b128); the lanes of a warp that carry the key of its first usable lane are
//                        aggregated with one ballot.  The all-ones key (the all-T pattern at exactly 64 taxa) doubles
//                        as the EMPTY marker, so it is counted in a separate cell (d_special)
//   spb_compact_hash_wide / spb_hash_merge_wide   table -> (key, count) list and back (multi-GPU merge)
//   spb_thin_gram_wide   exact Gram F F^T of the REDUCED flattening (constructions.py:31-55) of a split whose side A
//                        has 1 or 2 taxa, straight from the hashed table: rows = the 4^a row patterns, columns = the
//                        distinct patterns of the other taxa; G[r1][r2] = sum over patterns p with row part r1 of
//                        count(p) * count(p with its row part replaced by r2) -- one hash lookup per (p, r2), no
//                        sort and no 4^b-sized index.  All-zero rows drop out of the score by themselves.
//   spb_project_wide     digits of an ordered list of taxon positions of every key of a pattern list: flattening row /
//                        column indices (sides of <= 31 taxa) and the keys of a sub-alignment
//   spb_pair_tables_wide joint 4x4 tables of every taxon pair of a weighted pattern list ({pattern: value} mappings),
//                        N = E^T diag(v) E on the fp64 tensor cores; deterministic, exact for integer values
#include "common.cuh"

using namespace spb;

namespace {

constexpr unsigned long long kAll = 0xFFFFFFFFFFFFFFFFull;

struct Key128 {
  unsigned long long lo, hi;
};

__device__ __forceinline__ bool is_empty(Key128 k) { return k.lo == kAll && k.hi == kAll; }
__device__ __forceinline__ bool same(Key128 a, Key128 b) { return a.lo == b.lo && a.hi == b.hi; }

// plain 16-byte read: only used by kernels that run after all insertions have completed
__device__ __forceinline__ Key128 load_key(const unsigned long long* keys, uint64_t slot) {
  const ulonglong2 v = *reinterpret_cast<const ulonglong2*>(keys + 2 * slot);
  return Key128{v.x, v.y};
}

__device__ __forceinline__ Key128 cas128(unsigned long long* ptr, Key128 cmp, Key128 val) {
  Key128 old;
  asm volatile(
      "{\n\t.reg .b128 c, v, o;\n\t"
      "mov.b128 c, {%2, %3};\n\t"
      "mov.b128 v, {%4, %5};\n\t"
      "atom.global.cas.b128 o, [%6], c, v;\n\t"
      "mov.b128 {%0, %1}, o;\n\t}"
      : "=l"(old.lo), "=l"(old.hi)
      : "l"(cmp.lo), "l"(cmp.hi), "l"(val.lo), "l"(val.hi), "l"(ptr)
      : "memory");
  return old;
}

__device__ __forceinline__ uint64_t hash128(Key128 k) { return mix64(k.lo ^ mix64(k.hi + 0x9E3779B97F4A7C15ull)); }

struct WideTable {
  unsigned long long* keys;  // [cap][2] = {lo, hi}, EMPTY = all ones
  uint32_t* counts;          // [cap]
  uint32_t* first;           // [cap + 1] first site of every pattern (optional; slot cap = the all-ones key)
  uint64_t mask;
  unsigned long long* special;  // count of the all-ones key
  uint32_t* overflow;
};

__device__ __forceinline__ void table_add(const WideTable& t, Key128 key, uint32_t c, uint32_t f) {
  if (is_empty(key)) {
    atomicAdd(t.special, (unsigned long long)c);
    if (t.first) atomicMin(t.first + t.mask + 1, f);
    return;
  }
  uint64_t h = hash128(key) & t.mask;
  for (uint64_t probe = 0; probe <= t.mask; ++probe) {
    // One 128-bit CAS per probe: it returns the slot's previous content atomically (a 16-byte key cannot be read
    // torn this way while other threads are inserting).  EMPTY -> we inserted; equal -> the key is already there.
    const Key128 k = cas128(t.keys + 2 * h, Key128{kAll, kAll}, key);
    if (is_empty(k) || same(k, key)) {
      atomicAdd(t.counts + h, c);
      if (t.first) atomicMin(t.first + h, f);
      return;
    }
    h = (h + 1) & t.mask;
  }
  atomicExch(t.overflow, 1u);
}

// count of `key` in the table (0 if absent)
__device__ __forceinline__ uint32_t table_find(const unsigned long long* keys, const uint32_t* counts, uint64_t mask,
                                               unsigned long long special, Key128 key) {
  if (is_empty(key)) return (uint32_t)special;
  uint64_t h = hash128(key) & mask;
  for (uint64_t probe = 0; probe <= mask; ++probe) {
    Key128 k = load_key(keys, h);
    if (is_empty(k)) return 0u;
    if (same(k, key)) return counts[h];
    h = (h + 1) & mask;
  }
  return 0u;
}

__device__ __forceinline__ uint32_t to_code(uint32_t c, int is_ascii) {
  if (!is_ascii) return c;
  uint32_t u = c & 0xDFu;
  return u == 'A' ? 0u : u == 'C' ? 1u : u == 'G' ? 2u : u == 'T' ? 3u : 255u;
}

// one thread = one site; lanes = consecutive sites (32-byte coalesced segments per taxon row)
__global__ void __launch_bounds__(256) pack_wide_kernel(const uint8_t* __restrict__ chars, int n, int64_t N, int64_t stride, int is_ascii,
                                                        unsigned long long* __restrict__ wide, uint32_t* __restrict__ valid) {
  const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  unsigned long long lo = 0, hi = 0;
  bool ok = s < N;
  if (ok) {
    for (int j = 0; j < n; ++j) {
      uint32_t c = to_code(__ldg(chars + (int64_t)j * stride + s), is_ascii);
      ok = ok && c <= 3u;
      hi = (hi << 2) | (lo >> 62);
      lo = (lo << 2) | (unsigned long long)(c & 3u);
    }
  }
  if (!ok) { lo = 0; hi = 0; }
  const unsigned m = __ballot_sync(0xFFFFFFFFu, ok);
  if (s < N) *reinterpret_cast<ulonglong2*>(wide + 2 * s) = make_ulonglong2(lo, hi);
  if ((threadIdx.x & 31) == 0 && (s >> 5) < (N + 31) / 32) valid[s >> 5] = m;
}

__global__ void __launch_bounds__(256) count_wide_kernel(const unsigned long long* __restrict__ wide, const uint32_t* __restrict__ valid,
                                                         int64_t site_begin, int64_t site_end, WideTable t, unsigned long long* usable) {
  const int lane = threadIdx.x & 31;
  unsigned long long my_usable = 0;
  // grid-stride over 32-site words so that a warp always holds 32 consecutive sites
  const int64_t w_begin = site_begin >> 5, w_end = (site_end + 31) >> 5;
  const int64_t warp_global = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t warps_total = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t w = w_begin + warp_global; w < w_end; w += warps_total) {
    const int64_t s = w * 32 + lane;
    const uint32_t vbits = __ldg(valid + w);
    const bool ok = ((vbits >> lane) & 1u) && s >= site_begin && s < site_end;
    Key128 key{0, 0};
    if (ok) {
      const ulonglong2 v = __ldg(reinterpret_cast<const ulonglong2*>(wide + 2 * s));
      key = Key128{v.x, v.y};
    }
    my_usable += ok ? 1u : 0u;
    const unsigned okmask = __ballot_sync(0xFFFFFFFFu, ok);
    if (okmask == 0u) continue;
    const int lead = __ffs(okmask) - 1;
    Key128 lk;
    lk.lo = __shfl_sync(0xFFFFFFFFu, key.lo, lead);
    lk.hi = __shfl_sync(0xFFFFFFFFu, key.hi, lead);
    const bool grp = ok && same(key, lk);
    const unsigned grpmask = __ballot_sync(0xFFFFFFFFu, grp);
    if (ok && (!grp || lane == lead)) table_add(t, key, lane == lead ? (uint32_t)__popc(grpmask) : 1u, (uint32_t)s);  // lead = earliest site
  }
  for (int o = 16; o > 0; o >>= 1) my_usable += __shfl_xor_sync(0xFFFFFFFFu, my_usable, o);
  if (lane == 0 && my_usable && usable) atomicAdd(usable, my_usable);
}

__global__ void merge_wide_kernel(const unsigned long long* __restrict__ keys, const uint32_t* __restrict__ counts,
                                  const uint32_t* __restrict__ first, int64_t num, WideTable t) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < num) table_add(t, Key128{keys[2 * i], keys[2 * i + 1]}, counts[i], first ? first[i] : 0xFFFFFFFFu);
}

// unordered compaction (the caller sorts): one atomic per warp
__global__ void compact_wide_kernel(const unsigned long long* __restrict__ hkeys, const uint32_t* __restrict__ hcounts,
                                    const uint32_t* __restrict__ hfirst, int64_t cap, unsigned long long* keys, uint32_t* counts,
                                    uint32_t* first, int64_t capacity, unsigned long long* num) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int lane = threadIdx.x & 31;
  Key128 k{kAll, kAll};
  if (i < cap) k = load_key(hkeys, (uint64_t)i);
  const bool used = !is_empty(k);
  const unsigned m = __ballot_sync(0xFFFFFFFFu, used);
  if (m == 0u) return;
  unsigned long long base = 0;
  if (lane == __ffs(m) - 1) base = atomicAdd(num, (unsigned long long)__popc(m));
  base = __shfl_sync(0xFFFFFFFFu, base, __ffs(m) - 1);
  if (used) {
    const int64_t o = (int64_t)base + __popc(m & ((1u << lane) - 1u));
    if (o < capacity) {
      keys[2 * o] = k.lo;
      keys[2 * o + 1] = k.hi;
      counts[o] = hcounts[i];
      if (first) first[o] = hfirst ? hfirst[i] : 0xFFFFFFFFu;
    }
  }
}

struct ThinSplit {
  int a;          // taxa on the thin side (1, 2 or 3)
  int shift[3];   // bit position of their digits inside the 128-bit key
};

__device__ __forceinline__ uint32_t get_digit(Key128 k, int shift) {
  return shift < 64 ? (uint32_t)((k.lo >> shift) & 3ull) : (uint32_t)((k.hi >> (shift - 64)) & 3ull);
}
__device__ __forceinline__ Key128 set_digit(Key128 k, int shift, uint32_t d) {
  if (shift < 64) k.lo = (k.lo & ~(3ull << shift)) | ((unsigned long long)d << shift);
  else k.hi = (k.hi & ~(3ull << (shift - 64))) | ((unsigned long long)d << (shift - 64));
  return k;
}

__device__ __forceinline__ uint64_t column_bit(Key128 p, const ThinSplit& sp, uint64_t bit_mask) {
  for (int t = 0; t < sp.a; ++t) p = set_digit(p, sp.shift[t], 0u);
  return hash128(p) & bit_mask;
}

// Column filter of a thin split.  The column of a pattern is its key with the thin side's digits zeroed; a pattern
// only has partners (same column, other row) if another pattern hashes to its column bit.  thin_mark_kernel sets
// seen[h(column)] for every pattern and multi[h] when the bit was already set; thin_gram_wide_kernel then skips the
// 4^a - 1 table lookups of every pattern whose multi bit is clear.  At 64 taxa nearly every site is its own pattern
// and almost no column holds two, so the lookups (random 32-byte DRAM reads, the whole cost of the kernel) drop from
// (4^a - 1) / 2 per pattern to the false-positive rate of the filter (about one pattern in six at 2 x cap bits).
__global__ void __launch_bounds__(256) thin_mark_kernel(const unsigned long long* __restrict__ hkeys, int64_t cap,
                                                        const unsigned long long* __restrict__ special, ThinSplit sp,
                                                        uint32_t* __restrict__ seen, uint32_t* __restrict__ multi, uint64_t bit_mask) {
  const unsigned long long spc = *special;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i <= cap; i += (int64_t)gridDim.x * blockDim.x) {
    Key128 p{kAll, kAll};
    if (i < cap) {
      p = load_key(hkeys, (uint64_t)i);
      if (is_empty(p)) continue;
    } else if (spc == 0ull) {
      continue;
    }
    const uint64_t h = column_bit(p, sp, bit_mask);
    const uint32_t bit = 1u << (h & 31);
    const uint32_t old = atomicOr(seen + (h >> 5), bit);
    if (old & bit) atomicOr(multi + (h >> 5), bit);
  }
}

__global__ void __launch_bounds__(256) thin_gram_wide_kernel(const unsigned long long* __restrict__ hkeys, const uint32_t* __restrict__ hcounts,
                                                             int64_t cap, const unsigned long long* __restrict__ special, ThinSplit sp,
                                                             const uint32_t* __restrict__ multi, uint64_t bit_mask,
                                                             double* __restrict__ G) {
  // per-CTA partial Gram in 64-bit integers: shared-memory integer atomics are native (a double atomicAdd in shared
  // memory is a CAS loop, which collapses on the few row patterns that carry most sites); sum count^2 <= N^2 < 2^64
  __shared__ unsigned long long sG[64 * 64];  // R x R, row stride R (R = 4, 16 or 64)
  const int R = 1 << (2 * sp.a);
  for (int i = threadIdx.x; i < R * R; i += blockDim.x) sG[i] = 0ull;
  __syncthreads();
  const unsigned long long spc = *special;
  const int lane = threadIdx.x & 31;
  // slot index cap stands for the all-ones pattern, which lives outside the table.  Warp-uniform trip count: the diagonal term is
  // aggregated over the warp with full-mask intrinsics before the lanes diverge into the look-ups.
  for (int64_t base = (int64_t)blockIdx.x * blockDim.x + (threadIdx.x & ~31); base <= cap; base += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = base + lane;
    Key128 p{kAll, kAll};
    uint32_t cp = 0;
    bool valid = false;
    if (i < cap) {
      p = load_key(hkeys, (uint64_t)i);
      valid = !is_empty(p);
      if (valid) cp = hcounts[i];
    } else if (i == cap && spc != 0ull) {
      valid = true;
      cp = (uint32_t)spc;
    }
    uint32_t r1 = 0;
    for (int t = 0; t < sp.a; ++t) r1 = (r1 << 2) | get_digit(p, sp.shift[t]);
    // Diagonal term count^2.  Nearly all sites sit in a handful of rows, so one shared-memory atomic per pattern serialises the CTA
    // on a few addresses (and 16 register accumulators cost half the resident warps of this latency-bound kernel: measured 3.2 ms
    // against 2.4 ms per split).  Patterns seen once -- almost all at 64 taxa -- are counted per (warp, row) with one atomic.
    {
      const uint32_t tag = valid ? ((r1 << 1) | (cp == 1u ? 1u : 0u)) : 0xFFFFFFFFu;
      const unsigned peers = __match_any_sync(0xFFFFFFFFu, tag);
      if (valid) {
        if (cp == 1u) {
          if (lane == __ffs(peers) - 1) atomicAdd(&sG[r1 * R + r1], (unsigned long long)__popc(peers));
        } else {
          atomicAdd(&sG[r1 * R + r1], (unsigned long long)cp * (unsigned long long)cp);
        }
      }
    }
    if (!valid) continue;
    // every unordered pair of patterns that differ only in their row part is found once, from its smaller row
    if (multi) {
      const uint64_t h = column_bit(p, sp, bit_mask);
      if (!((multi[h >> 5] >> (h & 31)) & 1u)) continue;  // no other pattern shares this column
    }
    for (int r2 = (int)r1 + 1; r2 < R; ++r2) {
      Key128 q = p;
      for (int t = 0; t < sp.a; ++t) q = set_digit(q, sp.shift[t], ((uint32_t)r2 >> (2 * (sp.a - 1 - t))) & 3u);
      const uint32_t cq = table_find(hkeys, hcounts, (uint64_t)cap - 1, spc, q);
      if (cq) {
        const unsigned long long v = (unsigned long long)cp * (unsigned long long)cq;
        atomicAdd(&sG[r1 * R + r2], v);
        atomicAdd(&sG[r2 * R + r1], v);
      }
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < R * R; i += blockDim.x) {
    const unsigned long long v = sG[i];
    if (v) atomicAdd(G + i, (double)v);  // integer-valued partial sums: exact and order independent below 2^53
  }
}

// ---- pattern lists with 128-bit keys ({pattern: value} mappings of 32..64 taxa) ----

struct Projection {
  int m;                      // positions read, most significant first
  uint8_t shift[SPB_MAX_TAXA];  // bit position of each position's digit inside the 128-bit key
};

// digits of `pr` positions of every key, packed base 4: a uint64 word per key for m <= 31, a {lo, hi} key for more
__global__ void __launch_bounds__(256) project_wide_kernel(const unsigned long long* __restrict__ keys, int64_t num, Projection pr,
                                                           unsigned long long* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= num) return;
  const ulonglong2 v = __ldg(reinterpret_cast<const ulonglong2*>(keys + 2 * i));
  const Key128 k{v.x, v.y};
  unsigned long long lo = 0, hi = 0;
  for (int t = 0; t < pr.m; ++t) {
    hi = (hi << 2) | (lo >> 62);
    lo = (lo << 2) | get_digit(k, pr.shift[t]);
  }
  if (pr.m <= 31) {
    out[i] = lo;
  } else {
    *reinterpret_cast<ulonglong2*>(out + 2 * i) = make_ulonglong2(lo, hi);
  }
}

// Joint tables of every taxon pair from a weighted pattern list: with E the P x 4n one-hot matrix of the digits (column
// 4 t + x = [taxon t of the pattern is in state x]), N = E^T diag(v) E, i.e. N[4i + x][4j + y] = sum_p v_p [p_i = x][p_j = y].
// The 4n x 4n product runs on the fp64 tensor cores (DMMA m8n8k4) with the fragments generated from the keys: lane l
// holds A[l / 4][l % 4] = v_p [digit of row l / 4], B[l % 4][l / 4] = [digit of column l / 4] of pattern p = base + l % 4.
// Grid: x = pattern chunk, y = 32 x 32 output block of the upper block triangle.  A warp keeps the 4 x 4 tiles of its
// block in registers over every 4th step of its chunk; the 4 warps are added in warp order and the chunk partials by
// pair_wide_reduce_kernel in chunk order, so the result does not depend on scheduling.  Products are v * 1 or v * 0:
// integer-valued tables are summed exactly (below 2^53).  Values must be finite (inf * 0 would spread NaN to the
// other cells of a row).
constexpr int kPairWarps = 4;
constexpr int kPairBlock = 32;                  // output rows / columns per block
constexpr int64_t kPairChunkMin = 4096;         // patterns per chunk at least ...
constexpr int64_t kPairChunksMax = 64;          // ... and at most this many chunks (the workspace is chunks x blocks x 8 KB)

__device__ __forceinline__ double one_hot(unsigned long long lo, unsigned long long hi, int shift, uint32_t state, double v) {
  const uint32_t d = shift < 64 ? (uint32_t)((lo >> shift) & 3ull) : (uint32_t)((hi >> (shift - 64)) & 3ull);
  return d == state ? v : 0.0;
}

__device__ __forceinline__ void dmma884(double& d0, double& d1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};" : "+d"(d0), "+d"(d1) : "d"(a), "d"(b));
}

__global__ void __launch_bounds__(32 * kPairWarps) pair_wide_kernel(const unsigned long long* __restrict__ keys, const double* __restrict__ vals,
                                                                    int64_t num, int n, int nblocks, int64_t chunk, double* __restrict__ ws) {
  __shared__ double red[kPairWarps][kPairBlock][kPairBlock];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, kq = lane & 3, grp = lane >> 2;
  int bi = 0, rem = blockIdx.y;
  while (rem >= nblocks - bi) { rem -= nblocks - bi; ++bi; }
  const int bj = bi + rem;
  // row / column 32 b + 8 t + grp of the product = taxon 8 b + 2 t + grp / 4 in state grp % 4; -1 = padding past 4n
  const uint32_t state = (uint32_t)(grp & 3);
  int sa[4], sb[4];
#pragma unroll
  for (int t = 0; t < 4; ++t) {
    const int ta = 8 * bi + 2 * t + (grp >> 2), tb = 8 * bj + 2 * t + (grp >> 2);
    sa[t] = ta < n ? 2 * (n - 1 - ta) : -1;
    sb[t] = tb < n ? 2 * (n - 1 - tb) : -1;
  }
  double acc[4][4][2];
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) acc[a][b][0] = acc[a][b][1] = 0.0;
  const int64_t p_begin = (int64_t)blockIdx.x * chunk;
  const int64_t p_end = min(num, p_begin + chunk);
  for (int64_t p0 = p_begin + 4 * warp; p0 < p_end; p0 += 4 * kPairWarps) {
    const int64_t p = p0 + kq;
    unsigned long long lo = 0, hi = 0;
    double v = 0.0;
    if (p < p_end) {
      const ulonglong2 k = __ldg(reinterpret_cast<const ulonglong2*>(keys + 2 * p));
      lo = k.x;
      hi = k.y;
      v = __ldg(vals + p);
    }
    double fa[4], fb[4];
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      fa[t] = sa[t] >= 0 ? one_hot(lo, hi, sa[t], state, v) : 0.0;
      fb[t] = sb[t] >= 0 ? one_hot(lo, hi, sb[t], state, 1.0) : 0.0;
    }
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int b = 0; b < 4; ++b) dmma884(acc[a][b][0], acc[a][b][1], fa[a], fb[b]);
  }
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) {
      red[warp][8 * a + grp][8 * b + 2 * kq] = acc[a][b][0];
      red[warp][8 * a + grp][8 * b + 2 * kq + 1] = acc[a][b][1];
    }
  __syncthreads();
  double* out = ws + ((int64_t)blockIdx.x * gridDim.y + blockIdx.y) * (kPairBlock * kPairBlock);
  for (int e = threadIdx.x; e < kPairBlock * kPairBlock; e += 32 * kPairWarps) {
    const int r = e / kPairBlock, c = e - r * kPairBlock;
    double s = red[0][r][c];
#pragma unroll
    for (int w = 1; w < kPairWarps; ++w) s += red[w][r][c];
    out[e] = s;
  }
}

// chunk partials -> N double [n][n][4][4]; entries below the block diagonal (and below the diagonal of a diagonal block)
// are read from their mirror image, so N[j][i] is exactly N[i][j]^T
__global__ void pair_wide_reduce_kernel(const double* __restrict__ ws, int64_t nchunks, int nblocks, int n, double* __restrict__ N) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)n * n * 16) return;
  const int ij = (int)(idx >> 4), cell = (int)(idx & 15);
  const int i = ij / n, j = ij - i * n;
  int r = 4 * i + (cell >> 2), c = 4 * j + (cell & 3);
  if (r > c) { const int t = r; r = c; c = t; }
  const int rb = r / kPairBlock, cb = c / kPairBlock;
  const int blk = rb * nblocks - rb * (rb - 1) / 2 + (cb - rb);
  const int64_t nbp = (int64_t)nblocks * (nblocks + 1) / 2;
  const double* src = ws + (int64_t)blk * (kPairBlock * kPairBlock) + (r % kPairBlock) * kPairBlock + (c % kPairBlock);
  double s = 0.0;
  for (int64_t q = 0; q < nchunks; ++q) s += src[q * nbp * (kPairBlock * kPairBlock)];
  N[idx] = s;
}

// chunk length (a multiple of 16 patterns) and number of chunks of a pattern list: a function of `num` only, so that the
// summation order -- and with it every bit of the result -- is the same on every device
void pair_wide_plan(int64_t num, int64_t* chunk, int64_t* nchunks) {
  int64_t c = (num + kPairChunkMin - 1) / kPairChunkMin;
  if (c > kPairChunksMax) c = kPairChunksMax;
  if (c < 1) c = 1;
  int64_t len = (num + c - 1) / c;
  len = (len + 15) / 16 * 16;
  if (len < 16) len = 16;
  *chunk = len;
  *nchunks = (num + len - 1) / len;
  if (*nchunks < 1) *nchunks = 1;
}

int pair_wide_blocks(int n) { return (4 * n + kPairBlock - 1) / kPairBlock; }

int check_table(const uint64_t* d_hkeys, const uint32_t* d_hcounts, int64_t cap, const char* who) {
  SPB_REQUIRE(d_hkeys && d_hcounts, "%s: NULL table", who);
  SPB_REQUIRE(cap >= 2 && (cap & (cap - 1)) == 0, "%s: capacity must be a power of two", who);
  SPB_REQUIRE((reinterpret_cast<uintptr_t>(d_hkeys) & 15) == 0, "%s: the key array must be 16-byte aligned", who);
  return SPB_OK;
}

}  // namespace

extern "C" int spb_pack_wide(const uint8_t* d_chars, int n_taxa, int64_t n_sites, int64_t row_stride, int is_ascii, uint64_t* d_wide,
                             uint32_t* d_valid, void* stream) {
  SPB_REQUIRE(d_chars && d_wide && d_valid && n_taxa >= 1 && n_taxa <= SPB_MAX_TAXA && n_sites >= 0 && row_stride >= n_sites,
              "spb_pack_wide: bad arguments (n_taxa=%d n_sites=%lld)", n_taxa, (long long)n_sites);
  SPB_REQUIRE((reinterpret_cast<uintptr_t>(d_wide) & 15) == 0, "spb_pack_wide: the key array must be 16-byte aligned");
  if (n_sites == 0) return SPB_OK;
  const int64_t padded = (n_sites + 31) / 32 * 32;  // whole warps, so that every validity word is written
  pack_wide_kernel<<<(unsigned)((padded + 255) / 256), 256, 0, (cudaStream_t)stream>>>(d_chars, n_taxa, n_sites, row_stride, is_ascii,
                                                                                      (unsigned long long*)d_wide, d_valid);
  SPB_LAUNCH_CHECK();
  return SPB_OK;
}

extern "C" int spb_count_hash_wide(const uint64_t* d_wide, const uint32_t* d_valid, int64_t site_begin, int64_t site_end,
                                   uint64_t* d_hkeys, uint32_t* d_hcounts, uint32_t* d_hfirst, int64_t cap, uint64_t* d_special,
                                   uint64_t* d_usable, uint32_t* d_overflow, void* stream) {
  SPB_REQUIRE(d_wide && d_valid && d_special && d_overflow, "spb_count_hash_wide: NULL buffer");
  int rc = check_table(d_hkeys, d_hcounts, cap, "spb_count_hash_wide");
  if (rc) return rc;
  SPB_REQUIRE(site_begin >= 0 && site_end >= site_begin && site_end < (1ll << 32), "spb_count_hash_wide: bad site range");
  if (site_end == site_begin) return SPB_OK;
  WideTable t{(unsigned long long*)d_hkeys, d_hcounts, d_hfirst, (uint64_t)cap - 1, (unsigned long long*)d_special, d_overflow};
  int64_t words = ((site_end + 31) >> 5) - (site_begin >> 5);
  int64_t grid = (int64_t)sm_count() * 8;
  if (grid > (words + 7) / 8) grid = (words + 7) / 8;
  if (grid < 1) grid = 1;
  count_wide_kernel<<<(unsigned)grid, 256, 0, (cudaStream_t)stream>>>((const unsigned long long*)d_wide, d_valid, site_begin, site_end, t,
                                                                    (unsigned long long*)d_usable);
  SPB_LAUNCH_CHECK();
  return SPB_OK;
}

extern "C" int spb_hash_merge_wide(const uint64_t* d_keys, const uint32_t* d_counts, const uint32_t* d_first, int64_t num,
                                   uint64_t* d_hkeys, uint32_t* d_hcounts, uint32_t* d_hfirst, int64_t cap, uint64_t* d_special,
                                   uint32_t* d_overflow, void* stream) {
  SPB_REQUIRE(d_special && d_overflow, "spb_hash_merge_wide: NULL buffer");
  int rc = check_table(d_hkeys, d_hcounts, cap, "spb_hash_merge_wide");
  if (rc) return rc;
  if (num <= 0) return SPB_OK;
  SPB_REQUIRE(d_keys && d_counts, "spb_hash_merge_wide: NULL list");
  WideTable t{(unsigned long long*)d_hkeys, d_hcounts, d_hfirst, (uint64_t)cap - 1, (unsigned long long*)d_special, d_overflow};
  merge_wide_kernel<<<(unsigned)((num + 255) / 256), 256, 0, (cudaStream_t)stream>>>((const unsigned long long*)d_keys, d_counts, d_first,
                                                                                    num, t);
  SPB_LAUNCH_CHECK();
  return SPB_OK;
}

extern "C" int spb_compact_hash_wide(const uint64_t* d_hkeys, const uint32_t* d_hcounts, const uint32_t* d_hfirst, int64_t cap,
                                     uint64_t* d_keys, uint32_t* d_counts, uint32_t* d_first, int64_t capacity, uint64_t* d_num,
                                     void* stream) {
  int rc = check_table(d_hkeys, d_hcounts, cap, "spb_compact_hash_wide");
  if (rc) return rc;
  SPB_REQUIRE(d_keys && d_counts && d_num && capacity >= 0, "spb_compact_hash_wide: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  SPB_CUDA(cudaMemsetAsync(d_num, 0, 8, st));
  compact_wide_kernel<<<(unsigned)((cap + 255) / 256), 256, 0, st>>>((const unsigned long long*)d_hkeys, d_hcounts, d_hfirst, cap,
                                                                   (unsigned long long*)d_keys, d_counts, d_first, capacity,
                                                                   (unsigned long long*)d_num);
  SPB_LAUNCH_CHECK();
  return SPB_OK;
}

extern "C" int spb_thin_gram_wide_filtered(const uint64_t* d_hkeys, const uint32_t* d_hcounts, int64_t cap, const uint64_t* d_special,
                                           int n_taxa, const uint8_t* h_idx_a, int a, uint32_t* d_filter, int64_t filter_words,
                                           double* d_G, void* stream) {
  int rc = check_table(d_hkeys, d_hcounts, cap, "spb_thin_gram_wide");
  if (rc) return rc;
  SPB_REQUIRE(d_special && d_G && h_idx_a, "spb_thin_gram_wide: NULL buffer");
  SPB_REQUIRE(n_taxa >= 2 && n_taxa <= SPB_MAX_TAXA && a >= 1 && a <= 3, "spb_thin_gram_wide: the thin side must have 1, 2 or 3 of <= 64 taxa");
  ThinSplit sp;
  sp.a = a;
  for (int t = 0; t < a; ++t) {
    SPB_REQUIRE(h_idx_a[t] < n_taxa && (t == 0 || h_idx_a[t] != h_idx_a[0]) && (t < 2 || h_idx_a[2] != h_idx_a[1]),
                "spb_thin_gram_wide: bad taxon positions");
    sp.shift[t] = 2 * (n_taxa - 1 - h_idx_a[t]);
  }
  for (int t = a; t < 3; ++t) sp.shift[t] = 0;
  cudaStream_t st = (cudaStream_t)stream;
  const int R = 1 << (2 * a);
  SPB_CUDA(cudaMemsetAsync(d_G, 0, (size_t)R * R * sizeof(double), st));
  int64_t grid = (int64_t)sm_count() * 8;
  if (grid > (cap + 256) / 256) grid = (cap + 256) / 256;
  const uint32_t* multi = nullptr;
  uint64_t bit_mask = 0;
  if (d_filter) {
    SPB_REQUIRE(filter_words >= 1 && (filter_words & (filter_words - 1)) == 0, "spb_thin_gram_wide: filter_words must be a power of two");
    SPB_CUDA(cudaMemsetAsync(d_filter, 0, (size_t)2 * filter_words * sizeof(uint32_t), st));
    bit_mask = (uint64_t)filter_words * 32 - 1;
    thin_mark_kernel<<<(unsigned)grid, 256, 0, st>>>((const unsigned long long*)d_hkeys, cap, (const unsigned long long*)d_special, sp,
                                                     d_filter, d_filter + filter_words, bit_mask);
    SPB_LAUNCH_CHECK();
    multi = d_filter + filter_words;
  }
  thin_gram_wide_kernel<<<(unsigned)grid, 256, 0, st>>>((const unsigned long long*)d_hkeys, d_hcounts, cap, (const unsigned long long*)d_special,
                                                        sp, multi, bit_mask, d_G);
  SPB_LAUNCH_CHECK();
  return SPB_OK;
}

extern "C" int64_t spb_thin_filter_words(int64_t cap) {
  int64_t w = 1;
  // bits per bitmap: 8 x cap by default (false-positive rate of the column filter ~ patterns / bits: 1 in 16 at a half-full
  // table; 2 x cap bits, the round-1 size, let one pattern in six through to its 4^a - 1 random table reads)
  static int per_cap = 0;
  if (!per_cap) {
    const char* e = getenv("SPB_THIN_FILTER_BITS_PER_SLOT");
    per_cap = e ? atoi(e) : 8;
    if (per_cap < 1 || per_cap > 64) per_cap = 8;
  }
  while (w * 32 < cap * per_cap) w *= 2;
  return w;
}

extern "C" int spb_thin_gram_wide(const uint64_t* d_hkeys, const uint32_t* d_hcounts, int64_t cap, const uint64_t* d_special, int n_taxa,
                                  const uint8_t* h_idx_a, int a, double* d_G, void* stream) {
  return spb_thin_gram_wide_filtered(d_hkeys, d_hcounts, cap, d_special, n_taxa, h_idx_a, a, nullptr, 0, d_G, stream);
}

extern "C" int spb_project_wide(const uint64_t* d_keys, int64_t num, int n_taxa, const uint8_t* h_pos, int m, uint64_t* d_out,
                                void* stream) {
  SPB_REQUIRE(n_taxa >= 1 && n_taxa <= SPB_MAX_TAXA && m >= 0 && m <= n_taxa && num >= 0,
              "spb_project_wide: bad arguments (n_taxa=%d m=%d)", n_taxa, m);
  SPB_REQUIRE(m == 0 || h_pos, "spb_project_wide: NULL position list");
  Projection pr;
  pr.m = m;
  for (int t = 0; t < m; ++t) {
    SPB_REQUIRE(h_pos[t] < n_taxa, "spb_project_wide: position %d out of range (n_taxa=%d)", (int)h_pos[t], n_taxa);
    pr.shift[t] = (uint8_t)(2 * (n_taxa - 1 - h_pos[t]));
  }
  if (num == 0) return SPB_OK;
  SPB_REQUIRE(d_keys && d_out, "spb_project_wide: NULL buffer");
  SPB_REQUIRE((reinterpret_cast<uintptr_t>(d_keys) & 15) == 0 && (m <= 31 || (reinterpret_cast<uintptr_t>(d_out) & 15) == 0),
              "spb_project_wide: 128-bit key arrays must be 16-byte aligned");
  project_wide_kernel<<<(unsigned)((num + 255) / 256), 256, 0, (cudaStream_t)stream>>>((const unsigned long long*)d_keys, num, pr,
                                                                                     (unsigned long long*)d_out);
  SPB_LAUNCH_CHECK();
  return SPB_OK;
}

extern "C" int64_t spb_pair_tables_wide_ws(int64_t num, int n_taxa) {
  if (n_taxa < 1 || n_taxa > SPB_MAX_TAXA || num < 0) return 0;
  int64_t chunk, nchunks;
  pair_wide_plan(num, &chunk, &nchunks);
  const int64_t nb = pair_wide_blocks(n_taxa);
  return nchunks * (nb * (nb + 1) / 2) * (kPairBlock * kPairBlock);
}

extern "C" int spb_pair_tables_wide(const uint64_t* d_keys, const double* d_vals, int64_t num, int n_taxa, double* d_N, double* d_ws,
                                    void* stream) {
  SPB_REQUIRE(d_N && n_taxa >= 1 && n_taxa <= SPB_MAX_TAXA && num >= 0, "spb_pair_tables_wide: bad arguments (n_taxa=%d)", n_taxa);
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t cells = (int64_t)n_taxa * n_taxa * 16;
  if (num == 0) {
    SPB_CUDA(cudaMemsetAsync(d_N, 0, (size_t)cells * sizeof(double), st));
    return SPB_OK;
  }
  SPB_REQUIRE(d_keys && d_vals && d_ws, "spb_pair_tables_wide: NULL buffer");
  SPB_REQUIRE((reinterpret_cast<uintptr_t>(d_keys) & 15) == 0, "spb_pair_tables_wide: the key array must be 16-byte aligned");
  int64_t chunk, nchunks;
  pair_wide_plan(num, &chunk, &nchunks);
  const int nb = pair_wide_blocks(n_taxa);
  const dim3 grid((unsigned)nchunks, (unsigned)(nb * (nb + 1) / 2));
  pair_wide_kernel<<<grid, 32 * kPairWarps, 0, st>>>((const unsigned long long*)d_keys, d_vals, num, n_taxa, nb, chunk, d_ws);
  SPB_LAUNCH_CHECK();
  pair_wide_reduce_kernel<<<(unsigned)((cells + 255) / 256), 256, 0, st>>>(d_ws, nchunks, nb, n_taxa, d_N);
  SPB_LAUNCH_CHECK();
  return SPB_OK;
}

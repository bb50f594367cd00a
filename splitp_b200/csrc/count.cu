// Kernel 1: site-pattern compression and counting over the 2-bit-packed (site-major) alignment.
// Replaces splitp/parsers/fasta.py:48-63 (get_pattern_counts) and the counting half of
// splitp/simulation.py:43-54.  Bit-exact integer work.
//
// Data flow per CTA (256 threads, tile = 8192 sites, persistent over tiles):
//   coalesced 128-bit loads of the tile's bit stream -> shared memory
//   -> per-site key extraction (funnel shifts), 32 consecutive sites per warp iteration
//   -> WARP-PRIVATE direct-mapped cache in shared memory (256 entries per warp):
//        hit  : one shared-memory atomicAdd on the entry's counter (lanes that carry the same key as lane 0 -- the
//               usual case, alignments are dominated by a few very frequent patterns -- are first aggregated with
//               one ballot, so the hot pattern costs one atomic per warp iteration);
//        miss : the missing lanes claim their slot, the winner evicts the resident entry to the global table and
//               installs its key, lanes with the same key then add to it, lanes that lost the slot to a different
//               key bypass the cache.
//      The cache absorbs the frequent patterns on chip: the global table sees one update per (warp, pattern)
//      residency instead of one per site.  No __match_any_sync: its cost grows with the number of distinct keys
//      in the warp and made the first two versions of this kernel issue-bound (profiles/r1_kernel_roofline_*).
//   -> global sink: direct-indexed table (n <= 14, one RED per eviction) or open-addressing hash table.
#include "common.cuh"
#include <type_traits>

using namespace spb;

namespace {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr int kTileSites = 32 * kThreads;  // 8192
constexpr int kCacheSlots = 256;           // per warp

struct DirectSink {
  uint32_t* table;
  uint32_t* first;
  __device__ __forceinline__ void add(uint64_t key, uint32_t c, uint32_t f) const {
    atomicAdd(table + key, c);
    if (first) atomicMin(first + key, f);
  }
};

struct HashSink {
  unsigned long long* keys;
  uint32_t* counts;
  uint32_t* first;
  uint64_t mask;
  uint32_t* overflow;
  __device__ __forceinline__ void add(uint64_t key, uint32_t c, uint32_t f) const {
    uint64_t h = mix64(key) & mask;
    for (uint64_t probe = 0; probe <= mask; ++probe) {
      unsigned long long k = keys[h];
      if (k == SPB_EMPTY_KEY) {
        unsigned long long old = atomicCAS(keys + h, (unsigned long long)SPB_EMPTY_KEY, (unsigned long long)key);
        if (old == SPB_EMPTY_KEY) k = key; else k = old;
      }
      if (k == key) {
        atomicAdd(counts + h, c);
        if (first) atomicMin(first + h, f);
        return;
      }
      h = (h + 1) & mask;
    }
    atomicExch(overflow, 1u);
  }
};

__device__ __forceinline__ uint32_t cache_slot(uint64_t key) {
  uint32_t x = (uint32_t)key ^ (uint32_t)(key >> 32) * 0x9E3779B1u;
  x ^= x >> 15;
  x *= 0x2C1B3C6Du;
  return (x >> 24) & (kCacheSlots - 1);
}

template <class Sink>
__global__ void __launch_bounds__(kThreads) count_kernel(const uint32_t* __restrict__ sm, int64_t sm_words,
                                                         const uint32_t* __restrict__ valid, int64_t valid_words, int n,
                                                         int64_t site_begin, int64_t site_end, int64_t tile_begin,
                                                         int64_t tile_end, Sink sink, unsigned long long* usable) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  unsigned long long* c_keys = reinterpret_cast<unsigned long long*>(smem_raw);  // [kWarps][kCacheSlots]
  uint32_t* c_cnt = reinterpret_cast<uint32_t*>(c_keys + kWarps * kCacheSlots);    // [kWarps][kCacheSlots]
  uint32_t* c_first = c_cnt + kWarps * kCacheSlots;                                // [kWarps][kCacheSlots]
  uint32_t* c_claim = c_first + kWarps * kCacheSlots;                              // [kWarps][kCacheSlots]
  uint32_t* s_tile = c_claim + kWarps * kCacheSlots;                               // 512*n words + 4 pad
  __shared__ uint32_t s_usable;

  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int bits = 2 * n;
  const int tile_words = (kTileSites / 32) * bits;  // 512 n
  const uint64_t kmask = (bits == 64) ? ~0ull : ((1ull << bits) - 1ull);
  const bool want_first = sink.first != nullptr;
  unsigned long long* wk = c_keys + wid * kCacheSlots;
  uint32_t* wc = c_cnt + wid * kCacheSlots;
  uint32_t* wf = c_first + wid * kCacheSlots;
  uint32_t* wclaim = c_claim + wid * kCacheSlots;

  for (int i = lane; i < kCacheSlots; i += 32) { wk[i] = SPB_EMPTY_KEY; wc[i] = 0; wf[i] = 0xFFFFFFFFu; }
  if (tid == 0) s_usable = 0;
  __syncthreads();

  uint32_t my_usable = 0;
  for (int64_t tile = tile_begin + blockIdx.x; tile < tile_end; tile += gridDim.x) {
    const int64_t base_site = tile * kTileSites;
    const int64_t base_word = tile * (int64_t)tile_words;
    __syncthreads();  // every warp is done reading the previous tile
    // coalesced 128-bit loads of the tile (tile_words is a multiple of 4, base_word of 4)
    for (int v = tid; v < tile_words / 4; v += kThreads) {
      int64_t gw = base_word + (int64_t)v * 4;
      uint4 x = make_uint4(0, 0, 0, 0);
      if (gw + 4 <= sm_words) x = __ldg(reinterpret_cast<const uint4*>(sm + gw));
      reinterpret_cast<uint4*>(s_tile)[v] = x;
    }
    if (tid < 4) s_tile[tile_words + tid] = 0;
    __syncthreads();
    // warp `wid` owns the 1024 consecutive sites [wid * 1024, wid * 1024 + 1024) of the tile
    const int64_t vw0 = (base_site >> 5) + wid * 32;
    const uint32_t vmine = (vw0 + lane < valid_words) ? __ldg(valid + vw0 + lane) : 0u;  // lane l: validity word of iteration l
#pragma unroll 1
    for (int it = 0; it < 32; ++it) {
      const int sl = wid * 1024 + it * 32 + lane;  // consecutive lanes = consecutive sites
      const int64_t site = base_site + sl;
      const uint32_t vbits = __shfl_sync(0xFFFFFFFFu, vmine, it);
      const bool ok = ((vbits >> lane) & 1u) && site >= site_begin && site < site_end;
      const uint32_t bp = (uint32_t)sl * (uint32_t)bits;
      const uint32_t w = bp >> 5, sh = bp & 31;
      const uint32_t w0 = s_tile[w], w1 = s_tile[w + 1], w2 = s_tile[w + 2];
      uint64_t key = ((uint64_t)__funnelshift_r(w1, w2, sh) << 32) | (uint64_t)__funnelshift_r(w0, w1, sh);
      key &= kmask;
      my_usable += ok ? 1u : 0u;
      const unsigned okmask = __ballot_sync(0xFFFFFFFFu, ok);
      if (okmask == 0u) continue;
      // aggregate the lanes that carry the key of the first usable lane (the frequent-pattern fast path)
      const int lead = __ffs(okmask) - 1;
      const uint32_t k_lo = __shfl_sync(0xFFFFFFFFu, (uint32_t)key, lead), k_hi = __shfl_sync(0xFFFFFFFFu, (uint32_t)(key >> 32), lead);
      const bool same = ok && key == (((uint64_t)k_hi << 32) | k_lo);
      const unsigned samemask = __ballot_sync(0xFFFFFFFFu, same);
      const bool active = ok && (!same || lane == lead);       // one representative for the aggregated group
      const uint32_t c = (lane == lead) ? (uint32_t)__popc(samemask) : 1u;
      const uint32_t slot = cache_slot(key);
      const unsigned long long k0 = wk[slot];
      const bool hit = active && k0 == key;
      if (hit) atomicAdd(wc + slot, c);
      const bool miss = active && !hit;
      if (__ballot_sync(0xFFFFFFFFu, miss) != 0u) {
        if (miss) wclaim[slot] = (uint32_t)lane;
        __syncwarp();
        if (miss && wclaim[slot] == (uint32_t)lane) {  // installer: evict the resident entry, install this key
          if (k0 != SPB_EMPTY_KEY) sink.add(k0, wc[slot], wf[slot]);
          wk[slot] = key; wc[slot] = 0u; wf[slot] = 0xFFFFFFFFu;
        }
        __syncwarp();
        if (miss) {
          if (wk[slot] == key) {
            atomicAdd(wc + slot, c);
            if (want_first) atomicMin(wf + slot, (uint32_t)site);
          } else {
            sink.add(key, c, (uint32_t)site);  // lost the slot to a different key: bypass the cache
          }
        }
        __syncwarp();
      }
    }
  }
  // flush the warp caches
  __syncwarp();
  for (int i = lane; i < kCacheSlots; i += 32)
    if (wk[i] != SPB_EMPTY_KEY) sink.add(wk[i], wc[i], wf[i]);
  // usable-site count: warp reduce, one atomic per CTA
  for (int o = 16; o > 0; o >>= 1) my_usable += __shfl_xor_sync(0xFFFFFFFFu, my_usable, o);
  if (lane == 0 && my_usable) atomicAdd(&s_usable, my_usable);
  __syncthreads();
  if (tid == 0 && usable && s_usable) atomicAdd(usable, (unsigned long long)s_usable);
}

template <class Sink>
int launch_count(const uint32_t* d_sm, const uint32_t* d_valid, int n, int64_t site_begin, int64_t site_end, Sink sink,
                 uint64_t* d_usable, cudaStream_t st) {
  if (site_end <= site_begin) return SPB_OK;
  size_t smem = (size_t)kWarps * kCacheSlots * 20 + ((size_t)(kTileSites / 32) * 2 * n + 4) * 4;
  SPB_CUDA(cudaFuncSetAttribute(count_kernel<Sink>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int occ = 1;
  SPB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, count_kernel<Sink>, kThreads, smem));
  if (occ < 1) occ = 1;
  int64_t tile_begin = site_begin / kTileSites, tile_end = (site_end + kTileSites - 1) / kTileSites;
  int64_t tiles = tile_end - tile_begin;
  int64_t grid = (int64_t)sm_count() * occ;
  if (grid > tiles) grid = tiles;
  // the caller's buffers are sized by spb_sm_words / spb_plane_words for the whole alignment; the
  // kernel only needs an upper bound that is safe to read: everything up to the last tile's end
  // that lies inside the allocation.  We pass the *allocation-independent* bound derived from
  // site_end, which is always inside the allocation.
  int64_t sm_words = ((site_end + 31) / 32) * 2 * (int64_t)n;
  sm_words = (sm_words + 3) / 4 * 4;
  int64_t valid_words = (site_end + 31) / 32;
  count_kernel<Sink><<<(unsigned)grid, kThreads, smem, st>>>(d_sm, sm_words, d_valid, valid_words, n, site_begin, site_end,
                                                             tile_begin, tile_end, sink, (unsigned long long*)d_usable);
  SPB_LAUNCH_CHECK();
  return SPB_OK;
}

// ------------------------------------------------------------------------------------------
// Round-2 counting kernel ("stream" kernel, used whenever first-site indices are not requested).
//
// ncu on the cache kernel above (12 taxa x 10^8 sites): DRAM 2.6 %, issue slots 21 %, top stall = short scoreboard --
// a per-site chain of dependent shared-memory round trips (tile word -> key -> cache tag -> counter) plus shared-memory
// atomics at 2 clk per lane (B300_MICROARCH: ATOMS spread-address), i.e. SLOWER than fire-and-forget global reductions
// (REDG: 1.29 clk per lane) into a table that the 126 MB L2 holds entirely (4^12 x 4 B = 64 MB).  So this kernel has no
// shared memory at all:
//   * a lane owns 16 CONSECUTIVE sites = NT 32-bit words of the bit stream (NT = taxa, compile-time), read with
//     128-bit loads; all 16 keys are extracted with compile-time shifts (2 ALU ops each) -- 16 independent chains;
//   * the constant patterns (AAAA.., CCCC.., GGGG.., TTTT..: 34 % of the sites of a 12-taxon JC tree with branch
//     length 0.05) never leave the registers: key == (key & 3) * 0x5555.. adds 1 << 8c to a packed 4 x 8-bit counter;
//   * every other usable site is ONE predicated RED.ADD (direct table) or one hash insert (open addressing).
// Floors: REDG issue 1.29 clk per lane and SM -> 0.66 x 1.29 = 0.85 clk per site = 1.17 sites / clk / SM = 3.4e11 sites/s
// = 1.0 TB/s of packed input at 12 taxa (16 % of the HBM copy peak) when only the constant patterns are aggregated.
struct StreamDirectSink {  // no first-site tracking: one RED per update, nothing else
  uint32_t* table;
  __device__ __forceinline__ void add(uint64_t key, uint32_t c, uint32_t) const { atomicAdd(table + key, c); }
  // (ptxas lowers a conditional RED to BSSY / BRA / RED / BSYNC even when it is written as `@p red` in PTX; the extra
  // three instructions per site do not matter: the kernel is bound by the RED rate, not by issue slots)
  __device__ __forceinline__ void add_if(bool p, uint64_t key) const { if (p) atomicAdd(table + key, 1u); }
};

struct StreamHashSink {
  unsigned long long* keys;
  uint32_t* counts;
  uint64_t mask;
  uint32_t* overflow;
  __device__ __forceinline__ void add(uint64_t key, uint32_t c, uint32_t) const {
    uint64_t h = mix64(key) & mask;
    for (uint64_t probe = 0; probe <= mask; ++probe) {
      unsigned long long k = keys[h];
      if (k == SPB_EMPTY_KEY) {
        const unsigned long long old = atomicCAS(keys + h, (unsigned long long)SPB_EMPTY_KEY, (unsigned long long)key);
        k = (old == SPB_EMPTY_KEY) ? key : old;
      }
      if (k == key) { atomicAdd(counts + h, c); return; }
      h = (h + 1) & mask;
    }
    atomicExch(overflow, 1u);
  }
  __device__ __forceinline__ void add_if(bool p, uint64_t key) const { if (p) add(key, 1u, 0u); }
};

template <int NT, class Sink>
__global__ void __launch_bounds__(256) count_stream_kernel(const uint32_t* __restrict__ sm, const uint16_t* __restrict__ valid16,
                                                           int64_t chunk_begin, int64_t chunk_end, int64_t site_begin,
                                                           int64_t site_end, Sink sink, unsigned long long* usable) {
  constexpr int BITS = 2 * NT;
  constexpr uint64_t MASK = (BITS == 64) ? ~0ull : ((1ull << BITS) - 1ull);
  constexpr uint64_t ONES = 0x5555555555555555ull & MASK;
  uint32_t cst0 = 0, cst1 = 0, cst2 = 0, cst3 = 0, nus = 0;
  const int64_t stride = (int64_t)gridDim.x * 256;
  for (int64_t ch = chunk_begin + (int64_t)blockIdx.x * 256 + threadIdx.x; ch < chunk_end; ch += stride) {
    uint32_t w[NT + 2];
    const uint32_t* src = sm + ch * NT;
    if constexpr (NT % 4 == 0) {
#pragma unroll
      for (int v = 0; v < NT / 4; ++v) {
        const uint4 x = __ldg(reinterpret_cast<const uint4*>(src) + v);
        w[4 * v] = x.x; w[4 * v + 1] = x.y; w[4 * v + 2] = x.z; w[4 * v + 3] = x.w;
      }
    } else if constexpr (NT % 2 == 0) {
#pragma unroll
      for (int v = 0; v < NT / 2; ++v) {
        const uint2 x = __ldg(reinterpret_cast<const uint2*>(src) + v);
        w[2 * v] = x.x; w[2 * v + 1] = x.y;
      }
    } else {
#pragma unroll
      for (int v = 0; v < NT; ++v) w[v] = __ldg(src + v);
    }
    w[NT] = 0u; w[NT + 1] = 0u;
    uint32_t vb = __ldg(valid16 + ch);
    const int64_t s0 = ch * 16;
    if (s0 < site_begin || s0 + 16 > site_end) {  // boundary chunk of the requested site range
#pragma unroll
      for (int s = 0; s < 16; ++s)
        if (s0 + s < site_begin || s0 + s >= site_end) vb &= ~(1u << s);
    }
    nus += __popc(vb);
    uint32_t packed = 0u;
#pragma unroll
    for (int s = 0; s < 16; ++s) {
      const int o = s * BITS, wi = o >> 5, sh = o & 31;
      uint64_t key;
      if (sh + BITS <= 32) key = (uint64_t)(w[wi] >> sh);
      else if (sh + BITS <= 64) key = (uint64_t)__funnelshift_r(w[wi], w[wi + 1], sh) | ((uint64_t)(BITS > 32 ? (sh ? __funnelshift_r(w[wi + 1], w[wi + 2], sh) : w[wi + 1]) : 0u) << 32);
      else key = (uint64_t)__funnelshift_r(w[wi], w[wi + 1], sh) | ((uint64_t)__funnelshift_r(w[wi + 1], w[wi + 2], sh) << 32);
      key &= MASK;
      const bool ok = (vb >> s) & 1u;
      const uint32_t c = (uint32_t)key & 3u;
      const bool is_const = key == (uint64_t)c * ONES;
      if (ok && is_const) packed += 1u << (8 * c);
      sink.add_if(ok && !is_const, key);
    }
    cst0 += packed & 255u; cst1 += (packed >> 8) & 255u; cst2 += (packed >> 16) & 255u; cst3 += packed >> 24;
  }
  // constant patterns and the usable-site count: warp reduction, then one update per warp
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    cst0 += __shfl_xor_sync(0xFFFFFFFFu, cst0, o); cst1 += __shfl_xor_sync(0xFFFFFFFFu, cst1, o);
    cst2 += __shfl_xor_sync(0xFFFFFFFFu, cst2, o); cst3 += __shfl_xor_sync(0xFFFFFFFFu, cst3, o);
    nus += __shfl_xor_sync(0xFFFFFFFFu, nus, o);
  }
  if ((threadIdx.x & 31) == 0) {
    if (cst0) sink.add(0ull, cst0, 0xFFFFFFFFu);
    if (cst1) sink.add(ONES, cst1, 0xFFFFFFFFu);
    if (cst2) sink.add(2ull * ONES, cst2, 0xFFFFFFFFu);
    if (cst3) sink.add(3ull * ONES, cst3, 0xFFFFFFFFu);
    if (usable && nus) atomicAdd(usable, (unsigned long long)nus);
  }
}

template <int NT, class Sink>
int launch_stream_nt(const uint32_t* d_sm, const uint32_t* d_valid, int64_t site_begin, int64_t site_end, Sink sink,
                     uint64_t* d_usable, cudaStream_t st) {
  const int64_t chunk_begin = site_begin / 16, chunk_end = (site_end + 15) / 16;
  const int64_t chunks = chunk_end - chunk_begin;
  int64_t grid = (chunks + 255) / 256;
  const int64_t cap = (int64_t)sm_count() * 8;  // 8 resident CTAs of 256 threads per SM; grid-stride beyond that
  if (grid > cap) grid = cap;
  count_stream_kernel<NT, Sink><<<(unsigned)grid, 256, 0, st>>>(d_sm, reinterpret_cast<const uint16_t*>(d_valid), chunk_begin, chunk_end,
                                                               site_begin, site_end, sink, (unsigned long long*)d_usable);
  SPB_LAUNCH_CHECK();
  return SPB_OK;
}

template <class Sink>
int launch_stream(const uint32_t* d_sm, const uint32_t* d_valid, int n, int64_t site_begin, int64_t site_end, Sink sink,
                  uint64_t* d_usable, cudaStream_t st) {
  if (site_end <= site_begin) return SPB_OK;
#define SPB_NT(N_) case N_: return launch_stream_nt<N_, Sink>(d_sm, d_valid, site_begin, site_end, sink, d_usable, st);
  switch (n) {
    SPB_NT(1) SPB_NT(2) SPB_NT(3) SPB_NT(4) SPB_NT(5) SPB_NT(6) SPB_NT(7) SPB_NT(8) SPB_NT(9) SPB_NT(10) SPB_NT(11) SPB_NT(12)
    SPB_NT(13) SPB_NT(14)
    default: break;
  }
  if constexpr (!std::is_same<Sink, StreamDirectSink>::value) {  // the direct table stops at 14 taxa
    switch (n) {
      SPB_NT(15) SPB_NT(16) SPB_NT(17) SPB_NT(18) SPB_NT(19) SPB_NT(20) SPB_NT(21) SPB_NT(22) SPB_NT(23)
      SPB_NT(24) SPB_NT(25) SPB_NT(26) SPB_NT(27) SPB_NT(28) SPB_NT(29) SPB_NT(30) SPB_NT(31)
      default: break;
    }
  }
#undef SPB_NT
  set_error("count: bad taxon count %d", n);
  return SPB_ERR_ARG;
}

// ------------------------------------------------------------------------------------------
// "Classified" counting kernel (direct tables): the stream kernel above plus on-chip aggregation of the SINGLE-MUTATION
// patterns.  On a 12-taxon JC tree (branch length 0.05) 34 % of the sites are constant patterns, 37 % differ from a
// constant pattern in exactly one taxon (4 x 12 x 3 = 144 patterns) and 29 % are spread over ~10^5 rarer patterns.  The
// stream kernel sends 66 % of the sites to L2 as REDs, more than half of them to those 144 addresses, where they
// serialise in the L2 atomic units (measured: 3.4e10 RED/s).  Here
//   * c = majority of the three low digits; x = key ^ c * 0x5555..: x == 0 is a constant pattern (registers, as before);
//   * x with exactly one non-zero digit (position p, value y) is single-mutation class (c, p, y): it increments a
//     WARP-PRIVATE 32-bit counter in shared memory (fire-and-forget atomic); at the end of the kernel every warp issues one
//     RED per class;
//   * only the remaining sites (29 %) issue a RED, spread over ~10^5 addresses.
// ------------------------------------------------------------------------------------------
template <int NT>
__global__ void __launch_bounds__(256) count_class_kernel(const uint32_t* __restrict__ sm, const uint16_t* __restrict__ valid16,
                                                          int64_t chunk_begin, int64_t chunk_end, int64_t site_begin,
                                                          int64_t site_end, uint32_t* __restrict__ table, unsigned long long* usable) {
  constexpr int BITS = 2 * NT;
  constexpr uint32_t MASK = (BITS == 32) ? ~0u : ((1u << BITS) - 1u);
  constexpr uint32_t ONES = 0x55555555u & MASK;
  constexpr int NCLS = 12 * NT;                 // (c, p, y): 4 x NT x 3
  constexpr int NCLS_PAD = (NCLS + 31) / 32 * 32;
  // warp-private 32-bit class counters, updated with fire-and-forget shared-memory atomics.  (v1 kept lane-private byte
  // counters updated by load / add / store: no atomics, but the 16 updates of a chunk formed one dependent chain through
  // shared memory -- ncu: 56 % of the stall samples on the short scoreboard at 50 % occupancy, 1.12 ms per 10^8 sites.)
  __shared__ uint32_t hist_all[8 * NCLS_PAD];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint32_t* hist = hist_all + warp * NCLS_PAD;
  for (int i = lane; i < NCLS_PAD; i += 32) hist[i] = 0u;
  __syncwarp();
  uint32_t cst0 = 0, cst1 = 0, cst2 = 0, cst3 = 0, nus = 0;
  const int64_t stride = (int64_t)gridDim.x * 256;
  auto load_chunk = [&](uint32_t (&w)[NT + 2], uint32_t& vb, int64_t ch) {
    if (ch < chunk_end) {
      const uint32_t* src = sm + ch * NT;
      if constexpr (NT % 4 == 0) {
#pragma unroll
        for (int v = 0; v < NT / 4; ++v) {
          const uint4 x = __ldg(reinterpret_cast<const uint4*>(src) + v);
          w[4 * v] = x.x; w[4 * v + 1] = x.y; w[4 * v + 2] = x.z; w[4 * v + 3] = x.w;
        }
      } else if constexpr (NT % 2 == 0) {
#pragma unroll
        for (int v = 0; v < NT / 2; ++v) {
          const uint2 x = __ldg(reinterpret_cast<const uint2*>(src) + v);
          w[2 * v] = x.x; w[2 * v + 1] = x.y;
        }
      } else {
#pragma unroll
        for (int v = 0; v < NT; ++v) w[v] = __ldg(src + v);
      }
      vb = __ldg(valid16 + ch);
    } else {
#pragma unroll
      for (int v = 0; v < NT; ++v) w[v] = 0u;
      vb = 0u;
    }
    w[NT] = 0u; w[NT + 1] = 0u;
  };
  uint32_t wa[NT + 2], wb[NT + 2];
  uint32_t va, vbn;
  int64_t ch = chunk_begin + (int64_t)blockIdx.x * 256 + threadIdx.x;
  load_chunk(wa, va, ch);
  for (; ch < chunk_end; ch += stride) {
    load_chunk(wb, vbn, ch + stride);  // the next chunk is in flight while this one is classified
    uint32_t vb = va;
    const int64_t s0 = ch * 16;
    if (s0 < site_begin || s0 + 16 > site_end) {
#pragma unroll
      for (int s = 0; s < 16; ++s)
        if (s0 + s < site_begin || s0 + s >= site_end) vb &= ~(1u << s);
    }
    nus += __popc(vb);
    uint32_t packed = 0u;
#pragma unroll
    for (int s = 0; s < 16; ++s) {
      const int o = s * BITS, wi = o >> 5, sh = o & 31;
      uint32_t key = (sh + BITS <= 32) ? (wa[wi] >> sh) : __funnelshift_r(wa[wi], wa[wi + 1], sh);
      key &= MASK;
      const bool ok = (vb >> s) & 1u;
      const uint32_t d0 = key & 3u, d1 = (key >> 2) & 3u, d2 = (key >> 4) & 3u;
      const uint32_t c = (NT >= 3) ? ((d0 == d1) ? d0 : d2) : d0;
      const uint32_t x = key ^ (c * ONES);
      const int p = (31 - __clz(x | 1u)) >> 1;         // digit of the highest set bit: the mutated digit if there is exactly one
      const uint32_t y = x >> (2 * p);
      const bool single = x != 0u && (x & ~(3u << (2 * p))) == 0u;
      if (ok && x == 0u) packed += 1u << (8 * c);
      if (ok && single) atomicAdd(hist + (c * NT + p) * 3 + (y - 1), 1u);
      if (ok && x != 0u && !single) atomicAdd(table + key, 1u);
    }
    cst0 += packed & 255u; cst1 += (packed >> 8) & 255u; cst2 += (packed >> 16) & 255u; cst3 += packed >> 24;
#pragma unroll
    for (int v = 0; v < NT + 2; ++v) wa[v] = wb[v];
    va = vbn;
  }
  __syncwarp();
  for (int cls = lane; cls < NCLS; cls += 32) {
    const uint32_t v = hist[cls];
    if (v) {
      const int y = cls % 3 + 1, cp = cls / 3, p = cp % NT, c = cp / NT;
      atomicAdd(table + (((uint32_t)c * ONES) ^ ((uint32_t)y << (2 * p))), v);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    cst0 += __shfl_xor_sync(0xFFFFFFFFu, cst0, o); cst1 += __shfl_xor_sync(0xFFFFFFFFu, cst1, o);
    cst2 += __shfl_xor_sync(0xFFFFFFFFu, cst2, o); cst3 += __shfl_xor_sync(0xFFFFFFFFu, cst3, o);
    nus += __shfl_xor_sync(0xFFFFFFFFu, nus, o);
  }
  if (lane == 0) {
    if (cst0) atomicAdd(table, cst0);
    if (cst1) atomicAdd(table + ONES, cst1);
    if (cst2) atomicAdd(table + 2u * ONES, cst2);
    if (cst3) atomicAdd(table + 3u * ONES, cst3);
    if (usable && nus) atomicAdd(usable, (unsigned long long)nus);
  }
}

template <int NT>
int launch_class_nt(const uint32_t* d_sm, const uint32_t* d_valid, int64_t site_begin, int64_t site_end, uint32_t* d_table,
                    uint64_t* d_usable, cudaStream_t st) {
  const size_t smem = 0;
  int occ = 1;
  SPB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, count_class_kernel<NT>, 256, smem));
  if (occ < 1) occ = 1;
  const int64_t chunk_begin = site_begin / 16, chunk_end = (site_end + 15) / 16;
  int64_t grid = (chunk_end - chunk_begin + 255) / 256;
  const int64_t cap = (int64_t)sm_count() * occ;
  if (grid > cap) grid = cap;
  count_class_kernel<NT><<<(unsigned)grid, 256, smem, st>>>(d_sm, reinterpret_cast<const uint16_t*>(d_valid), chunk_begin, chunk_end,
                                                          site_begin, site_end, d_table, (unsigned long long*)d_usable);
  SPB_LAUNCH_CHECK();
  return SPB_OK;
}

int launch_class(const uint32_t* d_sm, const uint32_t* d_valid, int n, int64_t site_begin, int64_t site_end, uint32_t* d_table,
                 uint64_t* d_usable, cudaStream_t st) {
  if (site_end <= site_begin) return SPB_OK;
#define SPB_NT(N_) case N_: return launch_class_nt<N_>(d_sm, d_valid, site_begin, site_end, d_table, d_usable, st);
  switch (n) {
    SPB_NT(1) SPB_NT(2) SPB_NT(3) SPB_NT(4) SPB_NT(5) SPB_NT(6) SPB_NT(7) SPB_NT(8) SPB_NT(9) SPB_NT(10) SPB_NT(11) SPB_NT(12)
    SPB_NT(13) SPB_NT(14)
    default: break;
  }
#undef SPB_NT
  set_error("count: bad taxon count %d for the direct table", n);
  return SPB_ERR_ARG;
}

// Which kernel counts when first-site indices are not requested.  Measured on B200 (profiles/r2_count_kernels.txt, 10^8 sites):
// direct table, 12 taxa: cache kernel 1.47 ms, stream kernel 1.96 ms -- two thirds of the sites are ~260 single-mutation
// patterns, and fire-and-forget REDs to so few addresses serialise in the L2 atomic units (3.4e10 RED/s in total);
// hash table, 20 taxa: stream 3.39 ms, cache 3.59 ms; 31 taxa: 2.55 ms against 2.70 ms.  So: stream for hashed tables,
// the classified kernel (stream + on-chip single-mutation classes) for direct tables.  The cache kernel is the route when
// first-site indices are requested or the site stream is not 16-byte aligned.
enum CountKernel { kCountCache = 0, kCountStream = 1, kCountClass = 2 };
static CountKernel pick_count_kernel(const void* d_sm, const void* d_first, bool hashed) {
  if (d_first != nullptr || (reinterpret_cast<uintptr_t>(d_sm) & 15) != 0) return kCountCache;
  return hashed ? kCountStream : kCountClass;
}

// ------------------------------------------------------------------------------------------
// compaction (ordered stream compaction of non-empty cells): 3 phases, block = 4096 cells
// ------------------------------------------------------------------------------------------
constexpr int kCThreads = 1024;
constexpr int kCPer = 4;
constexpr int kCBlock = kCThreads * kCPer;

__device__ __forceinline__ uint32_t block_exclusive_scan(uint32_t v, uint32_t* total) {
  __shared__ uint32_t warp_sums[32];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
  uint32_t x = v;
  for (int o = 1; o < 32; o <<= 1) {
    uint32_t y = __shfl_up_sync(0xFFFFFFFFu, x, o);
    if (lane >= o) x += y;
  }
  __syncthreads();  // protect warp_sums reuse
  if (lane == 31) warp_sums[wid] = x;
  __syncthreads();
  if (wid == 0) {
    uint32_t s = (lane < nw) ? warp_sums[lane] : 0u;
    for (int o = 1; o < 32; o <<= 1) {
      uint32_t y = __shfl_up_sync(0xFFFFFFFFu, s, o);
      if (lane >= o) s += y;
    }
    warp_sums[lane] = s;
  }
  __syncthreads();
  uint32_t offset = (wid > 0) ? warp_sums[wid - 1] : 0u;
  if (total) *total = warp_sums[nw - 1];
  return offset + x - v;
}

struct DirectSrc {
  const uint32_t* table;
  __device__ __forceinline__ bool used(int64_t i) const { return table[i] != 0u; }
  __device__ __forceinline__ uint64_t key(int64_t i) const { return (uint64_t)i; }
  __device__ __forceinline__ uint32_t count(int64_t i) const { return table[i]; }
};
struct HashSrc {
  const uint64_t* keys;
  const uint32_t* counts;
  __device__ __forceinline__ bool used(int64_t i) const { return keys[i] != SPB_EMPTY_KEY; }
  __device__ __forceinline__ uint64_t key(int64_t i) const { return keys[i]; }
  __device__ __forceinline__ uint32_t count(int64_t i) const { return counts[i]; }
};
// flags array source (used by the reduced flattening rank computation)
struct FlagSrc {
  const uint32_t* flags;
  __device__ __forceinline__ bool used(int64_t i) const { return flags[i] != 0u; }
};

template <class Src>
__global__ void __launch_bounds__(kCThreads) compact_count_kernel(Src src, int64_t cells, uint32_t* tmp) {
  int64_t base = (int64_t)blockIdx.x * kCBlock + (int64_t)threadIdx.x * kCPer;
  uint32_t c = 0;
#pragma unroll
  for (int q = 0; q < kCPer; ++q) c += (base + q < cells && src.used(base + q)) ? 1u : 0u;
  uint32_t total;
  block_exclusive_scan(c, &total);
  if (threadIdx.x == 0) tmp[blockIdx.x] = total;
}

__global__ void __launch_bounds__(kCThreads) compact_scan_kernel(uint32_t* tmp, int64_t nblocks, unsigned long long* num) {
  __shared__ uint32_t carry_s;
  if (threadIdx.x == 0) carry_s = 0;
  __syncthreads();
  for (int64_t base = 0; base < nblocks; base += kCThreads) {
    int64_t i = base + threadIdx.x;
    uint32_t v = (i < nblocks) ? tmp[i] : 0u;
    uint32_t total;
    uint32_t ex = block_exclusive_scan(v, &total);
    uint32_t carry = carry_s;
    if (i < nblocks) tmp[i] = ex + carry;
    __syncthreads();
    if (threadIdx.x == 0) carry_s = carry + total;
    __syncthreads();
  }
  if (threadIdx.x == 0 && num) *num = carry_s;
}

template <class Src>
__global__ void __launch_bounds__(kCThreads) compact_write_kernel(Src src, const uint32_t* first, int64_t cells,
                                                                  const uint32_t* tmp, uint64_t* keys, uint32_t* counts,
                                                                  uint32_t* first_out, int64_t capacity) {
  int64_t base = (int64_t)blockIdx.x * kCBlock + (int64_t)threadIdx.x * kCPer;
  uint32_t c = 0;
  bool u[kCPer];
#pragma unroll
  for (int q = 0; q < kCPer; ++q) { u[q] = (base + q < cells) && src.used(base + q); c += u[q] ? 1u : 0u; }
  uint32_t ex = block_exclusive_scan(c, nullptr);
  int64_t o = (int64_t)tmp[blockIdx.x] + ex;
#pragma unroll
  for (int q = 0; q < kCPer; ++q) {
    if (u[q]) {
      if (o < capacity) {
        keys[o] = src.key(base + q);
        counts[o] = src.count(base + q);
        if (first_out) first_out[o] = first ? first[base + q] : 0u;
      }
      ++o;
    }
  }
}

// rank[i] = number of used cells before i (exclusive), rank[cells] = total
__global__ void __launch_bounds__(kCThreads) rank_write_kernel(const uint32_t* flags, int64_t cells, const uint32_t* tmp,
                                                               uint32_t* rank) {
  int64_t base = (int64_t)blockIdx.x * kCBlock + (int64_t)threadIdx.x * kCPer;
  uint32_t c = 0;
  bool u[kCPer];
#pragma unroll
  for (int q = 0; q < kCPer; ++q) { u[q] = (base + q < cells) && flags[base + q] != 0u; c += u[q] ? 1u : 0u; }
  uint32_t ex = block_exclusive_scan(c, nullptr);
  uint32_t o = tmp[blockIdx.x] + ex;
#pragma unroll
  for (int q = 0; q < kCPer; ++q) {
    if (base + q < cells) rank[base + q] = o;
    if (u[q]) ++o;
  }
}

// table[keys[i]] += counts[i]: merges (key, count) lists of other ranks into a direct-indexed table
__global__ void direct_merge_kernel(const uint64_t* __restrict__ keys, const uint32_t* __restrict__ counts, int64_t num,
                                    uint32_t* __restrict__ table) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < num) atomicAdd(table + keys[i], counts[i]);
}

__global__ void hash_merge_kernel(const uint64_t* keys, const uint32_t* counts, const uint32_t* first, int64_t num,
                                  HashSink sink) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < num) sink.add(keys[i], counts[i], first ? first[i] : 0xFFFFFFFFu);
}

template <class Src>
int run_compact(Src src, const uint32_t* first, int64_t cells, uint64_t* d_keys, uint32_t* d_counts, uint32_t* d_first_out,
                int64_t capacity, uint64_t* d_num, uint32_t* d_tmp, cudaStream_t st) {
  int64_t nb = (cells + kCBlock - 1) / kCBlock;
  if (nb == 0) { SPB_CUDA(cudaMemsetAsync(d_num, 0, 8, st)); return SPB_OK; }
  compact_count_kernel<Src><<<(unsigned)nb, kCThreads, 0, st>>>(src, cells, d_tmp);
  SPB_LAUNCH_CHECK();
  compact_scan_kernel<<<1, kCThreads, 0, st>>>(d_tmp, nb, (unsigned long long*)d_num);
  SPB_LAUNCH_CHECK();
  compact_write_kernel<Src><<<(unsigned)nb, kCThreads, 0, st>>>(src, first, cells, d_tmp, d_keys, d_counts, d_first_out, capacity);
  SPB_LAUNCH_CHECK();
  return SPB_OK;
}

}  // namespace

namespace spb {
// used by flatten.cu (reduced format): exclusive rank of the set flags; total to rank[cells]
int rank_flags(const uint32_t* d_flags, int64_t cells, uint32_t* d_rank, uint32_t* d_tmp, cudaStream_t st) {
  int64_t nb = (cells + kCBlock - 1) / kCBlock;
  FlagSrc src{d_flags};
  compact_count_kernel<FlagSrc><<<(unsigned)nb, kCThreads, 0, st>>>(src, cells, d_tmp);
  SPB_LAUNCH_CHECK();
  compact_scan_kernel<<<1, kCThreads, 0, st>>>(d_tmp, nb, (unsigned long long*)nullptr);
  SPB_LAUNCH_CHECK();
  rank_write_kernel<<<(unsigned)nb, kCThreads, 0, st>>>(d_flags, cells, d_tmp, d_rank);
  SPB_LAUNCH_CHECK();
  return SPB_OK;
}
}  // namespace spb

extern "C" int64_t spb_compact_tmp_words(int64_t cells) { return (cells + kCBlock - 1) / kCBlock + 8; }

extern "C" int spb_count_direct(const uint32_t* d_sm, const uint32_t* d_valid, int n_taxa, int64_t site_begin,
                                int64_t site_end, uint32_t* d_table, uint32_t* d_first, uint64_t* d_usable, void* stream) {
  SPB_REQUIRE(d_sm && d_valid && d_table, "spb_count_direct: NULL buffer");
  SPB_REQUIRE(n_taxa >= 1 && n_taxa <= 14, "spb_count_direct: direct table needs 1 <= n_taxa <= 14 (got %d)", n_taxa);
  SPB_REQUIRE(site_begin >= 0 && site_end >= site_begin && site_end < (1ll << 32), "spb_count_direct: bad site range");
  DirectSink sink{d_table, d_first};
  const CountKernel which = pick_count_kernel(d_sm, d_first, false);
  if (which == kCountClass) return launch_class(d_sm, d_valid, n_taxa, site_begin, site_end, d_table, d_usable, (cudaStream_t)stream);
  if (which == kCountStream)
    return launch_stream(d_sm, d_valid, n_taxa, site_begin, site_end, StreamDirectSink{d_table}, d_usable, (cudaStream_t)stream);
  return launch_count(d_sm, d_valid, n_taxa, site_begin, site_end, sink, d_usable, (cudaStream_t)stream);
}

extern "C" int spb_count_hash(const uint32_t* d_sm, const uint32_t* d_valid, int n_taxa, int64_t site_begin,
                              int64_t site_end, uint64_t* d_hkeys, uint32_t* d_hcounts, uint32_t* d_hfirst, int64_t cap,
                              uint64_t* d_usable, uint32_t* d_overflow, void* stream) {
  SPB_REQUIRE(d_sm && d_valid && d_hkeys && d_hcounts && d_overflow, "spb_count_hash: NULL buffer");
  SPB_REQUIRE(n_taxa >= 1 && n_taxa <= 31, "spb_count_hash: uint64 keys need n_taxa <= 31 (got %d)", n_taxa);
  SPB_REQUIRE(cap >= 2 && (cap & (cap - 1)) == 0, "spb_count_hash: capacity must be a power of two");
  SPB_REQUIRE(site_begin >= 0 && site_end >= site_begin && site_end < (1ll << 32), "spb_count_hash: bad site range");
  HashSink sink{(unsigned long long*)d_hkeys, d_hcounts, d_hfirst, (uint64_t)cap - 1, d_overflow};
  if (pick_count_kernel(d_sm, d_hfirst, true) == kCountStream)
    return launch_stream(d_sm, d_valid, n_taxa, site_begin, site_end,
                         StreamHashSink{(unsigned long long*)d_hkeys, d_hcounts, (uint64_t)cap - 1, d_overflow}, d_usable, (cudaStream_t)stream);
  return launch_count(d_sm, d_valid, n_taxa, site_begin, site_end, sink, d_usable, (cudaStream_t)stream);
}

extern "C" int spb_compact_direct(const uint32_t* d_table, const uint32_t* d_first, int64_t cells, uint64_t* d_keys,
                                  uint32_t* d_counts, uint32_t* d_first_out, int64_t capacity, uint64_t* d_num,
                                  uint32_t* d_tmp, void* stream) {
  SPB_REQUIRE(d_table && d_keys && d_counts && d_num && d_tmp && cells >= 0, "spb_compact_direct: bad arguments");
  return run_compact(DirectSrc{d_table}, d_first, cells, d_keys, d_counts, d_first_out, capacity, d_num, d_tmp,
                     (cudaStream_t)stream);
}

extern "C" int spb_compact_hash(const uint64_t* d_hkeys, const uint32_t* d_hcounts, const uint32_t* d_hfirst, int64_t cap,
                                uint64_t* d_keys, uint32_t* d_counts, uint32_t* d_first_out, int64_t capacity,
                                uint64_t* d_num, uint32_t* d_tmp, void* stream) {
  SPB_REQUIRE(d_hkeys && d_hcounts && d_keys && d_counts && d_num && d_tmp && cap >= 0, "spb_compact_hash: bad arguments");
  return run_compact(HashSrc{d_hkeys, d_hcounts}, d_hfirst, cap, d_keys, d_counts, d_first_out, capacity, d_num, d_tmp,
                     (cudaStream_t)stream);
}

extern "C" int spb_direct_merge(const uint64_t* d_keys, const uint32_t* d_counts, int64_t num, int64_t cells, uint32_t* d_table,
                                void* stream) {
  SPB_REQUIRE(d_table && cells >= 1, "spb_direct_merge: bad table");
  if (num <= 0) return SPB_OK;
  SPB_REQUIRE(d_keys && d_counts, "spb_direct_merge: NULL buffer");
  (void)cells;  // keys come from spb_compact_direct of a table of the same size: always in range
  direct_merge_kernel<<<(unsigned)((num + 255) / 256), 256, 0, (cudaStream_t)stream>>>(d_keys, d_counts, num, d_table);
  SPB_LAUNCH_CHECK();
  return SPB_OK;
}

extern "C" int spb_hash_merge(const uint64_t* d_keys, const uint32_t* d_counts, const uint32_t* d_first, int64_t num,
                              uint64_t* d_hkeys, uint32_t* d_hcounts, uint32_t* d_hfirst, int64_t cap,
                              uint32_t* d_overflow, void* stream) {
  SPB_REQUIRE(d_keys && d_counts && d_hkeys && d_hcounts && d_overflow, "spb_hash_merge: NULL buffer");
  SPB_REQUIRE(cap >= 2 && (cap & (cap - 1)) == 0, "spb_hash_merge: capacity must be a power of two");
  if (num <= 0) return SPB_OK;
  HashSink sink{(unsigned long long*)d_hkeys, d_hcounts, d_hfirst, (uint64_t)cap - 1, d_overflow};
  hash_merge_kernel<<<(unsigned)((num + 255) / 256), 256, 0, (cudaStream_t)stream>>>(d_keys, d_counts, d_first, num, sink);
  SPB_LAUNCH_CHECK();
  return SPB_OK;
}

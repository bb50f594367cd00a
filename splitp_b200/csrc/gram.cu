// Kernel 4: exact integer Gram contraction G = S0 * S0^T of a u8 matrix on the 5th-generation tensor cores.
//
// Why u8: a flattening built from site-pattern COUNTS is an integer matrix, so F F^T is an integer matrix.
// The split score (splitp/phylogenetics.py:293-300) is 1 - top4/total, a difference of nearly equal numbers
// for a true split, and SURVEY.md 7.3 shows that any fp32-accumulated Gram misses the tolerance.  We split
// F = S0 + H with S0 = low byte of every count (dense, u8) and H = the few counts >= 256 (sparse triplets):
//     F F^T = S0 S0^T + S0 H^T + H S0^T + H H^T.
// S0 S0^T runs on tcgen05.mma kind::i8 (u8 x u8 -> s32 in TMEM, exact: 255^2 * K < 2^31 for K <= 33025 per
// accumulation, enforced through the split-K chunk size) and the three sparse terms are added by
// spb_gram_hi_correction with integer-valued fp64 atomics (exact below 2^53).
//
// Operand layout ("tiled"): S0 is stored as [rows_pad/128][pitch/128] tiles of 128 rows x 128 bytes, each tile
// 16 KB contiguous in the K-major SWIZZLE_128B canonical layout of the UMMA shared-memory descriptor
//     offset(r, k) = r*128 + (((k >> 4) ^ (r & 7)) << 4) + (k & 15).
// The flattening scatter (spb_flatten_u8, layout = SPB_S0_TILED) writes this layout directly, so a whole operand
// tile is ONE 1-D bulk-TMA copy (cp.async.bulk, 16 KB) completing on an mbarrier: no tensor map, no swizzle
// work on the load path, perfectly coalesced HBM/L2 reads.
//
// Kernel structure (persistent, one CTA per SM, 320 threads):
//   warp 0   : TMA producer   (bulk copies into a 4-stage shared-memory ring)
//   warp 1   : MMA issuer     (tcgen05.mma M=128, N=BN, K=32 x 4 per stage; accumulators in TMEM, 2 stages)
//   warps 2-9: epilogue       (tcgen05.ld -> fp64 stores incl. the mirrored half, or 64-bit integer atomics
//                              when K is split across CTAs)
// Only tiles touching the upper triangle (in 256-wide blocks) are computed; the rest is mirrored.
#include "common.cuh"
#include "ptx.cuh"

using namespace spb;

namespace {

constexpr int kTile = 128;               // rows and K-bytes per operand tile
constexpr int kTileBytes = kTile * kTile;  // 16 KB
constexpr int kStages = 4;
constexpr int kUmmaThreads = 320;  // TMA warp + MMA warp + 8 epilogue warps

// mbarrier / bulk-copy wrappers: ptx.cuh
__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(cols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// D[tmem] (+)= A[smem] * B[smem]^T, u8 x u8 -> s32
__device__ __forceinline__ void umma_i8(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
        "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]),
        "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]),
        "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// K-major, SWIZZLE_128B shared-memory matrix descriptor (sm_100 "version 1"): rows are 128 B apart, 8-row groups
// 1024 B apart (SBO); LBO is unused for swizzled K-major operands.
__device__ __forceinline__ uint64_t make_desc_sw128(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);  // start address, bits [0,14)
  d |= (uint64_t)1 << 16;                     // leading byte offset (ignored), bits [16,30)
  d |= (uint64_t)(1024 >> 4) << 32;           // stride byte offset, bits [32,46)
  d |= (uint64_t)1 << 46;                     // descriptor version (Blackwell)
  d |= (uint64_t)2 << 61;                     // layout type: SWIZZLE_128B
  return d;
}

// instruction descriptor, kind::i8: D = s32, A = B = u8, both K-major, dense
__host__ __device__ constexpr uint32_t make_idesc_i8(int M, int N) {
  return (2u << 4) | (0u << 7) | (0u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// K tiles of matrix b: all KT of the allocation pitch, or (ncols != NULL) the tiles holding its ncols[b] occupied columns (the
// columns beyond them are zero).  At least one tile, so every work item issues an MMA and writes its accumulator.
__device__ __forceinline__ int k_tiles(const int32_t* ncols, int b, int KT) {
  if (!ncols) return KT;
  const int t = (ncols[b] + kTile - 1) / kTile;
  return t < 1 ? 1 : (t > KT ? KT : t);
}

// ---------------------------------------------------------------------------------------------------
// work decomposition shared by all roles.  Tiles: row tile i (128 rows) x column tile j (BN columns), computed
// only if the tile's 256-block column index >= its 256-block row index.  Work item = (tile, k-split).
// ---------------------------------------------------------------------------------------------------
struct Work {
  int b, i, j, ks;  // batch entry, row tile, column tile, k-split
};

template <int BN>
__device__ __forceinline__ bool tile_needed(int i, int j) {
  // 256-granular block indices of the tile's first row and LAST column
  int rb = (i * kTile) >> 8;
  int cb = (j * BN + BN - 1) >> 8;
  return cb >= rb;
}

template <int BN>
__device__ __forceinline__ bool get_work(int w, int T, int TN, int tiles, int ksplit, Work* out) {
  const int per = tiles * ksplit;
  out->b = w / per;
  w -= out->b * per;
  int tile = w / ksplit;
  int ks = w - tile * ksplit;
  int seen = 0;
  for (int i = 0; i < T; ++i) {
    for (int j = 0; j < TN; ++j) {
      if (!tile_needed<BN>(i, j)) continue;
      if (seen == tile) { out->i = i; out->j = j; out->ks = ks; return true; }
      ++seen;
    }
  }
  return false;
}

// K-tile range [kt0, kt1) of a work item; false when it is empty (a K split of a matrix with fewer occupied tiles than the
// split has parts: the work item is skipped by all three roles alike).  With column counts every matrix splits its own K tiles
// into ksplit equal parts (at most kt_per_split each, as the host planned them for the full pitch).
__device__ __forceinline__ bool k_range(const int32_t* ncols, const Work& wk, int KT, int ksplit, int kt_per_split, int* kt0, int* kt1) {
  const int kb = k_tiles(ncols, wk.b, KT);
  const int per = ncols ? (kb + ksplit - 1) / ksplit : kt_per_split;
  *kt0 = wk.ks * per;
  *kt1 = min(kb, *kt0 + per);
  return *kt0 < *kt1;
}

template <int BN>
int count_tiles(int T, int TN) {
  int c = 0;
  for (int i = 0; i < T; ++i)
    for (int j = 0; j < TN; ++j) {
      int rb = (i * kTile) >> 8, cb = (j * BN + BN - 1) >> 8;
      if (cb >= rb) ++c;
    }
  return c;
}

// ---------------------------------------------------------------------------------------------------
// the tensor-core kernel
// ---------------------------------------------------------------------------------------------------
template <int BN>
__global__ void __launch_bounds__(kUmmaThreads, 1)
gram_u8_umma_kernel(const uint8_t* __restrict__ s0_base, int64_t s0_stride, int T, int KT, int tiles, int ksplit, int kt_per_split,
                    const int32_t* __restrict__ ncols, int num_work, int64_t ldg, double* __restrict__ G_base, int64_t g_stride,
                    unsigned long long* __restrict__ acc_base) {
  constexpr int kStageBytes = kTileBytes + BN * kTile;  // A tile + B tile(s)
  constexpr uint32_t kTmemCols = 2 * BN;                 // two accumulator stages (power of two >= 32)
  constexpr uint32_t kIdesc = make_idesc_i8(kTile, BN);
  extern __shared__ __align__(1024) uint8_t smem[];
  // carve-up: [stages][A | B] then barriers
  // SWIZZLE_128B operands need 1024-byte aligned tiles: align the ring by hand (the launch adds 1 KB of slack)
  uint8_t* ring = smem + ((1024u - (smem_u32(smem) & 1023u)) & 1023u);
  uint64_t* bars = reinterpret_cast<uint64_t*>(ring + (size_t)kStages * kStageBytes);
  uint64_t* full_bar = bars;                  // [kStages]
  uint64_t* empty_bar = bars + kStages;       // [kStages]
  uint64_t* tfull_bar = bars + 2 * kStages;   // [2]
  uint64_t* tempty_bar = bars + 2 * kStages + 2;  // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kStages + 4);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int TN = (T * kTile) / BN;

  if (warp == 0 && lane == 0) {
    for (int s = 0; s < kStages; ++s) { mbar_init(smem_u32(full_bar + s), 1); mbar_init(smem_u32(empty_bar + s), 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(smem_u32(tfull_bar + s), 1); mbar_init(smem_u32(tempty_bar + s), 8); }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(smem_u32(tmem_slot), kTmemCols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===== TMA producer =====
    if (lane == 0) {
      uint32_t stage = 0, phase = 0;
      for (int w = blockIdx.x; w < num_work; w += gridDim.x) {
        Work wk;
        if (!get_work<BN>(w, T, TN, tiles, ksplit, &wk)) break;
        int kt0, kt1;
        if (!k_range(ncols, wk, KT, ksplit, kt_per_split, &kt0, &kt1)) continue;
        const uint8_t* s0t = s0_base + (size_t)wk.b * s0_stride;
        for (int kt = kt0; kt < kt1; ++kt) {
          mbar_wait(smem_u32(empty_bar + stage), phase ^ 1);
          const uint32_t fb = smem_u32(full_bar + stage);
          mbar_expect_tx(fb, (uint32_t)kStageBytes);
          uint8_t* sa = ring + (size_t)stage * kStageBytes;
          bulk_g2s(smem_u32(sa), s0t + ((size_t)wk.i * KT + kt) * kTileBytes, kTileBytes, fb);
#pragma unroll
          for (int h = 0; h < BN / kTile; ++h) {
            const int rt = wk.j * (BN / kTile) + h;
            bulk_g2s(smem_u32(sa + kTileBytes + h * kTileBytes), s0t + ((size_t)rt * KT + kt) * kTileBytes, kTileBytes, fb);
          }
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer (one thread) =====
    if (lane == 0) {
      uint32_t stage = 0, phase = 0;
      uint32_t acc = 0, acc_phase = 0;
      for (int w = blockIdx.x; w < num_work; w += gridDim.x) {
        Work wk;
        if (!get_work<BN>(w, T, TN, tiles, ksplit, &wk)) break;
        int kt0, kt1;
        if (!k_range(ncols, wk, KT, ksplit, kt_per_split, &kt0, &kt1)) continue;
        mbar_wait(smem_u32(tempty_bar + acc), acc_phase ^ 1);  // epilogue has drained this accumulator
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * BN;
        for (int kt = kt0; kt < kt1; ++kt) {
          mbar_wait(smem_u32(full_bar + stage), phase);
          tc_fence_after();
          const uint32_t sa = smem_u32(ring + (size_t)stage * kStageBytes);
          const uint64_t da = make_desc_sw128(sa);
          const uint64_t db = make_desc_sw128(sa + kTileBytes);
#pragma unroll
          for (int k = 0; k < kTile / 32; ++k) {
            // advance 32 bytes along K inside the 128-byte swizzle row: +2 in the (addr >> 4) field
            umma_i8(d_tmem, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), kIdesc, (kt > kt0 || k > 0) ? 1u : 0u);
          }
          umma_commit(smem_u32(empty_bar + stage));  // frees the smem slot once the MMAs have read it
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
        umma_commit(smem_u32(tfull_bar + acc));  // accumulator complete -> epilogue
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
    }
  } else {
    // ===== epilogue: 8 warps; warp q = warp % 4 may only touch TMEM lanes [32q, 32q+32), so two warps share each
    // lane quarter and split the BN accumulator columns between them (half = 0 / 1) =====
    const int q = warp & 3;
    const int half = (warp - 2) >> 2;
    uint32_t acc = 0, acc_phase = 0;
    for (int w = blockIdx.x; w < num_work; w += gridDim.x) {
      Work wk;
      if (!get_work<BN>(w, T, TN, tiles, ksplit, &wk)) break;
      int kt0, kt1;
      if (!k_range(ncols, wk, KT, ksplit, kt_per_split, &kt0, &kt1)) continue;
      mbar_wait(smem_u32(tfull_bar + acc), acc_phase);
      tc_fence_after();
      const int row = wk.i * kTile + q * 32 + lane;
      const int rb = row >> 8;
      double* G = G_base + (size_t)wk.b * g_stride;
      unsigned long long* acc64 = acc_base ? acc_base + (size_t)wk.b * ldg * ldg : nullptr;
#pragma unroll 1
      for (int c0 = half * (BN / 2); c0 < (half + 1) * (BN / 2); c0 += 32) {
        uint32_t v[32];
        tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + acc * BN + c0, v);
        const int col0 = wk.j * BN + c0;
        if (acc64) {
          // split-K: exact 64-bit integer accumulation; the finalize kernel converts and mirrors
          unsigned long long* dst = acc64 + (size_t)row * ldg + col0;
#pragma unroll
          for (int e = 0; e < 32; ++e)
            if (v[e]) atomicAdd(dst + e, (unsigned long long)v[e]);
        } else {
          double* dst = G + (size_t)row * ldg + col0;
#pragma unroll
          for (int e = 0; e < 32; e += 2) {
            double2 d2 = make_double2((double)(int)v[e], (double)(int)v[e + 1]);
            *reinterpret_cast<double2*>(dst + e) = d2;
          }
          if ((col0 >> 8) > rb) {  // mirrored half: lanes walk consecutive rows => coalesced
#pragma unroll
            for (int e = 0; e < 32; ++e) G[(size_t)(col0 + e) * ldg + row] = (double)(int)v[e];
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(tempty_bar + acc));
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    tmem_dealloc(tmem_base, kTmemCols);
  }
}

// ---------------------------------------------------------------------------------------------------
// CTA-pair kernel (tcgen05 cta_group::2): the version used whenever K needs no split.
//
// Why: ncu on the single-CTA kernel above (round 1, 4096^2 Gram): tensor pipe 45.8 % active while the operand feed
// ran at l1tex__m_xbar2l1tex_read_bytes = 11.5 TB/s, the L2 -> SM ceiling of the part (B300_MICROARCH: ~6300 B/clk
// chip-wide).  A single CTA pulls 48 KB (A tile + two B tiles) per four M128 N256 K32 MMAs = 85 MAC / byte; at the
// kind::i8 rate of 128 clk per MMA (scripts/mma_rate.cu) all 148 SMs would need 14.2 KB/clk.  A CTA pair computes a
// 256 x 256 output block with ONE M256 N256 K32 instruction per 32 bytes of K: every CTA loads its own 128 rows of A and
// only ITS HALF of B (128 of the 256 columns), 32 KB per stage = 128 MAC / byte, 1.5x less L2 traffic per MMA, and the
// 16 KB saved per stage buy a 6-stage ring instead of 4.
//
// Roles per CTA (320 threads, both CTAs of the pair run the same code):
//   warp 0    : TMA producer for THIS CTA's shared memory (A tile of rows 256 bi + 128 rank .., B tile 2 bj + rank)
//   warp 1    : rank 0 = MMA issuer for the pair (one thread; tcgen05.mma.cta_group::2, commits multicast to both CTAs);
//               rank 1 = relay: forwards "my stage s is full" to the leader's peer_full barrier (plain bulk copies
//               can only signal a barrier of their own CTA, and the MMA reads both CTAs' shared memory)
//   warps 2-9 : epilogue of THIS CTA's 128 accumulator rows (TMEM is per CTA): tcgen05.ld -> int32 / fp64 stores of
//               the block and of its mirror image; accumulator release goes to the leader's tempty barrier
// Work item = (matrix, block row bi, block column bj >= bi) in 256-row blocks, dealt round-robin to the pairs.
// ---------------------------------------------------------------------------------------------------
constexpr int kStages2 = 6;
constexpr int kStage2Bytes = 2 * kTileBytes;  // this CTA's A tile + its half of B

__device__ __forceinline__ void tmem_alloc2(uint32_t dst_smem, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(cols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc2(uint32_t taddr, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
// arrives (once the MMAs issued so far have completed) on the barrier at this offset in BOTH CTAs of the pair
__device__ __forceinline__ void umma_commit2(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
               "h"((uint16_t)3)
               : "memory");
}
__device__ __forceinline__ void umma_i8_2(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::i8 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void st_global_v8(int32_t* p, const uint32_t* v) {
  asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]),
               "r"(v[5]), "r"(v[6]), "r"(v[7])
               : "memory");
}

struct Work2 {
  int b, bi, bj;
};
// w -> (matrix, block row, block column): row-major over the upper triangle, row bi holds the blocks bj = bi .. B - 1
__device__ __forceinline__ void get_work2(int w, int B, int nblk, Work2* out) {
  out->b = w / nblk;
  int t = w - out->b * nblk;
  int bi = 0;
  while (t >= B - bi) { t -= B - bi; ++bi; }
  out->bi = bi;
  out->bj = bi + t;
}

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kUmmaThreads, 1)
gram_u8_umma2_kernel(const uint8_t* __restrict__ s0_base, int64_t s0_stride, int B, int KT, const int32_t* __restrict__ ncols, int nblk,
                     int num_work, int64_t ldg, double* __restrict__ G_base, int64_t g_stride, int32_t* __restrict__ Gi_base) {
  constexpr uint32_t kIdesc = make_idesc_i8(256, 256);
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* ring = smem + ((1024u - (smem_u32(smem) & 1023u)) & 1023u);  // same offset in both CTAs (same kernel, same layout)
  uint64_t* bars = reinterpret_cast<uint64_t*>(ring + (size_t)kStages2 * kStage2Bytes);
  uint64_t* full_bar = bars;                         // [kStages2] this CTA's stage has landed
  uint64_t* empty_bar = bars + kStages2;             // [kStages2] the pair's MMAs have read the stage (multicast commit)
  uint64_t* peer_full_bar = bars + 2 * kStages2;     // [kStages2] leader only: the peer's stage has landed (relay)
  uint64_t* tfull_bar = bars + 3 * kStages2;         // [2] accumulator complete (multicast commit)
  uint64_t* tempty_bar = bars + 3 * kStages2 + 2;    // [2] leader only: both CTAs' epilogues have drained the accumulator
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 3 * kStages2 + 4);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;

  if (warp == 0 && lane == 0) {
    for (int s = 0; s < kStages2; ++s) {
      mbar_init(smem_u32(full_bar + s), 1);
      mbar_init(smem_u32(empty_bar + s), 1);
      mbar_init(smem_u32(peer_full_bar + s), 1);
    }
    for (int s = 0; s < 2; ++s) { mbar_init(smem_u32(tfull_bar + s), 1); mbar_init(smem_u32(tempty_bar + s), 16); }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc2(smem_u32(tmem_slot), 512);
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();  // barriers of BOTH CTAs are initialised before anyone arrives remotely
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===== TMA producer (each CTA feeds its own shared memory) =====
    if (lane == 0) {
      uint32_t stage = 0, phase = 0;
      for (int w = pair; w < num_work; w += npairs) {
        Work2 wk;
        get_work2(w, B, nblk, &wk);
        const uint8_t* s0t = s0_base + (size_t)wk.b * s0_stride;
        const uint8_t* a_src = s0t + (size_t)(2 * wk.bi + (int)rank) * KT * kTileBytes;
        const uint8_t* b_src = s0t + (size_t)(2 * wk.bj + (int)rank) * KT * kTileBytes;
        const int kb = k_tiles(ncols, wk.b, KT);
        for (int kt = 0; kt < kb; ++kt) {
          mbar_wait(smem_u32(empty_bar + stage), phase ^ 1);
          const uint32_t fb = smem_u32(full_bar + stage);
          mbar_expect_tx(fb, (uint32_t)kStage2Bytes);
          uint8_t* sa = ring + (size_t)stage * kStage2Bytes;
          bulk_g2s(smem_u32(sa), a_src + (size_t)kt * kTileBytes, kTileBytes, fb);
          bulk_g2s(smem_u32(sa + kTileBytes), b_src + (size_t)kt * kTileBytes, kTileBytes, fb);
          if (++stage == kStages2) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0 && rank == 0) {
      // ===== MMA issuer of the pair =====
      uint32_t stage = 0, phase = 0, acc = 0, acc_phase = 0;
      for (int w = pair; w < num_work; w += npairs) {
        const int kb = k_tiles(ncols, w / nblk, KT);
        mbar_wait(smem_u32(tempty_bar + acc), acc_phase ^ 1);  // both epilogues have drained this accumulator
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * 256;
        for (int kt = 0; kt < kb; ++kt) {
          mbar_wait(smem_u32(full_bar + stage), phase);
          mbar_wait(smem_u32(peer_full_bar + stage), phase);
          tc_fence_after();
          const uint32_t sa = smem_u32(ring + (size_t)stage * kStage2Bytes);
          const uint64_t da = make_desc_sw128(sa);
          const uint64_t db = make_desc_sw128(sa + kTileBytes);
#pragma unroll
          for (int k = 0; k < kTile / 32; ++k)
            umma_i8_2(d_tmem, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), kIdesc, (kt > 0 || k > 0) ? 1u : 0u);
          umma_commit2(smem_u32(empty_bar + stage));  // frees the slot in both CTAs once the MMAs have read it
          if (++stage == kStages2) { stage = 0; phase ^= 1; }
        }
        umma_commit2(smem_u32(tfull_bar + acc));  // accumulator complete -> both epilogues
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
    } else if (lane == 0) {
      // ===== relay: "stage s of CTA 1 is full" -> leader =====
      uint32_t stage = 0, phase = 0;
      for (int w = pair; w < num_work; w += npairs) {
        const int kb = k_tiles(ncols, w / nblk, KT);
        for (int kt = 0; kt < kb; ++kt) {
          mbar_wait(smem_u32(full_bar + stage), phase);
          mbar_arrive_remote(map_to_cta(smem_u32(peer_full_bar + stage), 0));
          if (++stage == kStages2) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else {
    // ===== epilogue of this CTA's 128 rows: warp q = warp % 4 owns TMEM lanes [32q, 32q + 32), two warps per quarter
    // split the 256 accumulator columns =====
    const int q = warp & 3;
    const int half = (warp - 2) >> 2;
    const uint32_t tempty_leader = map_to_cta(smem_u32(tempty_bar), 0);
    uint32_t acc = 0, acc_phase = 0;
    for (int w = pair; w < num_work; w += npairs) {
      Work2 wk;
      get_work2(w, B, nblk, &wk);
      mbar_wait(smem_u32(tfull_bar + acc), acc_phase);
      tc_fence_after();
      const int row = (2 * wk.bi + (int)rank) * kTile + q * 32 + lane;
      const bool mirror = wk.bj > wk.bi;
#pragma unroll 1
      for (int c0 = half * 128; c0 < (half + 1) * 128; c0 += 32) {
        uint32_t v[32];
        tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + acc * 256 + c0, v);
        const int col0 = wk.bj * 256 + c0;
        if (Gi_base) {
          int32_t* Gi = Gi_base + (size_t)wk.b * g_stride;
          int32_t* dst = Gi + (size_t)row * ldg + col0;
#pragma unroll
          for (int e = 0; e < 32; e += 8) st_global_v8(dst + e, v + e);  // 256-bit stores: whole 32-byte sectors
          if (mirror) {  // lanes walk consecutive rows => coalesced 128-byte segments
#pragma unroll
            for (int e = 0; e < 32; ++e) Gi[(size_t)(col0 + e) * ldg + row] = (int)v[e];
          }
        } else {
          double* G = G_base + (size_t)wk.b * g_stride;
          double* dst = G + (size_t)row * ldg + col0;
#pragma unroll
          for (int e = 0; e < 32; e += 2) *reinterpret_cast<double2*>(dst + e) = make_double2((double)(int)v[e], (double)(int)v[e + 1]);
          if (mirror) {
#pragma unroll
            for (int e = 0; e < 32; ++e) G[(size_t)(col0 + e) * ldg + row] = (double)(int)v[e];
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (rank == 0) mbar_arrive(smem_u32(tempty_bar + acc));
        else mbar_arrive_remote(tempty_leader + acc * 8);
      }
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();  // no multicast commit / remote arrive may target a CTA that has exited
  if (warp == 1) {
    __syncwarp();
    tmem_dealloc2(tmem_base, 512);
  }
}

// split-K finalize: 64-bit integer accumulators (upper 256-block triangle valid) -> symmetric fp64 G
__global__ void gram_finalize_kernel(const unsigned long long* __restrict__ acc_base, int64_t R, int64_t ldg, double* __restrict__ G_base,
                                     int64_t g_stride) {
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= R * R) return;
  const unsigned long long* acc64 = acc_base + (size_t)blockIdx.y * R * R;
  double* G = G_base + (size_t)blockIdx.y * g_stride;
  int64_t r = idx / R, c = idx - r * R;
  unsigned long long v = ((c >> 8) >= (r >> 8)) ? acc64[r * ldg + c] : acc64[c * ldg + r];
  G[r * ldg + c] = (double)(long long)v;
}

// ---------------------------------------------------------------------------------------------------
// small row counts (rows_pad <= 64): dp4a on the "k4-major" layout.
//   SPB_S0_K4MAJOR: the 4 bytes k = 4w .. 4w+3 of row r form one 32-bit word stored at word index w * rows_pad + r,
//   so (a) a K chunk of all rows is one contiguous piece of memory (straight 128-bit copies, no transpose) and
//   (b) the four rows 4t .. 4t+3 of one word column are ONE conflict-free LDS.128.
// Thread (ty, tx) of a group owns the 4 x 4 outputs rows 4ty.. x rows 4tx..; per word column it issues 2 LDS.128 and
// 16 dp4a.  256 / (rows_pad/4)^2 groups share the word columns of a chunk; accumulators stay in registers (u32 per
// chunk: 255^2 * 4 * 256 < 2^32, u64 across chunks) for the whole persistent CTA, then one 64-bit atomic per output.
// ---------------------------------------------------------------------------------------------------
constexpr int kSmallWords = 256;  // word columns (= 1024 k) per chunk

__global__ void __launch_bounds__(256) gram_u8_small_kernel(const uint32_t* __restrict__ s0w_base, int64_t s0_stride_words, int Rp,
                                                            int64_t words, const int32_t* __restrict__ ncols,
                                                            unsigned long long* __restrict__ acc_base) {
  extern __shared__ __align__(16) uint32_t s_chunk[];  // [kSmallWords][Rp]
  const uint32_t* s0w = s0w_base + (size_t)blockIdx.y * s0_stride_words;
  unsigned long long* acc64 = acc_base + (size_t)blockIdx.y * Rp * Rp;
  const int tid = threadIdx.x;
  const int q = Rp >> 2;                 // 4-row blocks per side
  const int per_group = q * q;           // threads of one group
  const int groups = 256 / per_group;    // >= 1 for Rp <= 64
  const int grp = tid / per_group, t = tid - grp * per_group;
  const int ty = t / q, tx = t - ty * q;
  const bool active = grp < groups;
  unsigned long long tot[16];
#pragma unroll
  for (int e = 0; e < 16; ++e) tot[e] = 0ull;
  if (ncols) words = min(words, ((int64_t)ncols[blockIdx.y] + 3) / 4);  // word columns holding the occupied columns
  const int64_t nchunks = (words + kSmallWords - 1) / kSmallWords;
  for (int64_t ch = blockIdx.x; ch < nchunks; ch += gridDim.x) {
    const int64_t w0 = ch * kSmallWords;
    const int nw = (int)min((int64_t)kSmallWords, words - w0);
    __syncthreads();
    const uint4* src = reinterpret_cast<const uint4*>(s0w + w0 * Rp);  // Rp % 4 == 0: 16-byte aligned
    for (int v = tid; v < nw * Rp / 4; v += 256) reinterpret_cast<uint4*>(s_chunk)[v] = __ldg(src + v);
    __syncthreads();
    if (active) {
      uint32_t part[16];
#pragma unroll
      for (int e = 0; e < 16; ++e) part[e] = 0u;
      for (int w = grp; w < nw; w += groups) {
        const uint4 x = *reinterpret_cast<const uint4*>(s_chunk + w * Rp + 4 * ty);
        const uint4 y = *reinterpret_cast<const uint4*>(s_chunk + w * Rp + 4 * tx);
        const uint32_t xs[4] = {x.x, x.y, x.z, x.w}, ys[4] = {y.x, y.y, y.z, y.w};
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) part[i * 4 + j] = __dp4a(xs[i], ys[j], part[i * 4 + j]);
      }
#pragma unroll
      for (int e = 0; e < 16; ++e) tot[e] += part[e];
    }
  }
  if (active) {
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (tot[i * 4 + j]) atomicAdd(acc64 + (int64_t)(4 * ty + i) * Rp + 4 * tx + j, tot[i * 4 + j]);
  }
}

// acc64 [Rp][Rp] -> fp64 G [ld][ld] leading Rp x Rp block
__global__ void gram_small_finalize_kernel(const unsigned long long* __restrict__ acc_base, int R, int64_t ld, double* __restrict__ G_base,
                                           int64_t g_stride) {
  int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= R * R) return;
  int r = idx / R, c = idx - r * R;
  G_base[(size_t)blockIdx.y * g_stride + (int64_t)r * ld + c] = (double)(long long)acc_base[(size_t)blockIdx.y * R * R + idx];
}

// ---------------------------------------------------------------------------------------------------
// generic SIMT Gram for any layout / size: the on-device cross-check of the tensor-core kernel (tests)
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ int64_t s0_offset(int layout, int64_t rows_pad, int64_t pitch, int64_t r, int64_t k) {
  if (layout == SPB_S0_ROWMAJOR) return r * pitch + k;
  if (layout == SPB_S0_K4MAJOR) return ((k >> 2) * rows_pad + r) * 4 + (k & 3);
  int64_t KT = pitch / kTile;
  int64_t rt = r / kTile, kt = k / kTile;
  int rr = (int)(r - rt * kTile), kk = (int)(k - kt * kTile);
  return (rt * KT + kt) * kTileBytes + rr * 128 + ((((kk >> 4) ^ (rr & 7))) << 4) + (kk & 15);
}

__global__ void gram_u8_simt_kernel(const uint8_t* __restrict__ s0, int layout, int64_t R, int64_t pitch, int64_t ldg,
                                    double* __restrict__ G) {
  int64_t r1 = blockIdx.y, r2 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r2 >= R) return;
  unsigned long long s = 0;
  for (int64_t k = 0; k < pitch; ++k)
    s += (unsigned long long)s0[s0_offset(layout, R, pitch, r1, k)] * (unsigned long long)s0[s0_offset(layout, R, pitch, r2, k)];
  G[r1 * ldg + r2] = (double)s;
}

// ---------------------------------------------------------------------------------------------------
// sparse high-part corrections: G += S0 H^T + H S0^T + H H^T
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) hi_cross_kernel(const uint8_t* __restrict__ s0_base, int64_t s0_stride, int layout, int64_t R,
                                                       int64_t pitch, const int32_t* __restrict__ hi_rc_base,
                                                       const uint32_t* __restrict__ hi_val_base, const uint32_t* __restrict__ hi_num_base,
                                                       int64_t hi_cap, int64_t ldg, double* __restrict__ G_base, int64_t g_stride) {
  const int b = blockIdx.z;
  const uint8_t* s0 = s0_base + (size_t)b * s0_stride;
  const int32_t* hi_rc = hi_rc_base + (size_t)b * 2 * hi_cap;
  const uint32_t* hi_val = hi_val_base + (size_t)b * hi_cap;
  double* G = G_base + (size_t)b * g_stride;
  int64_t n = hi_num_base[b];
  if (n > hi_cap) n = hi_cap;
  for (int64_t e = blockIdx.y; e < n; e += gridDim.y) {
    const int64_t r = hi_rc[2 * e], c = hi_rc[2 * e + 1];
    const double v = (double)hi_val[e];
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < R; i += (int64_t)gridDim.x * blockDim.x) {
      uint32_t s = s0[s0_offset(layout, R, pitch, i, c)];
      if (s) {
        double t = v * (double)s;
        atomicAdd(G + i * ldg + r, t);  // (S0 H^T)[i][r]
        atomicAdd(G + r * ldg + i, t);  // (H S0^T)[r][i]
      }
    }
  }
}

// one thread per ordered pair (e1, e2) of high entries; pairs in the same column contribute v1 * v2 to G[r1][r2]
__global__ void __launch_bounds__(256) hi_self_kernel(const int32_t* __restrict__ hi_rc_base, const uint32_t* __restrict__ hi_val_base,
                                                      const uint32_t* __restrict__ hi_num_base, int64_t hi_cap, int64_t ldg,
                                                      double* __restrict__ G_base, int64_t g_stride) {
  const int b = blockIdx.y;
  const int32_t* hi_rc = hi_rc_base + (size_t)b * 2 * hi_cap;
  const uint32_t* hi_val = hi_val_base + (size_t)b * hi_cap;
  double* G = G_base + (size_t)b * g_stride;
  int64_t n = hi_num_base[b];
  if (n > hi_cap) n = hi_cap;
  const int64_t pairs = n * n;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < pairs; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t e1 = t / n, e2 = t - e1 * n;
    if (hi_rc[2 * e1 + 1] == hi_rc[2 * e2 + 1])
      atomicAdd(G + (int64_t)hi_rc[2 * e1] * ldg + hi_rc[2 * e2], (double)hi_val[e1] * (double)hi_val[e2]);  // (H H^T)[r1][r2]
  }
}

// ---------------------------------------------------------------------------------------------------
// The same correction kept OUT of G (32-bit integer Gram): C = S0 H^T + H S0^T + H H^T is non-zero only in the rows
// and columns that hold a high entry, so the rows C[hr[p]][:] of the m distinct high rows ("strip", fp64, exact
// integers) describe all of it: C[i][j] = Cs[pos[i]][j] if pos[i] >= 0, else Cs[pos[j]][i] if pos[j] >= 0, else 0.
// ---------------------------------------------------------------------------------------------------
// one block per matrix: pos[i] = index of row i among the distinct high rows (ascending) or -1; hr = their list; hm = m
__global__ void __launch_bounds__(1024) hi_rows_kernel(const int32_t* __restrict__ hi_rc_base, const uint32_t* __restrict__ hi_num_base,
                                                       int64_t hi_cap, int64_t R, int32_t* __restrict__ pos_base,
                                                       int32_t* __restrict__ hr_base, int64_t cs_rows, int32_t* __restrict__ hm) {
  __shared__ int s_part[1024];
  const int b = blockIdx.x, tid = threadIdx.x;
  const int32_t* hi_rc = hi_rc_base + (size_t)b * 2 * hi_cap;
  int32_t* pos = pos_base + (size_t)b * R;
  int32_t* hr = hr_base + (size_t)b * cs_rows;
  int64_t n = hi_num_base[b];
  if (n > hi_cap) n = hi_cap;
  for (int64_t i = tid; i < R; i += 1024) pos[i] = 0;
  __syncthreads();
  for (int64_t e = tid; e < n; e += 1024) pos[hi_rc[2 * e]] = 1;
  __syncthreads();
  const int64_t per = (R + 1023) / 1024;
  const int64_t i0 = tid * per, i1 = min(R, i0 + per);
  int cnt = 0;
  for (int64_t i = i0; i < i1; ++i) cnt += pos[i];
  s_part[tid] = cnt;
  __syncthreads();
  for (int o = 1; o < 1024; o <<= 1) {  // inclusive scan
    int v = tid >= o ? s_part[tid - o] : 0;
    __syncthreads();
    s_part[tid] += v;
    __syncthreads();
  }
  int run = s_part[tid] - cnt;
  for (int64_t i = i0; i < i1; ++i) {
    if (pos[i]) {
      if (run < cs_rows) { pos[i] = run; hr[run] = (int32_t)i; } else pos[i] = -1;
      ++run;
    } else {
      pos[i] = -1;
    }
  }
  if (tid == 1023) hm[b] = (int32_t)min((int64_t)s_part[1023], cs_rows);
}

__global__ void __launch_bounds__(256) hi_strip_cross_kernel(const uint8_t* __restrict__ s0_base, int64_t s0_stride, int layout, int64_t R,
                                                             int64_t pitch, const int32_t* __restrict__ hi_rc_base,
                                                             const uint32_t* __restrict__ hi_val_base,
                                                             const uint32_t* __restrict__ hi_num_base, int64_t hi_cap,
                                                             const int32_t* __restrict__ pos_base, double* __restrict__ Cs_base,
                                                             int64_t cs_rows) {
  const int b = blockIdx.z;
  const uint8_t* s0 = s0_base + (size_t)b * s0_stride;
  const int32_t* hi_rc = hi_rc_base + (size_t)b * 2 * hi_cap;
  const uint32_t* hi_val = hi_val_base + (size_t)b * hi_cap;
  const int32_t* pos = pos_base + (size_t)b * R;
  double* Cs = Cs_base + (size_t)b * cs_rows * R;
  int64_t n = hi_num_base[b];
  if (n > hi_cap) n = hi_cap;
  for (int64_t e = blockIdx.y; e < n; e += gridDim.y) {
    const int64_t r = hi_rc[2 * e], c = hi_rc[2 * e + 1];
    const int pr = pos[r];
    const double v = (double)hi_val[e];
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < R; i += (int64_t)gridDim.x * blockDim.x) {
      uint32_t s = s0[s0_offset(layout, R, pitch, i, c)];
      if (s) {
        double t = v * (double)s;
        if (pr >= 0) atomicAdd(Cs + (int64_t)pr * R + i, t);      // (H S0^T)[r][i]
        const int pi = pos[i];
        if (pi >= 0) atomicAdd(Cs + (int64_t)pi * R + r, t);      // (S0 H^T)[i][r], kept only for strip rows
      }
    }
  }
}

__global__ void __launch_bounds__(256) hi_strip_self_kernel(const int32_t* __restrict__ hi_rc_base, const uint32_t* __restrict__ hi_val_base,
                                                            const uint32_t* __restrict__ hi_num_base, int64_t hi_cap, int64_t R,
                                                            const int32_t* __restrict__ pos_base, double* __restrict__ Cs_base,
                                                            int64_t cs_rows) {
  const int b = blockIdx.y;
  const int32_t* hi_rc = hi_rc_base + (size_t)b * 2 * hi_cap;
  const uint32_t* hi_val = hi_val_base + (size_t)b * hi_cap;
  const int32_t* pos = pos_base + (size_t)b * R;
  double* Cs = Cs_base + (size_t)b * cs_rows * R;
  int64_t n = hi_num_base[b];
  if (n > hi_cap) n = hi_cap;
  const int64_t pairs = n * n;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < pairs; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t e1 = t / n, e2 = t - e1 * n;
    if (hi_rc[2 * e1 + 1] == hi_rc[2 * e2 + 1]) {
      const int p1 = pos[hi_rc[2 * e1]];
      if (p1 >= 0) atomicAdd(Cs + (int64_t)p1 * R + hi_rc[2 * e2], (double)hi_val[e1] * (double)hi_val[e2]);  // (H H^T)[r1][r2]
    }
  }
}

// ---------------------------------------------------------------------------------------------------
// The cross terms of the strip from the PATTERN TABLE instead of from S0 (round 2).  hi_strip_cross_kernel reads, for every
// high entry (r, c, v), the whole column c of S0: rows_pad bytes, each in its own 128-byte line of the tiled layout (1 M sector
// reads per 4096^2 matrix with 256 high entries).  But S0 holds one cell per pattern of the table, so the same sum is a join of
// the pattern list with the high list on the column index: chain the high entries of every column (colmap / next), then one
// pass over the patterns -- (r', c', s = count & 255) -- walks the chain of column c'.  60 k patterns instead of 1 M cells.
// Values are integers below 2^53: the atomics are exact and order-independent.
// ---------------------------------------------------------------------------------------------------
struct SplitBatchG {  // as SplitBatch of flatten.cu: the splits of one launch, passed by value
  SplitDev s[SPB_MAX_BATCH];
};

__global__ void hi_chain_kernel(const int32_t* __restrict__ hi_rc_base, const uint32_t* __restrict__ hi_num_base, int64_t hi_cap,
                                int32_t* __restrict__ colmap_base, int64_t pitch, int32_t* __restrict__ next_base) {
  const int b = blockIdx.y;
  int64_t n = hi_num_base[b];
  if (n > hi_cap) n = hi_cap;
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  const int32_t c = hi_rc_base[((size_t)b * hi_cap + e) * 2 + 1];
  next_base[(size_t)b * hi_cap + e] = atomicExch(colmap_base + (size_t)b * pitch + c, (int32_t)e + 1);  // 0 = end of chain
}

__global__ void __launch_bounds__(256) hi_join_kernel(const uint64_t* __restrict__ keys, const uint32_t* __restrict__ counts, int64_t num,
                                                      const __grid_constant__ SplitBatchG sb, int64_t R, int64_t pitch,
                                                      const int32_t* __restrict__ hi_rc_base, const uint32_t* __restrict__ hi_val_base,
                                                      int64_t hi_cap, const int32_t* __restrict__ colmap_base,
                                                      const int32_t* __restrict__ next_base, const int32_t* __restrict__ pos_base,
                                                      double* __restrict__ Cs_base, int64_t cs_rows, const uint32_t* __restrict__ colrank,
                                                      int64_t cr_words) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= num) return;
  const uint32_t s = counts[i] & 255u;
  if (s == 0) return;
  const int b = blockIdx.y;
  const SplitDev& sp = sb.s[b];
  const uint64_t k = keys[i];
  const int64_t ri = (int64_t)side_index(k, sp.sh_a, sp.a);
  int64_t ci = (int64_t)side_index(k, sp.sh_b, sp.b);
  if (colrank) {  // the high list holds ranked columns (spb_flatten_u8_batch_cols): look the pattern's column up the same way
    const uint32_t* cr = colrank + (size_t)b * 2 * cr_words;
    const uint32_t w = cr[ci >> 5];
    ci = (int64_t)cr[cr_words + (ci >> 5)] + __popc(w & ((1u << (ci & 31)) - 1u));
  }
  int32_t e = colmap_base[(size_t)b * pitch + ci];
  if (e == 0) return;
  const int32_t* hi_rc = hi_rc_base + (size_t)b * 2 * hi_cap;
  const uint32_t* hi_val = hi_val_base + (size_t)b * hi_cap;
  const int32_t* next = next_base + (size_t)b * hi_cap;
  const int32_t* pos = pos_base + (size_t)b * R;
  double* Cs = Cs_base + (size_t)b * cs_rows * R;
  const int pi = pos[ri];
  while (e) {
    const int32_t e0 = e - 1;
    const int64_t r = hi_rc[2 * e0];
    const double t = (double)hi_val[e0] * (double)s;
    const int pr = pos[r];
    if (pr >= 0) atomicAdd(Cs + (int64_t)pr * R + ri, t);   // (H S0^T)[r][i]
    if (pi >= 0) atomicAdd(Cs + (int64_t)pi * R + r, t);    // (S0 H^T)[i][r], kept only for strip rows
    e = next[e0];
  }
}

// zero the strip rows that are in use (rows >= hm[b] are never read)
__global__ void strip_zero_kernel(double* __restrict__ Cs_base, int64_t cs_rows, int64_t R, const int32_t* __restrict__ hm) {
  const int b = blockIdx.z, p = blockIdx.y;
  if (p >= hm[b]) return;
  double2* row = reinterpret_cast<double2*>(Cs_base + ((size_t)b * cs_rows + p) * R);
  for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < R / 2; j += (int64_t)gridDim.x * blockDim.x) row[j] = make_double2(0.0, 0.0);
}

struct UmmaPlan {
  int BN, T, KT, tiles, ksplit, kt_per_split, num_work;
  size_t smem;
};

UmmaPlan plan_umma(int64_t rows_pad, int64_t pitch, int nb) {
  UmmaPlan p;
  p.BN = rows_pad >= 256 ? 256 : 128;
  p.T = (int)(rows_pad / kTile);
  p.KT = (int)(pitch / kTile);
  int TN = (int)(rows_pad / p.BN);
  p.tiles = p.BN == 256 ? count_tiles<256>(p.T, TN) : count_tiles<128>(p.T, TN);
  // split K only when the batch does not give every SM a tile; one s32 accumulation must stay below 2^31:
  // 255^2 * 128 * kt <= 2^31 -> kt <= 258
  int sms = sm_count();
  int total = p.tiles * nb;
  int ks = 1;
  if (total < sms) ks = (sms + total - 1) / total;
  if (ks > p.KT) ks = p.KT;
  int per = (p.KT + ks - 1) / ks;
  if (per > 256) per = 256;
  ks = (p.KT + per - 1) / per;
  p.ksplit = ks;
  p.kt_per_split = per;
  p.num_work = total * ks;
  p.smem = (size_t)kStages * (kTileBytes + p.BN * kTile) + 16 * 8 + 1024;
  return p;
}

// Launches the CTA-pair kernel for nb matrices (no K split: one accumulation covers all of K, KT <= 256).
int launch_umma2(const uint8_t* d_s0, int64_t s0_stride, int nb, int64_t rows_pad, int64_t pitch, const int32_t* d_ncols, double* d_G,
                 int32_t* d_Gi, int64_t g_stride, cudaStream_t st) {
  const int B = (int)(rows_pad / 256), KT = (int)(pitch / kTile);
  const int nblk = B * (B + 1) / 2;
  const int num_work = nblk * nb;
  const size_t smem = (size_t)kStages2 * kStage2Bytes + 32 * 8 + 1024;
  static int max_pairs = 0;
  if (max_pairs == 0) {
    SPB_CUDA(cudaFuncSetAttribute(gram_u8_umma2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(2 * sm_count());
    cfg.blockDim = dim3(kUmmaThreads);
    cfg.dynamicSmemBytes = smem;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    int n = 0;
    if (cudaOccupancyMaxActiveClusters(&n, gram_u8_umma2_kernel, &cfg) != cudaSuccess || n < 1) { cudaGetLastError(); n = sm_count() / 2; }
    max_pairs = n;
  }
  const int pairs = num_work < max_pairs ? num_work : max_pairs;
  gram_u8_umma2_kernel<<<2 * pairs, kUmmaThreads, smem, st>>>(d_s0, s0_stride, B, KT, d_ncols, nblk, num_work, rows_pad, d_G, g_stride,
                                                             d_Gi);
  SPB_LAUNCH_CHECK();
  return SPB_OK;
}

}  // namespace

extern "C" int64_t spb_s0_bytes(int64_t rows_pad, int64_t pitch) { return rows_pad * pitch; }

extern "C" int64_t spb_gram_u8_ws(int64_t rows_pad, int64_t pitch, int layout, int nb) {
  if (nb < 1) nb = 1;
  if (layout == SPB_S0_K4MAJOR) return nb * rows_pad * rows_pad;
  if (layout != SPB_S0_TILED || rows_pad % kTile || pitch % kTile) return 0;
  UmmaPlan p = plan_umma(rows_pad, pitch, nb);
  return p.ksplit > 1 ? nb * rows_pad * rows_pad : 0;
}

// d_ncols: NULL (K = pitch) or int32 [nb] occupied columns per matrix (K = ncols[b]; S0 is zero beyond it).  The launch is
// planned for K = pitch; each matrix then runs only the K tiles that hold its columns.
extern "C" int spb_gram_u8_batch_cols(const uint8_t* d_s0, int64_t s0_stride, int nb, int64_t rows_pad, int64_t pitch, int layout,
                                      const int32_t* d_ncols, double* d_G, int64_t g_stride, uint64_t* d_ws, void* stream) {
  SPB_REQUIRE(d_s0 && d_G && rows_pad >= 1 && pitch >= 16 && pitch % 16 == 0 && nb >= 1 && nb <= 65535,
              "spb_gram_u8: bad arguments");
  SPB_REQUIRE(nb == 1 || (s0_stride >= rows_pad * pitch && s0_stride % 16 == 0 && g_stride >= rows_pad * rows_pad),
              "spb_gram_u8: bad batch strides");
  cudaStream_t st = (cudaStream_t)stream;
  if (layout == SPB_S0_K4MAJOR) {
    SPB_REQUIRE(rows_pad <= 64 && rows_pad % 4 == 0, "spb_gram_u8: the k4-major (dp4a) path handles rows_pad <= 64, rows_pad %% 4 == 0 "
                "(got %lld); use the tiled layout", (long long)rows_pad);
    SPB_REQUIRE(d_ws, "spb_gram_u8: workspace required (spb_gram_u8_ws)");
    int R = (int)rows_pad;
    SPB_CUDA(cudaMemsetAsync(d_ws, 0, (size_t)nb * R * R * 8, st));
    size_t smem = (size_t)kSmallWords * R * 4;
    SPB_CUDA(cudaFuncSetAttribute(gram_u8_small_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int64_t words = pitch / 4;
    int64_t nchunks = (words + kSmallWords - 1) / kSmallWords;
    int64_t gx = ((int64_t)sm_count() * 2 + nb - 1) / nb;
    if (gx > nchunks) gx = nchunks;
    if (gx < 1) gx = 1;
    dim3 grid((unsigned)gx, (unsigned)nb);
    gram_u8_small_kernel<<<grid, 256, smem, st>>>(reinterpret_cast<const uint32_t*>(d_s0), s0_stride / 4, R, words, d_ncols,
                                                  (unsigned long long*)d_ws);
    SPB_LAUNCH_CHECK();
    dim3 fg((R * R + 255) / 256, (unsigned)nb);
    gram_small_finalize_kernel<<<fg, 256, 0, st>>>((const unsigned long long*)d_ws, R, rows_pad, d_G, g_stride);
    SPB_LAUNCH_CHECK();
    return SPB_OK;
  }
  SPB_REQUIRE(layout == SPB_S0_TILED, "spb_gram_u8: layout %d has no Gram kernel (use SPB_S0_K4MAJOR or SPB_S0_TILED)", layout);
  SPB_REQUIRE(rows_pad % kTile == 0 && pitch % kTile == 0 && (rows_pad == kTile || rows_pad % 256 == 0),
              "spb_gram_u8: the tiled (tcgen05) path needs pitch %% 128 == 0 and rows_pad == 128 or a multiple of 256 "
              "(got rows_pad=%lld pitch=%lld)", (long long)rows_pad, (long long)pitch);
  SPB_REQUIRE(rows_pad <= 32768, "spb_gram_u8: rows_pad too large");
  UmmaPlan p = plan_umma(rows_pad, pitch, nb);
  unsigned long long* acc = nullptr;
  if (p.ksplit > 1) {
    SPB_REQUIRE(d_ws, "spb_gram_u8: workspace required (spb_gram_u8_ws)");
    acc = (unsigned long long*)d_ws;
    SPB_CUDA(cudaMemsetAsync(acc, 0, (size_t)nb * rows_pad * rows_pad * 8, st));
  }
  if (p.BN == 256 && p.ksplit == 1 && p.KT <= 256)
    return launch_umma2(d_s0, s0_stride, nb, rows_pad, pitch, d_ncols, d_G, nullptr, g_stride, st);
  int grid = p.num_work < sm_count() ? p.num_work : sm_count();
  if (p.BN == 256) {
    SPB_CUDA(cudaFuncSetAttribute(gram_u8_umma_kernel<256>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem));
    gram_u8_umma_kernel<256><<<grid, kUmmaThreads, p.smem, st>>>(d_s0, s0_stride, p.T, p.KT, p.tiles, p.ksplit, p.kt_per_split, d_ncols,
                                                               p.num_work, rows_pad, d_G, g_stride, acc);
  } else {
    SPB_CUDA(cudaFuncSetAttribute(gram_u8_umma_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem));
    gram_u8_umma_kernel<128><<<grid, kUmmaThreads, p.smem, st>>>(d_s0, s0_stride, p.T, p.KT, p.tiles, p.ksplit, p.kt_per_split, d_ncols,
                                                               p.num_work, rows_pad, d_G, g_stride, acc);
  }
  SPB_LAUNCH_CHECK();
  if (acc) {
    int64_t cells = rows_pad * rows_pad;
    dim3 fg((unsigned)((cells + 255) / 256), (unsigned)nb);
    gram_finalize_kernel<<<fg, 256, 0, st>>>(acc, rows_pad, rows_pad, d_G, g_stride);
    SPB_LAUNCH_CHECK();
  }
  return SPB_OK;
}

extern "C" int spb_gram_u8_batch(const uint8_t* d_s0, int64_t s0_stride, int nb, int64_t rows_pad, int64_t pitch, int layout,
                                 double* d_G, int64_t g_stride, uint64_t* d_ws, void* stream) {
  return spb_gram_u8_batch_cols(d_s0, s0_stride, nb, rows_pad, pitch, layout, nullptr, d_G, g_stride, d_ws, stream);
}

namespace spb {
int gram_u8_i32_launch(const uint8_t* d_s0, int64_t s0_stride, int nb, int64_t rows_pad, int64_t pitch, const int32_t* d_ncols,
                       int32_t* d_Gi, int64_t g_stride, cudaStream_t st) {
  SPB_REQUIRE(d_s0 && d_Gi && nb >= 1 && nb <= 65535, "spb_gram_u8_batch_i32: bad arguments");
  SPB_REQUIRE(rows_pad % 256 == 0 && rows_pad >= 256 && rows_pad <= 32768 && pitch % kTile == 0 && pitch >= kTile,
              "spb_gram_u8_batch_i32: needs the tiled layout with rows_pad %% 256 == 0 and pitch %% 128 == 0 (got %lld, %lld)",
              (long long)rows_pad, (long long)pitch);
  SPB_REQUIRE(pitch <= 256 * kTile, "spb_gram_u8_batch_i32: pitch %lld exceeds the %d columns one 32-bit accumulation can hold",
              (long long)pitch, 256 * kTile);
  SPB_REQUIRE(nb == 1 || (s0_stride >= rows_pad * pitch && s0_stride % 16 == 0 && g_stride >= rows_pad * rows_pad),
              "spb_gram_u8_batch_i32: bad batch strides");
  return launch_umma2(d_s0, s0_stride, nb, rows_pad, pitch, d_ncols, nullptr, d_Gi, g_stride, st);
}
}  // namespace spb

extern "C" int spb_gram_u8_batch_i32(const uint8_t* d_s0, int64_t s0_stride, int nb, int64_t rows_pad, int64_t pitch,
                                     int32_t* d_Gi, int64_t g_stride, void* stream) {
  return spb::gram_u8_i32_launch(d_s0, s0_stride, nb, rows_pad, pitch, nullptr, d_Gi, g_stride, (cudaStream_t)stream);
}

extern "C" int spb_gram_u8_batch_i32_cols(const uint8_t* d_s0, int64_t s0_stride, int nb, int64_t rows_pad, int64_t pitch,
                                          const int32_t* d_ncols, int32_t* d_Gi, int64_t g_stride, void* stream) {
  return spb::gram_u8_i32_launch(d_s0, s0_stride, nb, rows_pad, pitch, d_ncols, d_Gi, g_stride, (cudaStream_t)stream);
}

extern "C" int spb_gram_hi_strip_batch(const uint8_t* d_s0, int64_t s0_stride, int nb, int64_t rows_pad, int64_t pitch, int layout,
                                       const int32_t* d_hi_rc, const uint32_t* d_hi_val, const uint32_t* d_hi_num, int64_t hi_cap,
                                       double* d_Cs, int64_t cs_rows, int32_t* d_pos, int32_t* d_hr, int32_t* d_hm, void* stream) {
  SPB_REQUIRE(d_s0 && d_hi_rc && d_hi_val && d_hi_num && d_pos && d_hm && hi_cap >= 0 && nb >= 1 && nb <= 65535 && cs_rows >= 0,
              "spb_gram_hi_strip: bad arguments");
  SPB_REQUIRE(cs_rows == 0 || (d_Cs && d_hr), "spb_gram_hi_strip: NULL strip");
  cudaStream_t st = (cudaStream_t)stream;
  if (cs_rows) SPB_CUDA(cudaMemsetAsync(d_Cs, 0, (size_t)nb * cs_rows * rows_pad * sizeof(double), st));
  hi_rows_kernel<<<nb, 1024, 0, st>>>(d_hi_rc, d_hi_num, hi_cap, rows_pad, d_pos, d_hr, cs_rows, d_hm);
  SPB_LAUNCH_CHECK();
  if (hi_cap == 0 || cs_rows == 0) return SPB_OK;
  int64_t gy = hi_cap < 64 ? hi_cap : 64;
  dim3 grid((unsigned)((rows_pad + 255) / 256 > 16 ? 16 : (rows_pad + 255) / 256), (unsigned)gy, (unsigned)nb);
  hi_strip_cross_kernel<<<grid, 256, 0, st>>>(d_s0, s0_stride, layout, rows_pad, pitch, d_hi_rc, d_hi_val, d_hi_num, hi_cap, d_pos, d_Cs,
                                              cs_rows);
  SPB_LAUNCH_CHECK();
  int64_t gx = (4 * (int64_t)sm_count() + nb - 1) / nb;
  dim3 sg((unsigned)gx, (unsigned)nb);
  hi_strip_self_kernel<<<sg, 256, 0, st>>>(d_hi_rc, d_hi_val, d_hi_num, hi_cap, rows_pad, d_pos, d_Cs, cs_rows);
  SPB_LAUNCH_CHECK();
  return SPB_OK;
}

extern "C" int64_t spb_gram_hi_strip_table_ws(int nb, int64_t pitch, int64_t hi_cap) { return (int64_t)nb * (pitch + hi_cap); }

// d_colrank: NULL, or the column ranks the high list was scattered with (spb_col_ranks_batch, `words` per split)
extern "C" int spb_gram_hi_strip_batch_table_cols(const uint64_t* d_keys, const uint32_t* d_counts, int64_t num, const spb_split* h_splits,
                                                  int nb, int64_t rows_pad, int64_t pitch, const uint32_t* d_colrank, int64_t words,
                                                  const int32_t* d_hi_rc, const uint32_t* d_hi_val, const uint32_t* d_hi_num, int64_t hi_cap,
                                                  double* d_Cs, int64_t cs_rows, int32_t* d_pos, int32_t* d_hr, int32_t* d_hm, int32_t* d_ws,
                                                  void* stream) {
  SPB_REQUIRE(h_splits && d_hi_rc && d_hi_val && d_hi_num && d_pos && d_hm && d_ws && hi_cap >= 0 && nb >= 1 && nb <= SPB_MAX_BATCH &&
                  cs_rows >= 0 && cs_rows <= 65535 && rows_pad % 2 == 0,
              "spb_gram_hi_strip_table: bad arguments");
  SPB_REQUIRE(cs_rows == 0 || (d_Cs && d_hr), "spb_gram_hi_strip_table: NULL strip");
  SPB_REQUIRE(num <= 0 || (d_keys && d_counts), "spb_gram_hi_strip_table: NULL pattern table");
  SplitBatchG sb;
  for (int b = 0; b < nb; ++b) {
    int rc = make_split_dev(h_splits + b, &sb.s[b]);
    if (rc) return rc;
    const int64_t cols = d_colrank ? (num < (1ll << (2 * sb.s[b].b)) ? num : (1ll << (2 * sb.s[b].b))) : (1ll << (2 * sb.s[b].b));
    SPB_REQUIRE(sb.s[b].a + sb.s[b].b == sb.s[b].n && sb.s[b].a <= 15 && sb.s[b].b <= 15 && rows_pad >= (1ll << (2 * sb.s[b].a)) &&
                    pitch >= cols && (!d_colrank || words == ((1ll << (2 * sb.s[b].b)) + 31) / 32),
                "spb_gram_hi_strip_table: every split must cover all taxa and fit rows_pad x pitch");
  }
  cudaStream_t st = (cudaStream_t)stream;
  hi_rows_kernel<<<nb, 1024, 0, st>>>(d_hi_rc, d_hi_num, hi_cap, rows_pad, d_pos, d_hr, cs_rows, d_hm);
  SPB_LAUNCH_CHECK();
  if (hi_cap == 0 || cs_rows == 0) return SPB_OK;
  {
    dim3 zg((unsigned)((rows_pad / 2 + 255) / 256 > 8 ? 8 : (rows_pad / 2 + 255) / 256), (unsigned)cs_rows, (unsigned)nb);
    strip_zero_kernel<<<zg, 256, 0, st>>>(d_Cs, cs_rows, rows_pad, d_hm);
    SPB_LAUNCH_CHECK();
  }
  int32_t* colmap = d_ws;
  int32_t* next = d_ws + (size_t)nb * pitch;
  SPB_CUDA(cudaMemsetAsync(colmap, 0, (size_t)nb * pitch * sizeof(int32_t), st));
  {
    dim3 cg((unsigned)((hi_cap + 255) / 256), (unsigned)nb);
    hi_chain_kernel<<<cg, 256, 0, st>>>(d_hi_rc, d_hi_num, hi_cap, colmap, pitch, next);
    SPB_LAUNCH_CHECK();
  }
  if (num > 0) {
    dim3 jg((unsigned)((num + 255) / 256), (unsigned)nb);
    hi_join_kernel<<<jg, 256, 0, st>>>(d_keys, d_counts, num, sb, rows_pad, pitch, d_hi_rc, d_hi_val, hi_cap, colmap, next, d_pos, d_Cs,
                                       cs_rows, d_colrank, words);
    SPB_LAUNCH_CHECK();
  }
  int64_t gx = (4 * (int64_t)sm_count() + nb - 1) / nb;
  dim3 sg((unsigned)gx, (unsigned)nb);
  hi_strip_self_kernel<<<sg, 256, 0, st>>>(d_hi_rc, d_hi_val, d_hi_num, hi_cap, rows_pad, d_pos, d_Cs, cs_rows);
  SPB_LAUNCH_CHECK();
  return SPB_OK;
}

extern "C" int spb_gram_hi_strip_batch_table(const uint64_t* d_keys, const uint32_t* d_counts, int64_t num, const spb_split* h_splits,
                                             int nb, int64_t rows_pad, int64_t pitch, const int32_t* d_hi_rc, const uint32_t* d_hi_val,
                                             const uint32_t* d_hi_num, int64_t hi_cap, double* d_Cs, int64_t cs_rows, int32_t* d_pos,
                                             int32_t* d_hr, int32_t* d_hm, int32_t* d_ws, void* stream) {
  return spb_gram_hi_strip_batch_table_cols(d_keys, d_counts, num, h_splits, nb, rows_pad, pitch, nullptr, 0, d_hi_rc, d_hi_val, d_hi_num,
                                            hi_cap, d_Cs, cs_rows, d_pos, d_hr, d_hm, d_ws, stream);
}

extern "C" int spb_gram_u8(const uint8_t* d_s0, int64_t rows_pad, int64_t pitch, int layout, double* d_G, uint64_t* d_ws,
                           void* stream) {
  return spb_gram_u8_batch(d_s0, rows_pad * pitch, 1, rows_pad, pitch, layout, d_G, rows_pad * rows_pad, d_ws, stream);
}

// Test / cross-check entry: same result as spb_gram_u8 from a plain SIMT loop (any layout, any size).
extern "C" int spb_gram_u8_simt(const uint8_t* d_s0, int64_t rows_pad, int64_t pitch, int layout, double* d_G, void* stream) {
  SPB_REQUIRE(d_s0 && d_G && rows_pad >= 1 && pitch >= 1, "spb_gram_u8_simt: bad arguments");
  SPB_REQUIRE(layout == SPB_S0_ROWMAJOR || layout == SPB_S0_K4MAJOR || (rows_pad % kTile == 0 && pitch % kTile == 0),
              "spb_gram_u8_simt: bad tiled shape");
  dim3 grid((unsigned)((rows_pad + 127) / 128), (unsigned)rows_pad);
  gram_u8_simt_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>(d_s0, layout, rows_pad, pitch, rows_pad, d_G);
  SPB_LAUNCH_CHECK();
  return SPB_OK;
}

extern "C" int spb_gram_hi_correction_batch(const uint8_t* d_s0, int64_t s0_stride, int nb, int64_t rows_pad, int64_t pitch,
                                            int layout, const int32_t* d_hi_rc, const uint32_t* d_hi_val, const uint32_t* d_hi_num,
                                            int64_t hi_cap, double* d_G, int64_t g_stride, void* stream) {
  SPB_REQUIRE(d_s0 && d_hi_rc && d_hi_val && d_hi_num && d_G && hi_cap >= 0 && nb >= 1 && nb <= 65535,
              "spb_gram_hi_correction: bad arguments");
  if (hi_cap == 0) return SPB_OK;
  cudaStream_t st = (cudaStream_t)stream;
  int64_t gy = hi_cap < 64 ? hi_cap : 64;  // the entry loop strides over gridDim.y
  dim3 grid((unsigned)((rows_pad + 255) / 256 > 16 ? 16 : (rows_pad + 255) / 256), (unsigned)gy, (unsigned)nb);
  hi_cross_kernel<<<grid, 256, 0, st>>>(d_s0, s0_stride, layout, rows_pad, pitch, d_hi_rc, d_hi_val, d_hi_num, hi_cap, rows_pad, d_G,
                                        g_stride);
  SPB_LAUNCH_CHECK();
  int64_t gx = (4 * (int64_t)sm_count() + nb - 1) / nb;  // grid-stride over the n^2 pairs (n is only known on the device)
  dim3 sg((unsigned)gx, (unsigned)nb);
  hi_self_kernel<<<sg, 256, 0, st>>>(d_hi_rc, d_hi_val, d_hi_num, hi_cap, rows_pad, d_G, g_stride);
  SPB_LAUNCH_CHECK();
  return SPB_OK;
}

extern "C" int spb_gram_hi_correction(const uint8_t* d_s0, int64_t rows_pad, int64_t pitch, int layout, const int32_t* d_hi_rc,
                                      const uint32_t* d_hi_val, const uint32_t* d_hi_num, int64_t hi_cap, double* d_G,
                                      void* stream) {
  return spb_gram_hi_correction_batch(d_s0, rows_pad * pitch, 1, rows_pad, pitch, layout, d_hi_rc, d_hi_val, d_hi_num, hi_cap, d_G,
                                      rows_pad * rows_pad, stream);
}

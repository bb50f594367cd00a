// Kernel 2: flattening scatter.  Replaces splitp/constructions.py:31-55 (reduced), :58-102 (sparse) and
// defines FlatFormat.dense := sparse.todense().  Row = base-4 index over side A, col = base-4 index over
// side B, first listed taxon most significant (constructions.py:166-171).  Values are copied, never
// combined, so every format is bit-exact by construction; counts become probabilities with the same
// single IEEE division the reference performs (parsers/fasta.py:66-70).
#include "common.cuh"

namespace spb {
int rank_flags(const uint32_t* d_flags, int64_t cells, uint32_t* d_rank, uint32_t* d_tmp, cudaStream_t st);
}
using namespace spb;

namespace {

__device__ __forceinline__ double load_val(const void* vals, int kind, double divisor, int64_t i) {
  if (kind == SPB_VAL_U32) {
    double c = (double)reinterpret_cast<const uint32_t*>(vals)[i];
    return divisor > 0.0 ? c / divisor : c;
  }
  return reinterpret_cast<const double*>(vals)[i];
}

__global__ void coo_kernel(const uint64_t* __restrict__ keys, int64_t num, SplitDev sp, int64_t* rows, int64_t* cols) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= num) return;
  uint64_t k = keys[i];
  rows[i] = (int64_t)side_index(k, sp.sh_a, sp.a);
  cols[i] = (int64_t)side_index(k, sp.sh_b, sp.b);
}

// Assignment semantics of the reference (constructions.py:43,101): when several patterns land in the
// same cell (split does not cover all taxa) the LAST pattern in table order wins.  win[] holds the
// largest pattern index + 1 per cell; only that pattern writes.
__global__ void dense_win_kernel(const uint64_t* __restrict__ keys, int64_t num, SplitDev sp, const uint32_t* rank_r,
                                 const uint32_t* rank_c, int64_t C, uint32_t* win) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= num) return;
  uint64_t k = keys[i];
  uint64_t r = side_index(k, sp.sh_a, sp.a), c = side_index(k, sp.sh_b, sp.b);
  if (rank_r) { r = rank_r[r]; c = rank_c[c]; }
  atomicMax(win + r * C + c, (uint32_t)(i + 1));
}

__global__ void dense_fill_kernel(const uint64_t* __restrict__ keys, const void* __restrict__ vals, int kind, double divisor,
                                  int64_t num, SplitDev sp, const uint32_t* rank_r, const uint32_t* rank_c, int64_t C,
                                  const uint32_t* win, double* out) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= num) return;
  uint64_t k = keys[i];
  uint64_t r = side_index(k, sp.sh_a, sp.a), c = side_index(k, sp.sh_b, sp.b);
  if (rank_r) { r = rank_r[r]; c = rank_c[c]; }
  if (win && win[r * C + c] != (uint32_t)(i + 1)) return;
  out[r * C + c] = load_val(vals, kind, divisor, i);
}

__global__ void mark_kernel(const uint64_t* __restrict__ keys, int64_t num, SplitDev sp, uint32_t* flag_r, uint32_t* flag_c) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= num) return;
  uint64_t k = keys[i];
  flag_r[side_index(k, sp.sh_a, sp.a)] = 1u;
  flag_c[side_index(k, sp.sh_b, sp.b)] = 1u;
}

__device__ __forceinline__ int64_t s0_cell(int layout, int64_t rows_pad, int64_t pitch, uint64_t r, uint64_t c) {
  if (layout == SPB_S0_ROWMAJOR) return (int64_t)(r * (uint64_t)pitch + c);
  if (layout == SPB_S0_K4MAJOR) return (int64_t)(((c >> 2) * (uint64_t)rows_pad + r) * 4ull + (c & 3ull));  // csrc/gram.cu
  // 128 x 128-byte tiles, K-major SWIZZLE_128B inside the tile (the tcgen05 operand layout, csrc/gram.cu)
  uint64_t KT = (uint64_t)pitch >> 7;
  uint64_t rt = r >> 7, kt = c >> 7;
  uint32_t rr = (uint32_t)(r & 127), kk = (uint32_t)(c & 127);
  return (int64_t)((rt * KT + kt) * 16384ull + rr * 128u + ((((kk >> 4) ^ (rr & 7u))) << 4) + (kk & 15u));
}

struct SplitBatch {  // passed by value as a kernel parameter (64 x 140 bytes; CUDA >= 12.1 takes up to 32,764 bytes)
  SplitDev s[SPB_MAX_BATCH];
};

// ---------------------------------------------------------------------------------------------------
// Column ranks of a batch of count flattenings.  Only the columns that some pattern projects to are non-zero, so the u8
// scatter can store column c at its rank among the occupied columns: the Gram S0 S0^T, which contracts over the columns, is
// unchanged, and its K shrinks from 4^b to the occupied count.  Per split, `words` = ceil(4^b / 32) words of occupancy bits
// followed by `words` exclusive prefix counts of those bits (col_rank):
//     rank(c) = pre[c >> 5] + popc(bits[c >> 5] & ((1 << (c & 31)) - 1)).
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t col_rank(const uint32_t* cr, int64_t words, uint64_t c) {
  const uint32_t w = cr[c >> 5];
  return cr[words + (int64_t)(c >> 5)] + (uint32_t)__popc(w & ((1u << (c & 31u)) - 1u));
}

__global__ void col_mark_kernel(const uint64_t* __restrict__ keys, int64_t num, const __grid_constant__ SplitBatch sb,
                                uint32_t* __restrict__ cr_base, int64_t words) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= num) return;
  const int b = blockIdx.y;
  const SplitDev& sp = sb.s[b];
  const uint64_t c = side_index(keys[i], sp.sh_b, sp.b);
  uint32_t* w = cr_base + (size_t)b * 2 * words + (c >> 5);
  const uint32_t m = 1u << (c & 31u);
  if (!(*w & m)) atomicOr(w, m);  // most columns hold many patterns: skip the atomic once the bit is seen
}

// one block per split: exclusive prefix of the popcounts of its bit words; ncols[b] = occupied columns
constexpr int kRankThreads = 1024;
__global__ void __launch_bounds__(kRankThreads) col_prefix_kernel(uint32_t* __restrict__ cr_base, int64_t words, int32_t* __restrict__ ncols) {
  __shared__ uint32_t s_warp[kRankThreads / 32];
  uint32_t* bits = cr_base + (size_t)blockIdx.x * 2 * words;
  uint32_t* pre = bits + words;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t per = (words + kRankThreads - 1) / kRankThreads;  // contiguous words per thread
  const int64_t w0 = tid * per, w1 = min(words, w0 + per);
  uint32_t cnt = 0;
  for (int64_t w = w0; w < w1; ++w) cnt += __popc(bits[w]);
  uint32_t inc = cnt;  // inclusive scan over the block: warp shuffles, then the 32 warp totals
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    uint32_t v = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += v;
  }
  if (lane == 31) s_warp[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    uint32_t t = s_warp[lane], x = t;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      uint32_t v = __shfl_up_sync(0xffffffffu, x, o);
      if (lane >= o) x += v;
    }
    s_warp[lane] = x - t;  // exclusive warp offsets
  }
  __syncthreads();
  uint32_t run = s_warp[warp] + inc - cnt;
  for (int64_t w = w0; w < w1; ++w) {
    pre[w] = run;
    run += __popc(bits[w]);
  }
  if (tid == kRankThreads - 1) ncols[blockIdx.x] = (int32_t)run;
}

// blockIdx.y = batch entry: split sb.s[b], S0 buffer s0 + b * s0_stride, high-part buffers offset by b * hi_cap.
// counts == NULL: clear pass (writes zeros to the cells the scatter touched).
// colrank != NULL: column c of batch entry b is stored at its rank (col_rank over colrank + b * 2 * cr_words)
__global__ void u8_kernel(const uint64_t* __restrict__ keys, const uint32_t* __restrict__ counts, int64_t num,
                          const __grid_constant__ SplitBatch sb, const uint32_t* rank_r, const uint32_t* rank_c,
                          const uint32_t* __restrict__ colrank, int64_t cr_words, uint8_t* s0_base, int64_t s0_stride, int64_t rows_pad,
                          int64_t pitch, int layout, int32_t* hi_rc_base, uint32_t* hi_val_base, uint32_t* hi_num_base, int64_t hi_cap) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= num) return;
  const int b = blockIdx.y;
  const SplitDev& sp = sb.s[b];
  uint8_t* s0 = s0_base + (size_t)b * s0_stride;
  uint64_t k = keys[i];
  uint32_t cnt = counts ? counts[i] : 0u;
  uint64_t r = side_index(k, sp.sh_a, sp.a), c = side_index(k, sp.sh_b, sp.b);
  if (rank_r) { r = rank_r[r]; c = rank_c[c]; }
  if (colrank) c = col_rank(colrank + (size_t)b * 2 * cr_words, cr_words, c);
  s0[s0_cell(layout, rows_pad, pitch, r, c)] = (uint8_t)(cnt & 255u);
  if (cnt >= 256u) {
    uint32_t slot = atomicAdd(hi_num_base + b, 1u);
    if ((int64_t)slot < hi_cap) {
      int32_t* hi_rc = hi_rc_base + (size_t)b * 2 * hi_cap;
      hi_rc[2 * (int64_t)slot] = (int32_t)r;
      hi_rc[2 * (int64_t)slot + 1] = (int32_t)c;
      hi_val_base[(size_t)b * hi_cap + slot] = cnt - (cnt & 255u);
    }
  }
}

inline bool covers_all(const spb_split* s) {
  uint64_t m = 0;
  for (int i = 0; i < s->a; ++i) m |= 1ull << s->idx_a[i];
  for (int i = 0; i < s->b; ++i) m |= 1ull << s->idx_b[i];
  return s->a + s->b == s->n && m == ((s->n == 64) ? ~0ull : ((1ull << s->n) - 1ull));
}

inline unsigned nblk(int64_t n, int t) { return (unsigned)((n + t - 1) / t); }

}  // namespace

extern "C" int spb_flatten_coo(const uint64_t* d_keys, int64_t num, const spb_split* split, int64_t* d_rows, int64_t* d_cols,
                               void* stream) {
  SplitDev sp;
  int rc = make_split_dev(split, &sp);
  if (rc) return rc;
  SPB_REQUIRE(sp.a <= 31 && sp.b <= 31, "spb_flatten_coo: sides are limited to 31 taxa (int64 indices)");
  if (num <= 0) return SPB_OK;
  SPB_REQUIRE(d_keys && d_rows && d_cols, "spb_flatten_coo: NULL buffer");
  coo_kernel<<<nblk(num, 256), 256, 0, (cudaStream_t)stream>>>(d_keys, num, sp, d_rows, d_cols);
  SPB_LAUNCH_CHECK();
  return SPB_OK;
}

static int fill_common(const uint64_t* d_keys, const void* d_vals, int val_kind, double divisor, int64_t num,
                       const spb_split* split, const SplitDev& sp, const uint32_t* rank_r, const uint32_t* rank_c,
                       int64_t R, int64_t C, double* d_out, uint32_t* d_win, cudaStream_t st) {
  SPB_CUDA(cudaMemsetAsync(d_out, 0, (size_t)R * (size_t)C * sizeof(double), st));
  if (num <= 0) return SPB_OK;
  const uint32_t* win = nullptr;
  if (!covers_all(split)) {
    if (!d_win) {
      set_error("flattening: split does not cover all taxa; a winner workspace (uint32 per cell) is required");
      return SPB_ERR_ARG;
    }
    SPB_CUDA(cudaMemsetAsync(d_win, 0, (size_t)R * (size_t)C * sizeof(uint32_t), st));
    dense_win_kernel<<<nblk(num, 256), 256, 0, st>>>(d_keys, num, sp, rank_r, rank_c, C, d_win);
    SPB_LAUNCH_CHECK();
    win = d_win;
  }
  dense_fill_kernel<<<nblk(num, 256), 256, 0, st>>>(d_keys, d_vals, val_kind, divisor, num, sp, rank_r, rank_c, C, win, d_out);
  SPB_LAUNCH_CHECK();
  return SPB_OK;
}

// d_win: optional uint32 [4^a * 4^b] workspace, only needed when the split does not cover all taxa.
extern "C" int spb_flatten_dense_w(const uint64_t* d_keys, const void* d_vals, int val_kind, double divisor, int64_t num,
                                   const spb_split* split, double* d_out, uint32_t* d_win, void* stream) {
  SplitDev sp;
  int rc = make_split_dev(split, &sp);
  if (rc) return rc;
  SPB_REQUIRE(sp.a + sp.b <= 14, "spb_flatten_dense: 4^(a+b) cells with a+b=%d exceeds the dense limit (14)", sp.a + sp.b);
  SPB_REQUIRE(d_out && (num <= 0 || (d_keys && d_vals)), "spb_flatten_dense: NULL buffer");
  int64_t R = 1ll << (2 * sp.a), C = 1ll << (2 * sp.b);
  return fill_common(d_keys, d_vals, val_kind, divisor, num, split, sp, nullptr, nullptr, R, C, d_out, d_win,
                     (cudaStream_t)stream);
}

extern "C" int spb_flatten_dense(const uint64_t* d_keys, const void* d_vals, int val_kind, double divisor, int64_t num,
                                 const spb_split* split, double* d_out, void* stream) {
  return spb_flatten_dense_w(d_keys, d_vals, val_kind, divisor, num, split, d_out, nullptr, stream);
}

extern "C" int spb_flatten_reduced_plan(const uint64_t* d_keys, int64_t num, const spb_split* split, uint32_t* d_rank_r,
                                        uint32_t* d_rank_c, uint32_t* d_tmp, int64_t* h_shape, void* stream) {
  SplitDev sp;
  int rc = make_split_dev(split, &sp);
  if (rc) return rc;
  if (sp.a > 13 || sp.b > 13) {
    set_error("spb_flatten_reduced: sides are limited to 13 taxa in this version (a=%d b=%d)", sp.a, sp.b);
    return SPB_ERR_UNSUPPORTED;
  }
  SPB_REQUIRE(d_rank_r && d_rank_c && d_tmp && h_shape, "spb_flatten_reduced_plan: NULL buffer");
  cudaStream_t st = (cudaStream_t)stream;
  int64_t R = 1ll << (2 * sp.a), C = 1ll << (2 * sp.b);
  SPB_CUDA(cudaMemsetAsync(d_rank_r, 0, (size_t)(R + 1) * 4, st));
  SPB_CUDA(cudaMemsetAsync(d_rank_c, 0, (size_t)(C + 1) * 4, st));
  if (num > 0) {
    mark_kernel<<<nblk(num, 256), 256, 0, st>>>(d_keys, num, sp, d_rank_r, d_rank_c);
    SPB_LAUNCH_CHECK();
  }
  // flags and ranks alias: every thread reads its own flags before it writes their ranks
  rc = rank_flags(d_rank_r, R + 1, d_rank_r, d_tmp, st);
  if (rc) return rc;
  rc = rank_flags(d_rank_c, C + 1, d_rank_c, d_tmp, st);
  if (rc) return rc;
  uint32_t hr = 0, hc = 0;
  SPB_CUDA(cudaMemcpyAsync(&hr, d_rank_r + R, 4, cudaMemcpyDeviceToHost, st));
  SPB_CUDA(cudaMemcpyAsync(&hc, d_rank_c + C, 4, cudaMemcpyDeviceToHost, st));
  SPB_CUDA(cudaStreamSynchronize(st));
  h_shape[0] = hr;
  h_shape[1] = hc;
  return SPB_OK;
}

extern "C" int spb_flatten_reduced_fill_w(const uint64_t* d_keys, const void* d_vals, int val_kind, double divisor,
                                          int64_t num, const spb_split* split, const uint32_t* d_rank_r,
                                          const uint32_t* d_rank_c, int64_t R, int64_t C, double* d_out, uint32_t* d_win,
                                          void* stream) {
  SplitDev sp;
  int rc = make_split_dev(split, &sp);
  if (rc) return rc;
  if (R <= 0 || C <= 0) return SPB_OK;
  SPB_REQUIRE(d_out && d_rank_r && d_rank_c && (num <= 0 || (d_keys && d_vals)), "spb_flatten_reduced_fill: NULL buffer");
  return fill_common(d_keys, d_vals, val_kind, divisor, num, split, sp, d_rank_r, d_rank_c, R, C, d_out, d_win,
                     (cudaStream_t)stream);
}

extern "C" int spb_flatten_reduced_fill(const uint64_t* d_keys, const void* d_vals, int val_kind, double divisor, int64_t num,
                                        const spb_split* split, const uint32_t* d_rank_r, const uint32_t* d_rank_c,
                                        int64_t R, int64_t C, double* d_out, void* stream) {
  return spb_flatten_reduced_fill_w(d_keys, d_vals, val_kind, divisor, num, split, d_rank_r, d_rank_c, R, C, d_out, nullptr,
                                    stream);
}

static int u8_check(const spb_split* split, SplitDev* sp, const uint32_t* d_rank_r, const uint32_t* d_rank_c, uint8_t* d_s0,
                    int64_t rows_pad, int64_t pitch, int layout, int64_t col_bound) {
  int rc = make_split_dev(split, sp);
  if (rc) return rc;
  SPB_REQUIRE(covers_all(split), "spb_flatten_u8: the split must cover all %d taxa", sp->n);
  SPB_REQUIRE(d_s0 && rows_pad >= 1 && pitch >= 1, "spb_flatten_u8: bad buffers");
  SPB_REQUIRE(layout == SPB_S0_ROWMAJOR || layout == SPB_S0_TILED || layout == SPB_S0_K4MAJOR, "spb_flatten_u8: unknown layout %d",
              layout);
  if (layout == SPB_S0_ROWMAJOR) SPB_REQUIRE(pitch % 16 == 0, "spb_flatten_u8: row-major pitch must be a multiple of 16");
  else if (layout == SPB_S0_K4MAJOR)
    SPB_REQUIRE(pitch % 16 == 0 && rows_pad % 4 == 0, "spb_flatten_u8: k4-major layout needs pitch %% 16 == 0 and rows_pad %% 4 == 0");
  else SPB_REQUIRE(pitch % 128 == 0 && rows_pad % 128 == 0, "spb_flatten_u8: tiled layout needs rows_pad, pitch multiples of 128");
  SPB_REQUIRE((d_rank_r == nullptr) == (d_rank_c == nullptr), "spb_flatten_u8: give both rank arrays or neither");
  if (!d_rank_r) {
    SPB_REQUIRE(sp->a <= 15 && sp->b <= 15, "spb_flatten_u8: side too large without rank arrays");
    const int64_t cols = col_bound >= 0 && col_bound < (1ll << (2 * sp->b)) ? col_bound : (1ll << (2 * sp->b));
    SPB_REQUIRE(rows_pad >= (1ll << (2 * sp->a)) && pitch >= cols, "spb_flatten_u8: s0 too small");
  }
  return SPB_OK;
}

static int u8_batch_common(const uint64_t* d_keys, const uint32_t* d_counts, int64_t num, const spb_split* h_splits, int nb,
                           const uint32_t* d_rank_r, const uint32_t* d_rank_c, const uint32_t* d_colrank, int64_t cr_words,
                           uint8_t* d_s0, int64_t s0_stride, int64_t rows_pad, int64_t pitch, int layout, int flags, int32_t* d_hi_rc,
                           uint32_t* d_hi_val, uint32_t* d_hi_num, int64_t hi_cap, bool clear, cudaStream_t st) {
  SPB_REQUIRE(h_splits && nb >= 1 && nb <= SPB_MAX_BATCH, "spb_flatten_u8: batch size must be 1..%d (got %d)", SPB_MAX_BATCH, nb);
  SPB_REQUIRE(nb == 1 || (s0_stride >= rows_pad * pitch && !d_rank_r), "spb_flatten_u8: bad batch stride / rank arrays in a batch");
  SPB_REQUIRE(!d_colrank || !d_rank_r, "spb_flatten_u8: column ranks and reduced-format rank arrays exclude each other");
  SplitBatch sb;
  for (int b = 0; b < nb; ++b) {
    // ranked columns: at most min(4^b, num) of them are occupied
    int rc = u8_check(h_splits + b, &sb.s[b], d_rank_r, d_rank_c, d_s0, rows_pad, pitch, layout, d_colrank ? (num > 0 ? num : 0) : -1);
    if (rc) return rc;
    if (d_colrank)
      SPB_REQUIRE(cr_words == ((1ll << (2 * sb.s[b].b)) + 31) / 32, "spb_flatten_u8: column-rank words %lld do not match 4^%d columns",
                  (long long)cr_words, sb.s[b].b);
  }
  if (!clear) {
    SPB_REQUIRE(d_hi_rc && d_hi_val && d_hi_num, "spb_flatten_u8: NULL high-part buffers");
    if (!(flags & SPB_U8_NO_MEMSET)) {
      for (int b = 0; b < nb; ++b) SPB_CUDA(cudaMemsetAsync(d_s0 + (size_t)b * s0_stride, 0, (size_t)rows_pad * (size_t)pitch, st));
    }
    SPB_CUDA(cudaMemsetAsync(d_hi_num, 0, 4 * (size_t)nb, st));
  }
  if (num <= 0) return SPB_OK;
  SPB_REQUIRE(d_keys && (clear || d_counts), "spb_flatten_u8: NULL pattern table");
  dim3 grid(nblk(num, 256), (unsigned)nb);
  u8_kernel<<<grid, 256, 0, st>>>(d_keys, clear ? nullptr : d_counts, num, sb, d_rank_r, d_rank_c, d_colrank, cr_words, d_s0, s0_stride,
                                  rows_pad, pitch, layout, d_hi_rc, d_hi_val, d_hi_num, hi_cap);
  SPB_LAUNCH_CHECK();
  return SPB_OK;
}

extern "C" int spb_flatten_u8_batch(const uint64_t* d_keys, const uint32_t* d_counts, int64_t num, const spb_split* h_splits, int nb,
                                    uint8_t* d_s0, int64_t s0_stride, int64_t rows_pad, int64_t pitch, int layout, int flags,
                                    int32_t* d_hi_rc, uint32_t* d_hi_val, uint32_t* d_hi_num, int64_t hi_cap, void* stream) {
  return u8_batch_common(d_keys, d_counts, num, h_splits, nb, nullptr, nullptr, nullptr, 0, d_s0, s0_stride, rows_pad, pitch, layout,
                         flags, d_hi_rc, d_hi_val, d_hi_num, hi_cap, false, (cudaStream_t)stream);
}

extern "C" int spb_flatten_u8_clear_batch(const uint64_t* d_keys, int64_t num, const spb_split* h_splits, int nb, uint8_t* d_s0,
                                          int64_t s0_stride, int64_t rows_pad, int64_t pitch, int layout, void* stream) {
  return u8_batch_common(d_keys, nullptr, num, h_splits, nb, nullptr, nullptr, nullptr, 0, d_s0, s0_stride, rows_pad, pitch, layout, 0,
                         nullptr, nullptr, nullptr, 0, true, (cudaStream_t)stream);
}

extern "C" int spb_flatten_u8(const uint64_t* d_keys, const uint32_t* d_counts, int64_t num, const spb_split* split,
                              const uint32_t* d_rank_r, const uint32_t* d_rank_c, uint8_t* d_s0, int64_t rows_pad,
                              int64_t pitch, int layout, int flags, int32_t* d_hi_rc, uint32_t* d_hi_val, uint32_t* d_hi_num,
                              int64_t hi_cap, void* stream) {
  return u8_batch_common(d_keys, d_counts, num, split, 1, d_rank_r, d_rank_c, nullptr, 0, d_s0, rows_pad * pitch, rows_pad, pitch, layout,
                         flags, d_hi_rc, d_hi_val, d_hi_num, hi_cap, false, (cudaStream_t)stream);
}

extern "C" int spb_flatten_u8_clear(const uint64_t* d_keys, int64_t num, const spb_split* split, const uint32_t* d_rank_r,
                                    const uint32_t* d_rank_c, uint8_t* d_s0, int64_t rows_pad, int64_t pitch, int layout,
                                    void* stream) {
  return u8_batch_common(d_keys, nullptr, num, split, 1, d_rank_r, d_rank_c, nullptr, 0, d_s0, rows_pad * pitch, rows_pad, pitch, layout,
                         0, nullptr, nullptr, nullptr, 0, true, (cudaStream_t)stream);
}

extern "C" int64_t spb_col_rank_words(int b) { return ((1ll << (2 * b)) + 31) / 32; }

extern "C" int spb_col_ranks_batch(const uint64_t* d_keys, int64_t num, const spb_split* h_splits, int nb, uint32_t* d_colrank,
                                   int64_t words, int32_t* d_ncols, void* stream) {
  SPB_REQUIRE(h_splits && nb >= 1 && nb <= SPB_MAX_BATCH, "spb_col_ranks: batch size must be 1..%d (got %d)", SPB_MAX_BATCH, nb);
  SPB_REQUIRE(d_colrank && d_ncols && (num <= 0 || d_keys), "spb_col_ranks: NULL buffer");
  SplitBatch sb;
  for (int b = 0; b < nb; ++b) {
    int rc = make_split_dev(h_splits + b, &sb.s[b]);
    if (rc) return rc;
    SPB_REQUIRE(sb.s[b].b <= 15 && words == spb_col_rank_words(sb.s[b].b), "spb_col_ranks: %lld words do not match 4^%d columns",
                (long long)words, sb.s[b].b);
  }
  cudaStream_t st = (cudaStream_t)stream;
  SPB_CUDA(cudaMemsetAsync(d_colrank, 0, (size_t)nb * 2 * words * sizeof(uint32_t), st));
  if (num > 0) {
    col_mark_kernel<<<dim3(nblk(num, 256), (unsigned)nb), 256, 0, st>>>(d_keys, num, sb, d_colrank, words);
    SPB_LAUNCH_CHECK();
  }
  col_prefix_kernel<<<nb, kRankThreads, 0, st>>>(d_colrank, words, d_ncols);
  SPB_LAUNCH_CHECK();
  return SPB_OK;
}

extern "C" int spb_flatten_u8_batch_cols(const uint64_t* d_keys, const uint32_t* d_counts, int64_t num, const spb_split* h_splits, int nb,
                                         const uint32_t* d_colrank, int64_t words, uint8_t* d_s0, int64_t s0_stride, int64_t rows_pad,
                                         int64_t pitch, int layout, int flags, int32_t* d_hi_rc, uint32_t* d_hi_val, uint32_t* d_hi_num,
                                         int64_t hi_cap, void* stream) {
  SPB_REQUIRE(d_colrank, "spb_flatten_u8_batch_cols: NULL column ranks");
  return u8_batch_common(d_keys, d_counts, num, h_splits, nb, nullptr, nullptr, d_colrank, words, d_s0, s0_stride, rows_pad, pitch, layout,
                         flags, d_hi_rc, d_hi_val, d_hi_num, hi_cap, false, (cudaStream_t)stream);
}

extern "C" int spb_flatten_u8_clear_batch_cols(const uint64_t* d_keys, int64_t num, const spb_split* h_splits, int nb,
                                               const uint32_t* d_colrank, int64_t words, uint8_t* d_s0, int64_t s0_stride,
                                               int64_t rows_pad, int64_t pitch, int layout, void* stream) {
  SPB_REQUIRE(d_colrank, "spb_flatten_u8_clear_batch_cols: NULL column ranks");
  return u8_batch_common(d_keys, nullptr, num, h_splits, nb, nullptr, nullptr, d_colrank, words, d_s0, s0_stride, rows_pad, pitch, layout, 0,
                         nullptr, nullptr, nullptr, 0, true, (cudaStream_t)stream);
}

// Sparse flattenings: the product G Q = F (F^T Q) of the block-Krylov solver and the small Gram F F^T, from the pattern
// list of a split (one non-zero per distinct pattern), without materialising the flattening.  Layout: sparse.cuh.
//
// Segment sums.  Every output (a column of W = F^T Q, a row of AQ = F W) is the sum over one segment of the CSC / CSR
// entries.  Segment lengths are extremely skewed (a 2|18 split of 20 taxa has 16 rows of ~P/16 entries; a 10|10 split is
// close to a permutation), so a segment of L entries is cut into pieces at the global multiples of kSparsePiece:
// segment s owns pieces [s + off[s] / S, s + 1 + off[s + 1] / S), piece j of it covers the entries
// [max(off[s], (off[s] / S + j) S), min(off[s + 1], (off[s] / S + j + 1) S)) (the last one may be empty), so the piece
// numbering needs no prefix sum and the total is nseg + nnz / S.  Stage 1 (one thread per piece) sums its piece in
// entry order; a segment of one piece is written out directly, the others leave their partials.  Stage 2 (one warp per
// segment of several pieces) adds the partials, lane-strided and then by a fixed xor-shuffle tree.  No atomics: the
// result is bitwise reproducible, and exact when the values and Q are integers whose sums stay below 2^53.
#include "sparse.cuh"

namespace spb {
namespace {

__device__ __forceinline__ int64_t first_piece(const int64_t* off, int64_t s) { return s + off[s] / kSparsePiece; }

__device__ __forceinline__ void store_out(bool to_aq, double* out, int64_t s, int c, double v, int k, int64_t strideQ) {
  if (to_aq) {
    const int64_t b = s / k, r = s - b * k;
    out[b * strideQ + (int64_t)c * k + r] = v;
  } else {
    out[s * 8 + c] = v;
  }
}

// Stage 1: piece p of the segment list `off` (nseg segments): acc[c] = sum_e val[e] X[idx[e]][c], X rows of 64 bytes.
template <bool TO_AQ>
__global__ void __launch_bounds__(256) sparse_piece_kernel(const int64_t* __restrict__ off, const int32_t* __restrict__ idx,
                                                           const double* __restrict__ val, int64_t nseg, int64_t npieces,
                                                           const double* __restrict__ X, double* __restrict__ part,
                                                           double* __restrict__ out, int k, int64_t strideQ) {
  const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= npieces) return;
  int64_t lo = 0, hi = nseg - 1;  // the segment of p: the last s with first_piece(s) <= p (first_piece(0) = 0)
  while (lo < hi) {
    const int64_t mid = (lo + hi + 1) >> 1;
    if (first_piece(off, mid) <= p) lo = mid;
    else hi = mid - 1;
  }
  const int64_t s = lo;
  const int64_t o0 = off[s], o1 = off[s + 1];
  const int64_t first = s + o0 / kSparsePiece, count = s + 1 + o1 / kSparsePiece - first;
  const int64_t base = (o0 / kSparsePiece + (p - first)) * kSparsePiece;
  const int64_t e0 = base > o0 ? base : o0;
  const int64_t e1 = base + kSparsePiece < o1 ? base + kSparsePiece : o1;
  double acc[8];
#pragma unroll
  for (int c = 0; c < 8; ++c) acc[c] = 0.0;
#pragma unroll 4
  for (int64_t e = e0; e < e1; ++e) {
    const double v = __ldg(val + e);
    const double2* x = reinterpret_cast<const double2*>(X + (int64_t)__ldg(idx + e) * 8);
    const double2 x0 = __ldg(x), x1 = __ldg(x + 1), x2 = __ldg(x + 2), x3 = __ldg(x + 3);
    acc[0] = fma(v, x0.x, acc[0]); acc[1] = fma(v, x0.y, acc[1]);
    acc[2] = fma(v, x1.x, acc[2]); acc[3] = fma(v, x1.y, acc[3]);
    acc[4] = fma(v, x2.x, acc[4]); acc[5] = fma(v, x2.y, acc[5]);
    acc[6] = fma(v, x3.x, acc[6]); acc[7] = fma(v, x3.y, acc[7]);
  }
  if (count == 1) {
#pragma unroll
    for (int c = 0; c < 8; ++c) store_out(TO_AQ, out, s, c, acc[c], k, strideQ);
  } else {
    double2* dst = reinterpret_cast<double2*>(part + p * 8);
#pragma unroll
    for (int h = 0; h < 4; ++h) dst[h] = make_double2(acc[2 * h], acc[2 * h + 1]);
  }
}

// Stage 2: one warp per segment of several pieces.
template <bool TO_AQ>
__global__ void __launch_bounds__(256) sparse_combine_kernel(const int64_t* __restrict__ off, int64_t nseg, const double* __restrict__ part,
                                                             double* __restrict__ out, int k, int64_t strideQ) {
  const int64_t s = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (s >= nseg) return;
  const int64_t first = first_piece(off, s), count = first_piece(off, s + 1) - first;
  if (count == 1) return;
  double acc[8];
#pragma unroll
  for (int c = 0; c < 8; ++c) acc[c] = 0.0;
  for (int64_t q = lane; q < count; q += 32) {
    const double2* src = reinterpret_cast<const double2*>(part + (first + q) * 8);
#pragma unroll
    for (int h = 0; h < 4; ++h) {
      const double2 v = src[h];
      acc[2 * h] += v.x;
      acc[2 * h + 1] += v.y;
    }
  }
#pragma unroll
  for (int c = 0; c < 8; ++c)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc[c] += __shfl_xor_sync(0xFFFFFFFFu, acc[c], o);
  double mine = acc[0];
#pragma unroll
  for (int c = 1; c < 8; ++c) mine = lane == c ? acc[c] : mine;
  if (lane < 8) store_out(TO_AQ, out, s, lane, mine, k, strideQ);
}

// diag[s] = sum of v^2 over CSR row s: one warp per row, lane-strided, fixed xor-shuffle tree
__global__ void __launch_bounds__(256) sparse_diag_kernel(const int64_t* __restrict__ off, const double* __restrict__ val, int64_t nseg,
                                                          double* __restrict__ diag) {
  const int64_t s = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (s >= nseg) return;
  double acc = 0.0;
  for (int64_t e = off[s] + lane; e < off[s + 1]; e += 32) {
    const double v = val[e];
    acc = fma(v, v, acc);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xFFFFFFFFu, acc, o);
  if (lane == 0) diag[s] = acc;
}

template <bool TO_AQ>
int segment_product(const int64_t* off, const int32_t* idx, const double* val, int64_t nseg, int64_t nnz, const double* X, double* part,
                    double* out, int k, int64_t strideQ, cudaStream_t st) {
  if (nseg == 0) return SPB_OK;
  const int64_t npieces = nseg + nnz / kSparsePiece;
  sparse_piece_kernel<TO_AQ><<<(unsigned)((npieces + 255) / 256), 256, 0, st>>>(off, idx, val, nseg, npieces, X, part, out, k, strideQ);
  SPB_LAUNCH_CHECK();
  sparse_combine_kernel<TO_AQ><<<(unsigned)((nseg * 32 + 255) / 256), 256, 0, st>>>(off, nseg, part, out, k, strideQ);
  SPB_LAUNCH_CHECK();
  return SPB_OK;
}

// ------------------------------------------------------------------------------------------
// Small Gram side (k <= 128): G_b = F_b F_b^T from the CSC.  A CTA owns kGramChunk consecutive columns of one matrix and
// scatters them, kGramTile at a time, into a dense k x kGramTile tile in shared memory (entries of a column have distinct
// rows: plain stores); every thread keeps a (16 MA) / 16 x (16 MA) / 16 register block of G.  The CTA partials go to
// part[b][chunk][k][k] and are added in chunk order (deterministic, exact for integer values).
// ------------------------------------------------------------------------------------------
constexpr int kGramChunk = 8192;
constexpr int kGramTile = 32;
constexpr int kGramMaxK = 128;

template <int MA>
__global__ void __launch_bounds__(256) sparse_gram_small_kernel(const int64_t* __restrict__ col_off, const int32_t* __restrict__ col_row,
                                                                const double* __restrict__ col_val, const int64_t* __restrict__ colbase,
                                                                int k, int nchunks, double* __restrict__ part) {
  __shared__ double tile[16 * MA][kGramTile + 1];
  const int b = blockIdx.y, tid = threadIdx.x;
  const int ti = tid >> 4, tj = tid & 15;
  const int64_t c_begin = colbase[b] + (int64_t)blockIdx.x * kGramChunk;
  const int64_t c_lim = colbase[b + 1];
  const int64_t c_end = c_begin + kGramChunk < c_lim ? c_begin + kGramChunk : c_lim;
  const int64_t row0 = (int64_t)b * k;
  double acc[MA][MA];
#pragma unroll
  for (int a = 0; a < MA; ++a)
#pragma unroll
    for (int q = 0; q < MA; ++q) acc[a][q] = 0.0;
  for (int64_t c0 = c_begin; c0 < c_end; c0 += kGramTile) {
    const int cn = (int)(c_end - c0 < kGramTile ? c_end - c0 : kGramTile);
    for (int i = tid; i < 16 * MA * kGramTile; i += 256) tile[i / kGramTile][i % kGramTile] = 0.0;
    __syncthreads();
    if (tid < cn) {
      for (int64_t e = col_off[c0 + tid]; e < col_off[c0 + tid + 1]; ++e) tile[col_row[e] - row0][tid] = col_val[e];
    }
    __syncthreads();
#pragma unroll 4
    for (int t = 0; t < kGramTile; ++t) {
      double x[MA], y[MA];
#pragma unroll
      for (int a = 0; a < MA; ++a) { x[a] = tile[ti + 16 * a][t]; y[a] = tile[tj + 16 * a][t]; }
#pragma unroll
      for (int a = 0; a < MA; ++a)
#pragma unroll
        for (int q = 0; q < MA; ++q) acc[a][q] = fma(x[a], y[q], acc[a][q]);
    }
    __syncthreads();
  }
  double* out = part + ((int64_t)b * nchunks + blockIdx.x) * k * k;
#pragma unroll
  for (int a = 0; a < MA; ++a)
#pragma unroll
    for (int q = 0; q < MA; ++q) {
      const int i = ti + 16 * a, j = tj + 16 * q;
      if (i < k && j < k) out[i * k + j] = acc[a][q];
    }
}

__global__ void sparse_gram_reduce_kernel(const double* __restrict__ part, int k, int nchunks, double* __restrict__ G) {
  const int b = blockIdx.y;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= k * k) return;
  double s = 0.0;
  for (int ch = 0; ch < nchunks; ++ch) s += part[((int64_t)b * nchunks + ch) * k * k + i];
  G[(int64_t)b * k * k + i] = s;
}

inline int gram_chunks(int64_t max_cols) { return (int)((max_cols + kGramChunk - 1) / kGramChunk) > 0 ? (int)((max_cols + kGramChunk - 1) / kGramChunk) : 1; }

}  // namespace

int sparse_check(const SparseBatch& f) {
  SPB_REQUIRE(f.row_off && f.col_off && f.k >= 1 && f.batch >= 1 && f.batch <= 65535 && f.ncols >= 0 && f.nnz >= 0 &&
                  (int64_t)f.batch * f.k < (1ll << 31) && f.ncols < (1ll << 31) &&
                  (f.nnz == 0 || (f.row_col && f.row_val && f.col_row && f.col_val)),
              "sparse flattening batch: bad arguments (k=%d batch=%d ncols=%lld nnz=%lld)", f.k, f.batch, (long long)f.ncols,
              (long long)f.nnz);
  return SPB_OK;
}

int sparse_product_launch(const SparseBatch& f, const double* Qt, double* W, double* AQ, int64_t strideQ, double* part, cudaStream_t st) {
  int rc = segment_product<false>(f.col_off, f.col_row, f.col_val, f.ncols, f.nnz, Qt, part, W, f.k, 0, st);
  if (rc) return rc;
  return segment_product<true>(f.row_off, f.row_col, f.row_val, (int64_t)f.batch * f.k, f.nnz, W, part, AQ, f.k, strideQ, st);
}

int sparse_diag_launch(const SparseBatch& f, double* diag, cudaStream_t st) {
  const int64_t nseg = (int64_t)f.batch * f.k;
  sparse_diag_kernel<<<(unsigned)((nseg * 32 + 255) / 256), 256, 0, st>>>(f.row_off, f.row_val, nseg, diag);
  SPB_LAUNCH_CHECK();
  return SPB_OK;
}

}  // namespace spb

using namespace spb;

extern "C" int64_t spb_sparse_gram_small_ws(int64_t k, int64_t batch, int64_t max_cols) {
  return (int64_t)gram_chunks(max_cols) * batch * k * k;
}

extern "C" int spb_sparse_gram_small(const int64_t* d_col_off, const int32_t* d_col_row, const double* d_col_val, const int64_t* d_colbase,
                                     int64_t k, int64_t batch, int64_t max_cols, double* d_G, double* d_ws, void* stream) {
  SPB_REQUIRE(d_col_off && d_colbase && d_G && d_ws && k >= 1 && k <= kGramMaxK && batch >= 1 && batch <= 65535 && max_cols >= 0 &&
                  batch * k < (1ll << 31),
              "spb_sparse_gram_small: need 1 <= k <= %d (got %lld)", kGramMaxK, (long long)k);
  cudaStream_t st = (cudaStream_t)stream;
  const int nchunks = gram_chunks(max_cols);
  dim3 grid(nchunks, (unsigned)batch);
  const int ma = (int)((k + 15) / 16);
  switch (ma) {
#define SPB_SG(M_) case M_: sparse_gram_small_kernel<M_><<<grid, 256, 0, st>>>(d_col_off, d_col_row, d_col_val, d_colbase, (int)k, nchunks, d_ws); break;
    SPB_SG(1) SPB_SG(2) SPB_SG(3) SPB_SG(4) SPB_SG(5) SPB_SG(6) SPB_SG(7) SPB_SG(8)
#undef SPB_SG
  }
  SPB_LAUNCH_CHECK();
  dim3 rg((unsigned)((k * k + 255) / 256), (unsigned)batch);
  sparse_gram_reduce_kernel<<<rg, 256, 0, st>>>(d_ws, (int)k, nchunks, d_G);
  SPB_LAUNCH_CHECK();
  return SPB_OK;
}

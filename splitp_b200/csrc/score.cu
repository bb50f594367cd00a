// Split score (splitp/phylogenetics.py:280-328) from Gram matrices.
//
//   score = sqrt(1 - sum_{i<4} sigma_i^2 / sum_i sigma_i^2),  sigma = singular values of the (sub)flattening
//
// sigma_i^2 are the eigenvalues of G = F F^T.  Small G (k <= 128) goes through the shared-memory Jacobi
// solver and the trailing eigenvalues are summed directly.  Large G (the 4096 x 4096 Gram of a dense 6|6
// flattening) is reduced to a <= 96 x 96 Rayleigh-Ritz problem by a block-Krylov iteration with full
// re-orthogonalisation (fp64), whose projected matrix is again solved by the same Jacobi routine; the
// total is trace(G) = ||F||_F^2.
#include "common.cuh"
#include "jacobi.cuh"
#include "sparse.cuh"
#include <vector>

using namespace spb;

namespace {

// ------------------------------------------------------------------------------------------
// Batched fp64 GEMM, C[M][N] = A[M][K] * B[N][K]^T ("NT": both operands K-contiguous), optional split-K
// into a partial workspace (summed in a fixed order by reduce_kernel => deterministic).
// ------------------------------------------------------------------------------------------
constexpr int kBK = 16;

template <int BM, int BN, int TM, int TN>
__global__ void __launch_bounds__(256) gemm_nt_kernel(const double* __restrict__ A, int64_t lda, int64_t strideA,
                                                      const double* __restrict__ B, int64_t ldb, int64_t strideB,
                                                      double* __restrict__ C, int64_t ldc, int64_t strideC, int M, int N, int K,
                                                      int ksplit, int kchunk) {
  static_assert((BM / TM) * (BN / TN) == 256, "256 threads");
  constexpr int TX = BN / TN;  // threads along N
  __shared__ double As[kBK][BM + 2];
  __shared__ double Bs[kBK][BN + 2];
  const int tid = threadIdx.x;
  const int tx = tid % TX, ty = tid / TX;
  const int bt = blockIdx.z / ksplit, ks = blockIdx.z - bt * ksplit;
  const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
  const double* Ab = A + (int64_t)bt * strideA;
  const double* Bb = B + (int64_t)bt * strideB;
  const int kbeg = ks * kchunk;
  const int kend = min(K, kbeg + kchunk);
  double acc[TM][TN];
#pragma unroll
  for (int i = 0; i < TM; ++i)
#pragma unroll
    for (int j = 0; j < TN; ++j) acc[i][j] = 0.0;

  for (int k0 = kbeg; k0 < kend; k0 += kBK) {
    // tile loads: element (row r, k kk) for r < BM (A) / BN (B), kk < 16; consecutive threads walk k
    for (int idx = tid; idx < BM * kBK; idx += 256) {
      int r = idx / kBK, kk = idx - r * kBK;
      int gm = m0 + r, gk = k0 + kk;
      As[kk][r] = (gm < M && gk < kend) ? Ab[(int64_t)gm * lda + gk] : 0.0;
    }
    for (int idx = tid; idx < BN * kBK; idx += 256) {
      int r = idx / kBK, kk = idx - r * kBK;
      int gn = n0 + r, gk = k0 + kk;
      Bs[kk][r] = (gn < N && gk < kend) ? Bb[(int64_t)gn * ldb + gk] : 0.0;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < kBK; ++kk) {
      double a[TM], b[TN];
#pragma unroll
      for (int i = 0; i < TM; ++i) a[i] = As[kk][ty + i * (BM / TM)];
#pragma unroll
      for (int j = 0; j < TN; ++j) b[j] = Bs[kk][tx + j * TX];
#pragma unroll
      for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] = fma(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
  double* Cb = C + (int64_t)blockIdx.z * strideC;  // partial index = bt*ksplit + ks (strideC = M*N region when split)
#pragma unroll
  for (int i = 0; i < TM; ++i) {
    int gm = m0 + ty + i * (BM / TM);
    if (gm >= M) continue;
#pragma unroll
    for (int j = 0; j < TN; ++j) {
      int gn = n0 + tx + j * TX;
      if (gn < N) Cb[(int64_t)gm * ldc + gn] = acc[i][j];
    }
  }
}

// C[bt][i] = sum_ks part[(bt*ksplit+ks)][i]  (fixed order)
__global__ void reduce_kernel(const double* __restrict__ part, int64_t elems, int ksplit, double* __restrict__ C, int64_t strideC,
                              int M, int N, int64_t ldc) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int bt = blockIdx.y;
  if (i >= elems) return;
  double s = 0.0;
  for (int ks = 0; ks < ksplit; ++ks) s += part[((int64_t)bt * ksplit + ks) * elems + i];
  int r = (int)(i / N), c = (int)(i - (int64_t)r * N);
  C[(int64_t)bt * strideC + (int64_t)r * ldc + c] = s;
}

// Tall-skinny inner products of the Krylov solver: C[m][n] = sum_pos A[m][pos] * B[n][pos], M, N <= 96, K = k long.
// One CTA = one chunk of kDotChunk positions of one matrix: both operand panels are staged in shared memory with
// coalesced loads and every thread owns the outputs (ti + 16 a, tj + 16 b).  Partials go to part[(bt, chunk)][M][N]
// and are summed in chunk order by reduce_kernel (deterministic).
constexpr int kDotChunk = 128;
template <int MA, int NB>  // output register block per thread: rows ti + 16 a (a < MA), columns tj + 16 b (b < NB)
__global__ void __launch_bounds__(256) dot_kernel(const double* __restrict__ A, int64_t strideA, const double* __restrict__ B,
                                                  int64_t strideB, int M, int N, int k, int nchunks, double* __restrict__ part) {
  extern __shared__ __align__(16) double s_dot[];  // A panel [M][kDotChunk + 1], B panel [N][kDotChunk + 1]
  const int ldp = kDotChunk + 1;
  double* sA = s_dot;
  double* sB = s_dot + M * ldp;
  const int bt = blockIdx.y, ch = blockIdx.x;
  const int pos0 = ch * kDotChunk;
  const int len = min(kDotChunk, k - pos0);
  const double* Ab = A + (int64_t)bt * strideA;
  const double* Bb = B + (int64_t)bt * strideB;
  for (int idx = threadIdx.x; idx < M * kDotChunk; idx += 256) {
    int r = idx / kDotChunk, p = idx - r * kDotChunk;
    sA[r * ldp + p] = p < len ? Ab[(int64_t)r * k + pos0 + p] : 0.0;
  }
  for (int idx = threadIdx.x; idx < N * kDotChunk; idx += 256) {
    int r = idx / kDotChunk, p = idx - r * kDotChunk;
    sB[r * ldp + p] = p < len ? Bb[(int64_t)r * k + pos0 + p] : 0.0;
  }
  __syncthreads();
  const int ti = threadIdx.x >> 4, tj = threadIdx.x & 15;
  double acc[MA][NB];
  const double* xa[MA];
  const double* yb[NB];
#pragma unroll
  for (int a = 0; a < MA; ++a) {
    xa[a] = sA + min(ti + 16 * a, M - 1) * ldp;  // clamped rows are computed but never stored
#pragma unroll
    for (int b = 0; b < NB; ++b) acc[a][b] = 0.0;
  }
#pragma unroll
  for (int b = 0; b < NB; ++b) yb[b] = sB + min(tj + 16 * b, N - 1) * ldp;
#pragma unroll 4
  for (int p = 0; p < kDotChunk; ++p) {
    double x[MA], y[NB];
#pragma unroll
    for (int a = 0; a < MA; ++a) x[a] = xa[a][p];
#pragma unroll
    for (int b = 0; b < NB; ++b) y[b] = yb[b][p];
#pragma unroll
    for (int a = 0; a < MA; ++a)
#pragma unroll
      for (int b = 0; b < NB; ++b) acc[a][b] = fma(x[a], y[b], acc[a][b]);
  }
  double* out = part + ((int64_t)bt * nchunks + ch) * M * N;
#pragma unroll
  for (int a = 0; a < MA; ++a)
#pragma unroll
    for (int b = 0; b < NB; ++b) {
      int i = ti + 16 * a, j = tj + 16 * b;
      if (i < M && j < N) out[i * N + j] = acc[a][b];
    }
}

// D (8 x 8, fp64) += A (8 x 4) B (4 x 8) on the fp64 tensor cores.  Fragments (PTX m8n8k4 .f64): lane l holds A[l / 4][l % 4],
// B[l % 4][l / 4] and D[l / 4][2 (l % 4) + {0, 1}].
__device__ __forceinline__ void dmma884(double& d0, double& d1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};" : "+d"(d0), "+d"(d1) : "d"(a), "d"(b));
}

// The same inner products for M, N in {8, 16} (every product of the two-block Krylov cycle) on the fp64 tensor cores: ONE CTA per
// matrix, its 8 warps split the k positions, a lane loads 4 consecutive doubles of row l / 4 of every 8-row tile of A and of B
// per 16 positions (element t = k-slot l % 4 of MMA t), the warps' 8 x 8 tiles are added in warp order.  No partial buffer and
// no reduce launch: 63 + 63 launches of the c2 step (35 + 5 us each at 64 matrices) become 63.
template <int MT, int NT>
__global__ void __launch_bounds__(256) dot_dmma_kernel(const double* __restrict__ A, int64_t strideA, const double* __restrict__ B,
                                                       int64_t strideB, int k, double* __restrict__ Cout, int64_t ldc, int64_t strideC) {
  __shared__ double red[8][8 * MT][8 * NT];
  const int bt = blockIdx.x;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int kq = lane & 3, grp = lane >> 2;
  const double* Ab = A + (int64_t)bt * strideA + (int64_t)grp * k + 4 * kq;
  const double* Bb = B + (int64_t)bt * strideB + (int64_t)grp * k + 4 * kq;
  double acc[MT][NT][2];
#pragma unroll
  for (int a = 0; a < MT; ++a)
#pragma unroll
    for (int b = 0; b < NT; ++b) acc[a][b][0] = acc[a][b][1] = 0.0;
  const int per_warp = k / 8;  // a multiple of 16 (launcher)
  const int p_end = (warp + 1) * per_warp;
#pragma unroll 2
  for (int p = warp * per_warp; p < p_end; p += 16) {
    double2 a01[MT], a23[MT], b01[NT], b23[NT];
#pragma unroll
    for (int a = 0; a < MT; ++a) {
      a01[a] = *reinterpret_cast<const double2*>(Ab + (int64_t)(8 * a) * k + p);
      a23[a] = *reinterpret_cast<const double2*>(Ab + (int64_t)(8 * a) * k + p + 2);
    }
#pragma unroll
    for (int b = 0; b < NT; ++b) {
      b01[b] = *reinterpret_cast<const double2*>(Bb + (int64_t)(8 * b) * k + p);
      b23[b] = *reinterpret_cast<const double2*>(Bb + (int64_t)(8 * b) * k + p + 2);
    }
#pragma unroll
    for (int a = 0; a < MT; ++a)
#pragma unroll
      for (int b = 0; b < NT; ++b) {
        dmma884(acc[a][b][0], acc[a][b][1], a01[a].x, b01[b].x);
        dmma884(acc[a][b][0], acc[a][b][1], a01[a].y, b01[b].y);
        dmma884(acc[a][b][0], acc[a][b][1], a23[a].x, b23[b].x);
        dmma884(acc[a][b][0], acc[a][b][1], a23[a].y, b23[b].y);
      }
  }
#pragma unroll
  for (int a = 0; a < MT; ++a)
#pragma unroll
    for (int b = 0; b < NT; ++b) {
      red[warp][8 * a + grp][8 * b + 2 * kq] = acc[a][b][0];
      red[warp][8 * a + grp][8 * b + 2 * kq + 1] = acc[a][b][1];
    }
  __syncthreads();
  if (threadIdx.x < 64 * MT * NT) {
    const int i = threadIdx.x / (8 * NT), j = threadIdx.x - i * (8 * NT);
    double v = 0.0;
#pragma unroll
    for (int w = 0; w < 8; ++w) v += red[w][i][j];
    Cout[(int64_t)bt * strideC + (int64_t)i * ldc + j] = v;
  }
}

struct GemmArgs {
  const double* A; int64_t lda, strideA;
  const double* B; int64_t ldb, strideB;
  double* C; int64_t ldc, strideC;
  int M, N, K, batch;
};

static int gemm_nt(const GemmArgs& g, int ksplit, double* part, cudaStream_t st) {
  if (g.M <= 0 || g.N <= 0 || g.batch <= 0) return SPB_OK;
  if (ksplit < 1) ksplit = 1;
  int kchunk = ((g.K + ksplit - 1) / ksplit + kBK - 1) / kBK * kBK;
  if (kchunk < kBK) kchunk = kBK;
  ksplit = (g.K + kchunk - 1) / kchunk;
  if (ksplit < 1) ksplit = 1;
  double* out = g.C; int64_t ldc = g.ldc, strideC = g.strideC;
  if (ksplit > 1) { out = part; ldc = g.N; strideC = (int64_t)g.M * g.N; }
  dim3 grid((g.N + 63) / 64, (g.M + 63) / 64, g.batch * ksplit);
  gemm_nt_kernel<64, 64, 4, 4><<<grid, 256, 0, st>>>(g.A, g.lda, g.strideA, g.B, g.ldb, g.strideB, out, ldc, strideC, g.M, g.N, g.K,
                                                     ksplit, kchunk);
  SPB_LAUNCH_CHECK();
  if (ksplit > 1) {
    int64_t elems = (int64_t)g.M * g.N;
    dim3 rg((unsigned)((elems + 255) / 256), g.batch);
    reduce_kernel<<<rg, 256, 0, st>>>(part, elems, ksplit, g.C, g.strideC, g.M, g.N, g.ldc);
    SPB_LAUNCH_CHECK();
  }
  return SPB_OK;
}

// NOTE on strides with split-K: partial (bt, ks) lives at part[(bt*ksplit+ks)*M*N]; the kernel indexes C by
// blockIdx.z = bt*ksplit+ks with strideC = M*N, which is exactly that layout.  Without split-K blockIdx.z = bt.

static int choose_ksplit(int M, int N, int K, int batch) {
  int64_t tiles = (int64_t)((N + 63) / 64) * ((M + 63) / 64) * batch;
  int target = 2 * sm_count();
  if (tiles >= target) return 1;
  int ks = (int)((target + tiles - 1) / tiles);
  int maxks = K / 256;
  if (maxks < 1) maxks = 1;
  if (ks > maxks) ks = maxks;
  if (ks > 64) ks = 64;
  return ks;
}

// C (ldc, strideC) = A B^T for the tall-skinny Krylov operands; part must hold batch * ceil(k/128) * M * N doubles
static int dot_product(const double* A, int64_t strideA, const double* B, int64_t strideB, int M, int N, int k, int batch,
                       double* C, int64_t ldc, int64_t strideC, double* part, cudaStream_t st) {
  if ((M == 8 || M == 16) && (N == 8 || N == 16) && k % 128 == 0 && strideA % 2 == 0 && strideB % 2 == 0 &&
      reinterpret_cast<uintptr_t>(A) % 16 == 0 && reinterpret_cast<uintptr_t>(B) % 16 == 0) {
    if (M == 8 && N == 8) dot_dmma_kernel<1, 1><<<batch, 256, 0, st>>>(A, strideA, B, strideB, k, C, ldc, strideC);
    else if (M == 16 && N == 8) dot_dmma_kernel<2, 1><<<batch, 256, 0, st>>>(A, strideA, B, strideB, k, C, ldc, strideC);
    else if (M == 8 && N == 16) dot_dmma_kernel<1, 2><<<batch, 256, 0, st>>>(A, strideA, B, strideB, k, C, ldc, strideC);
    else dot_dmma_kernel<2, 2><<<batch, 256, 0, st>>>(A, strideA, B, strideB, k, C, ldc, strideC);
    SPB_LAUNCH_CHECK();
    return SPB_OK;
  }
  const int nchunks = (k + kDotChunk - 1) / kDotChunk;
  const size_t smem = (size_t)(M + N) * (kDotChunk + 1) * sizeof(double);
  dim3 grid(nchunks, batch);
  const int ma = (M + 15) >> 4, nb = (N + 15) >> 4;
#define SPB_DOT(MA_, NB_)                                                                                           \
  do {                                                                                                              \
    SPB_CUDA(cudaFuncSetAttribute(dot_kernel<MA_, NB_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));   \
    dot_kernel<MA_, NB_><<<grid, 256, smem, st>>>(A, strideA, B, strideB, M, N, k, nchunks, part);                  \
  } while (0)
  if (ma <= 1 && nb <= 1) SPB_DOT(1, 1);
  else if (ma <= 2 && nb <= 1) SPB_DOT(2, 1);
  else if (nb <= 1) SPB_DOT(6, 1);
  else if (ma <= 2 && nb <= 2) SPB_DOT(2, 2);
  else SPB_DOT(6, 6);
#undef SPB_DOT
  SPB_LAUNCH_CHECK();
  const int64_t elems = (int64_t)M * N;
  dim3 rg((unsigned)((elems + 255) / 256), batch);
  reduce_kernel<<<rg, 256, 0, st>>>(part, elems, nchunks, C, strideC, M, N, ldc);
  SPB_LAUNCH_CHECK();
  return SPB_OK;
}

// ------------------------------------------------------------------------------------------
// small path: Jacobi on the k x k Gram directly
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) score_small_kernel(const double* __restrict__ G, int k, int64_t ld, int64_t batch,
                                                          double* scores, double* eig) {
  extern __shared__ __align__(16) double s_A[];
  __shared__ JacobiScratch js;
  __shared__ double lam[kJacobiMaxK], tmp[kJacobiMaxK];
  const int m = jacobi_dim(k), lda = jacobi_ld(k);
  for (int64_t bt = blockIdx.x; bt < batch; bt += gridDim.x) {
    __syncthreads();
    const double* Gb = G + bt * ld * ld;
    for (int idx = threadIdx.x; idx < m * m; idx += blockDim.x) {
      int r = idx / m, c = idx - r * m;
      // symmetrise on load: the callers' Gram matrices are symmetric up to rounding; zero padding when k is odd
      s_A[r * lda + c] = (r < k && c < k) ? 0.5 * (Gb[(int64_t)r * ld + c] + Gb[(int64_t)c * ld + r]) : 0.0;
    }
    __syncthreads();
    jacobi_eig_smem(s_A, lda, k, nullptr, 0, &js);
    sort_diag_desc(s_A, lda, k, tmp, lam);
    if (threadIdx.x == 0) scores[bt] = (k <= 4) ? (lam[0] > 0.0 || k > 1 ? 0.0 : 0.0) : score_from_sorted(lam, k);
    if (eig) for (int i = threadIdx.x; i < k; i += blockDim.x) eig[bt * k + i] = lam[i];
  }
}

// ------------------------------------------------------------------------------------------
// large path: restarted block Krylov + Rayleigh-Ritz (all kernels batched over matrices)
//
// One cycle: Q_0 (8 x k, orthonormal) -> for j < nb: AQ_j = Q_j G (symv_block_kernel, HBM-bound: G is read once
// per block), next block = AQ_j orthogonalised twice against all previous blocks (classical Gram-Schmidt x2) and
// orthonormalised by SVQB; T = Q AQ^T (dim x dim, dim = 8 nb <= 96) is diagonalised by the shared-memory Jacobi
// solver WITH eigenvectors; the top-8 Ritz vectors (in place of Q_0) restart the next cycle and the residuals
// ||G y - theta y|| / theta_0 of the top 4 measure convergence.  The first cycle starts from the 8 heaviest rows of G
// (krylov_top8_kernel).  The host loop (spb_score_gram_large) runs cycles of 2, 2, 4, 4, 12, ... blocks until every
// matrix of the batch passes the Kato-Temple test: flattenings of alignments (spectrum decaying by 10^-3 .. 10^-7
// after the 4th eigenvalue) pass after one 16-dimensional cycle, i.e. after reading G twice; flat random spectra
// take a few larger cycles (tests/test_gpu_parity.py::test_split_score_flat_spectrum).
// ------------------------------------------------------------------------------------------
constexpr int kKB = 8;        // block size
constexpr int kKMaxBlocks = 12;
constexpr int kKDim = kKB * kKMaxBlocks;  // 96
constexpr int kInfo = 10;     // per-matrix status: top4, trace, residual, dim, cycles, delta_top, theta_4, theta_5 (1-based),
                              // converged (1 = passed the acceptance test, 0 = cycle budget exhausted), reserved
constexpr int kHeavyStart = 4;  // start block: this many heaviest rows of G, the remaining kKB - kHeavyStart vectors pseudo-random

// The matrix the Krylov solver works on: either fp64 G, or the exact 32-bit integer Gram G0 of the low bytes plus
// the high-part correction C kept as a strip of its m non-zero rows (gram.cu, "hi_strip"):
//   G = G0 + C,   C[i][j] = Cs[pos[i]][j] if pos[i] >= 0, else Cs[pos[j]][i] if pos[j] >= 0, else 0.
// The integer form halves the bytes every G Q product streams from HBM.
struct GramView {
  const double* Gf;    // [batch][ld][ld] or nullptr
  const int32_t* Gi;   // [batch][ld][ld] or nullptr
  int64_t ld;
  const double* Cs;    // [batch][cs_rows][ld]
  int64_t cs_rows;
  const int32_t* pos;  // [batch][ld]
  const int32_t* hr;   // [batch][cs_rows]
  const int32_t* hm;   // [batch]
};

__device__ __forceinline__ double view_entry(const GramView& g, int64_t bt, int64_t i, int64_t j) {
  if (g.Gf) return g.Gf[bt * g.ld * g.ld + i * g.ld + j];
  double v = (double)g.Gi[bt * g.ld * g.ld + i * g.ld + j];
  if (g.cs_rows) {
    const int32_t* pos = g.pos + bt * g.ld;
    const double* Cs = g.Cs + bt * g.cs_rows * g.ld;
    const int pi = pos[i];
    if (pi >= 0) v += Cs[(int64_t)pi * g.ld + j];
    else {
      const int pj = pos[j];
      if (pj >= 0) v += Cs[(int64_t)pj * g.ld + i];
    }
  }
  return v;
}

__global__ void gram_diag_kernel(const GramView g, int k, double* __restrict__ diag) {
  const int64_t bt = blockIdx.y;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < k) diag[bt * k + i] = view_entry(g, bt, i, i);
}

// Start block of the first cycle: the kHeavyStart rows of G with the largest diagonal entries, i.e. G e_j for the
// heaviest indices j, plus kKB - kHeavyStart pseudo-random vectors.  The heavy rows are columns of G, so the start
// block already contains one application of G at no cost, and for count flattenings they carry most of the dominant
// eigenvectors: 2 Krylov blocks from this start reach the residual that 4 to 8 blocks reach from a purely random start
// (12-taxon / 10^6-site Gram matrices).  The random vectors are what makes the solver correct on REDUCIBLE matrices
// (block-diagonal G, sparse flattenings with many components): rows of G never leave the connected components of
// their indices, so a start block made of rows only can converge -- with zero residual -- to the eigenpairs of a
// sub-matrix (e.g. blockdiag(20 I_8, ones(200, 200)): the 8 heaviest rows all lie in the first block).  A random vector
// has a component along every eigenvector with probability one, so a missed dominant direction shows up as a large
// residual and the cycle loop continues (tests/test_gpu_parity_r2.py::test_split_score_reducible_gram).
__global__ void __launch_bounds__(256) krylov_top8_kernel(const double* __restrict__ diag, int k, int* idx_out) {
  __shared__ double s_val[256];
  __shared__ int s_idx[256];
  __shared__ int chosen[kKB];
  const int64_t bt = blockIdx.x;
  const double* db = diag + bt * k;
  const int tid = threadIdx.x;
  for (int pick = 0; pick < kKB; ++pick) {
    double best = -1.0;
    int bi = -1;
    for (int i = tid; i < k; i += 256) {
      bool taken = false;
      for (int p = 0; p < pick; ++p) taken |= (chosen[p] == i);
      double v = taken ? -1.0 : fabs(db[i]);
      if (v > best) { best = v; bi = i; }
    }
    s_val[tid] = best; s_idx[tid] = bi;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
      if (tid < o) {
        // ties go to the smaller index: the result does not depend on the reduction order
        if (s_val[tid + o] > s_val[tid] || (s_val[tid + o] == s_val[tid] && s_idx[tid + o] >= 0 && (s_idx[tid] < 0 || s_idx[tid + o] < s_idx[tid]))) {
          s_val[tid] = s_val[tid + o]; s_idx[tid] = s_idx[tid + o];
        }
      }
      __syncthreads();
    }
    if (tid == 0) { chosen[pick] = s_idx[0] >= 0 ? s_idx[0] : pick; idx_out[bt * kKB + pick] = chosen[pick]; }
    __syncthreads();
  }
}

__global__ void krylov_start_rows_kernel(const GramView g, const int* __restrict__ idx, double* Q, int64_t strideQ, int k) {
  const int64_t bt = blockIdx.y;
  const int pos = blockIdx.x * blockDim.x + threadIdx.x;
  if (pos >= k) return;
#pragma unroll
  for (int c = 0; c < kHeavyStart; ++c) Q[bt * strideQ + (int64_t)c * k + pos] = view_entry(g, bt, idx[bt * kKB + c], pos);
#pragma unroll
  for (int c = kHeavyStart; c < kKB; ++c) {
    // counter-based pseudo-random entry in (-1, 1): depends only on (vector, position), so the result is reproducible
    // and independent of the batch composition; SVQB normalises the block afterwards
    const uint64_t hsh = mix64(((uint64_t)c << 40) ^ (uint64_t)pos ^ 0x9E3779B97F4A7C15ull);
    Q[bt * strideQ + (int64_t)c * k + pos] = (double)(int64_t)(hsh >> 11) * (1.0 / 4503599627370496.0) - 1.0;
  }
}

// Start block of the sparse operator (no entry of G can be read directly): unit vectors e_j of the kHeavyStart heaviest
// rows, multiplied by G afterwards (krylov_cycle), plus the same pseudo-random vectors as krylov_start_rows_kernel.
__global__ void krylov_start_sparse_kernel(const int* __restrict__ idx, double* Q, int64_t strideQ, int k) {
  const int64_t bt = blockIdx.y;
  const int pos = blockIdx.x * blockDim.x + threadIdx.x;
  if (pos >= k) return;
#pragma unroll
  for (int c = 0; c < kHeavyStart; ++c) Q[bt * strideQ + (int64_t)c * k + pos] = idx[bt * kKB + c] == pos ? 1.0 : 0.0;
#pragma unroll
  for (int c = kHeavyStart; c < kKB; ++c) {
    const uint64_t hsh = mix64(((uint64_t)c << 40) ^ (uint64_t)pos ^ 0x9E3779B97F4A7C15ull);
    Q[bt * strideQ + (int64_t)c * k + pos] = (double)(int64_t)(hsh >> 11) * (1.0 / 4503599627370496.0) - 1.0;
  }
}

// AQ[c][i] = sum_j G[i][j] Q[c][j], c < 8.  CTA = 32 rows of G; warp = 4 rows processed together; every lane owns two
// adjacent columns (128-bit loads of G and of the staged Q chunk: 8 x 16 bytes in flight per lane and iteration).
// The Q chunk (8 x 1024 doubles, 64 KB) is staged in shared memory and reused by all 32 rows.
constexpr int kSymvRows = 32;
constexpr int kSymvChunk = 1024;
__global__ void __launch_bounds__(256, 2) symv_block_kernel(const double* __restrict__ G, int64_t ld, int64_t strideG,
                                                         const double* __restrict__ Q, int64_t strideQ, double* __restrict__ AQ,
                                                         int k) {
  extern __shared__ __align__(16) double s_q[];  // [kKB][kSymvChunk]
  const int bt = blockIdx.y;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int row0 = blockIdx.x * kSymvRows + warp * 4;
  const double* Gb = G + (int64_t)bt * strideG;
  const double* Qb = Q + (int64_t)bt * strideQ;
  const bool vec_ok = ((ld & 1) == 0) && ((reinterpret_cast<uintptr_t>(Gb) & 15) == 0);  // 16-byte aligned row starts
  double acc[4][kKB];
#pragma unroll
  for (int r = 0; r < 4; ++r)
#pragma unroll
    for (int c = 0; c < kKB; ++c) acc[r][c] = 0.0;
  for (int j0 = 0; j0 < k; j0 += kSymvChunk) {
    const int len = min(kSymvChunk, k - j0);
    __syncthreads();
    for (int idx = threadIdx.x; idx < kKB * kSymvChunk; idx += 256) {
      int c = idx / kSymvChunk, j = idx - c * kSymvChunk;
      s_q[idx] = (j < len) ? Qb[(int64_t)c * k + j0 + j] : 0.0;
    }
    __syncthreads();
#pragma unroll 2
    for (int j = 2 * lane; j < len; j += 64) {
      double2 g[4];
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const double* p = Gb + (int64_t)(row0 + r) * ld + j0 + j;
        if (row0 + r >= k) g[r] = make_double2(0.0, 0.0);
        else if (vec_ok && j + 1 < len) g[r] = __ldg(reinterpret_cast<const double2*>(p));
        else g[r] = make_double2(__ldg(p), (j + 1 < len) ? __ldg(p + 1) : 0.0);
      }
#pragma unroll
      for (int c = 0; c < kKB; ++c) {
        const double2 q = *reinterpret_cast<const double2*>(s_q + c * kSymvChunk + j);  // padded with zeros beyond len
#pragma unroll
        for (int r = 0; r < 4; ++r) acc[r][c] = fma(g[r].y, q.y, fma(g[r].x, q.x, acc[r][c]));
      }
    }
  }
#pragma unroll
  for (int r = 0; r < 4; ++r)
#pragma unroll
    for (int c = 0; c < kKB; ++c) {
      double v = acc[r][c];
      for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
      if (lane == 0 && row0 + r < k) AQ[(int64_t)bt * strideQ + (int64_t)c * k + row0 + r] = v;
    }
}

// Entries of the 32-bit integer Gram G0 are sums of products of bytes, 0 <= x < 2^31: (2^52 + x) - 2^52 converts exactly
// with one DADD (an I2F.F64 conversion per element made the first int32 kernel conversion-bound).
__device__ __forceinline__ double u31_to_double(int x) { return __hiloint2double(0x43300000, x) - 4503599627370496.0; }

// G0 Q on the int32 Gram, column-owning form using the symmetry of G0: AQ[c][j] = sum_i G0[i][j] Q[c][i].  Every lane
// owns four adjacent columns j and keeps their 4 x 8 sums in registers for the whole kernel; a warp walks down rows
// (one coalesced 512-byte row segment per load) and reads the 8 Q values of the row as shared-memory BROADCASTS.
// Against a row-owning int32 kernel (the layout of symv_block_kernel with 128-bit loads; measured, then removed) this
// needs no cross-lane reduction and 8 instead of 20 shared-memory / L1 wavefronts per 128 matrix elements (ncu on the
// row-owning kernel: LSU wavefronts 59 % busy, fp64 pipe 34 %, DRAM 33 %: the shared-memory reads of Q were the limiter,
// not HBM; 25 us against 20.7 us per 4096^2 product).  The 16 warps of a CTA split the rows of every chunk;
// their partial sums are added in warp order through shared memory (deterministic).
constexpr int kColsWarps = 8;
constexpr int kColsCtasPerSm = 2;
constexpr int kColsPerLane = 2;
constexpr int kColsPerCta = 32 * kColsPerLane;
constexpr int kColsQRows = 64;   // rows of Q^T per warp-private staging buffer: 64 x 8 doubles = 4 KB, double-buffered
// Tuning history of this kernel (67 MB int32 per 4096^2 product; floors: 10.3 us from HBM, 8.1 us from the fp64 pipe):
//   v1 (round 1): 4 columns per lane, ONE 16-warp CTA per SM at 128 registers, Q staged per 1024-row chunk behind two CTA
//       barriers: 20.7 us (ncu: DRAM 40 %, fp64 41 %, 46 % of the stall samples are long-scoreboard waits on the G loads);
//   v2: 2 columns per lane, 24 warps per SM: 29.9 us cold / no change in the step (more warps, but each restarts its load
//       pipeline after every barrier with only 64 rows between barriers);
//   v2b: + software-pipelined loads (next batch of 8 rows in flight while this one is multiplied): 25.4 us cold, step
//       unchanged: 22 % of the samples still sit on the first use after each chunk barrier, 13 % on the Q staging stores;
//   v3 (this one): no CTA barrier in the main loop at all.  A warp owns a CONTIGUOUS run of rows for the whole kernel and
//       streams them with the two-batch load pipeline; the Q values of its rows come from a transposed copy Q^T [row][8]
//       (krylov_transpose_kernel), fetched 64 rows (one contiguous 4 KB piece) at a time into a warp-private,
//       double-buffered shared-memory tile with cp.async, read back as broadcasts.
// VEC: ld and k are even and the matrix is 8-byte aligned (always true for the Gram buffers of this library): every lane's
// column pair is one aligned 64-bit load and there is no column boundary inside a pair.
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// Qt[bt][row][c] = Q[bt][c][row] for row < k, zero for k <= row < k_pad
__global__ void krylov_transpose_kernel(const double* __restrict__ Q, int64_t strideQ, double* __restrict__ Qt, int64_t strideQt, int k,
                                        int k_pad) {
  const int64_t bt = blockIdx.y;
  const int row = blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= k_pad) return;
  double v[kKB];
#pragma unroll
  for (int c = 0; c < kKB; ++c) v[c] = row < k ? Q[bt * strideQ + (int64_t)c * k + row] : 0.0;
  double2* dst = reinterpret_cast<double2*>(Qt + bt * strideQt + (int64_t)row * kKB);
#pragma unroll
  for (int h = 0; h < kKB / 2; ++h) dst[h] = make_double2(v[2 * h], v[2 * h + 1]);
}

inline int symv_rows_per_warp(int k) { return ((k + kColsWarps - 1) / kColsWarps + kColsQRows - 1) / kColsQRows * kColsQRows; }
inline int symv_k_pad(int k) { return symv_rows_per_warp(k) * kColsWarps; }

template <bool VEC>
__global__ void __launch_bounds__(32 * kColsWarps, kColsCtasPerSm) symv_cols_i32_kernel(const int32_t* __restrict__ G, int64_t ld, int64_t strideG,
                                                                                     const double* __restrict__ Qt, int64_t strideQt,
                                                                                     double* __restrict__ AQ, int64_t strideQ, int k,
                                                                                     int rows_per_warp) {
  extern __shared__ __align__(16) double s_x[];  // [kColsWarps][2][kColsQRows][kKB]
  const int bt = blockIdx.y;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int col0 = blockIdx.x * kColsPerCta + kColsPerLane * lane;
  const int32_t* Gb = G + (int64_t)bt * strideG;
  const double* Qtb = Qt + (int64_t)bt * strideQt;
  double* xs = s_x + (size_t)warp * 2 * kColsQRows * kKB;
  constexpr int kUnroll = 8;
  double acc[kColsPerLane][kKB];
#pragma unroll
  for (int e = 0; e < kColsPerLane; ++e)
#pragma unroll
    for (int c = 0; c < kKB; ++c) acc[e][c] = 0.0;
  const int row_begin = warp * rows_per_warp;
  const int row_end = min(k, row_begin + rows_per_warp);
  auto fetch_q = [&](int chunk, int buf) {  // rows [row_begin + 64 chunk, + 64) of Q^T: 4 KB contiguous (Q^T is zero-padded to k_pad)
    const double* src = Qtb + (int64_t)(row_begin + chunk * kColsQRows) * kKB;
    double* dst = xs + buf * kColsQRows * kKB;
#pragma unroll
    for (int i = 0; i < kColsQRows * kKB / 64; ++i) cp_async16(dst + (i * 32 + lane) * 2, src + (i * 32 + lane) * 2);
    cp_async_commit();
  };
  auto load_batch = [&](int2 (&g)[kUnroll], int r) {
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
      const int32_t* p = Gb + (int64_t)(r + u) * ld + col0;
      if (r + u >= row_end || col0 >= k) g[u] = make_int2(0, 0);
      else if (VEC) g[u] = __ldg(reinterpret_cast<const int2*>(p));
      else g[u] = make_int2(__ldg(p), (col0 + 1 < k) ? __ldg(p + 1) : 0);
    }
  };
  auto mul_batch = [&](const int2 (&g)[kUnroll], const double* xrows) {
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
      const double gd0 = u31_to_double(g[u].x), gd1 = u31_to_double(g[u].y);
      const double2* xr = reinterpret_cast<const double2*>(xrows + u * kKB);
#pragma unroll
      for (int h = 0; h < kKB / 2; ++h) {
        const double2 x = xr[h];  // same address in every lane: broadcast
        acc[0][2 * h] = fma(gd0, x.x, acc[0][2 * h]);         acc[0][2 * h + 1] = fma(gd0, x.y, acc[0][2 * h + 1]);
        acc[1][2 * h] = fma(gd1, x.x, acc[1][2 * h]);         acc[1][2 * h + 1] = fma(gd1, x.y, acc[1][2 * h + 1]);
      }
    }
  };
  if (row_begin < row_end) {
    const int nchunks = (row_end - row_begin + kColsQRows - 1) / kColsQRows;
    int2 ga[kUnroll], gb[kUnroll];
    fetch_q(0, 0);
    load_batch(ga, row_begin);
    for (int ch = 0; ch < nchunks; ++ch) {
      if (ch + 1 < nchunks) { fetch_q(ch + 1, (ch + 1) & 1); cp_async_wait<1>(); } else cp_async_wait<0>();
      __syncwarp();
      const double* xc = xs + (ch & 1) * kColsQRows * kKB;
      const int r0 = row_begin + ch * kColsQRows;
#pragma unroll 1
      for (int b = 0; b < kColsQRows / kUnroll; b += 2) {  // batches of 8 rows, two per iteration (register double buffer)
        load_batch(gb, r0 + (b + 1) * kUnroll);
        mul_batch(ga, xc + b * kUnroll * kKB);
        load_batch(ga, r0 + (b + 2) * kUnroll);            // first batch of the next chunk when b + 2 == 8: rows >= row_end load zeros
        mul_batch(gb, xc + (b + 1) * kUnroll * kKB);
      }
      __syncwarp();  // every lane is done with this buffer before the fetch of chunk ch + 2 overwrites it
    }
  }
  // add the warps' sums in warp order: tot[c][kColsPerCta columns]
  __syncthreads();
  double* tot = s_x;
  for (int w = 0; w < kColsWarps; ++w) {
    if (warp == w) {
#pragma unroll
      for (int c = 0; c < kKB; ++c)
#pragma unroll
        for (int e = 0; e < kColsPerLane; ++e) {
          double* t = tot + c * kColsPerCta + kColsPerLane * lane + e;
          *t = (w == 0) ? acc[e][c] : *t + acc[e][c];
        }
    }
    __syncthreads();
  }
  double* out = AQ + (int64_t)bt * strideQ;
  for (int idx = threadIdx.x; idx < kKB * kColsPerCta; idx += 32 * kColsWarps) {
    const int c = idx / kColsPerCta, j = blockIdx.x * kColsPerCta + (idx % kColsPerCta);
    if (j < k) out[(int64_t)c * k + j] = tot[idx];
  }
}

// ---------------------------------------------------------------------------------------------------
// G0 Q on the fp64 tensor cores (DMMA m8n8k4): the 8 vectors of the block are exactly the N = 8 of the instruction.
//   D[v][n] += sum_{kq<4} A[v][kq] B[kq][n],  A[v][kq] = Q^T[r + kq][v],  B[kq][n] = G0[r + kq][column(n)]
// Fragment layout (PTX m8n8k4 .f64): lane l holds A[l / 4][l % 4], B[l % 4][l / 4] and D[l / 4][2 (l % 4) + {0, 1}].
// Lane l loads ONE 128-bit piece G0[r + l % 4][c0 + 4 (l / 4) .. + 3]: a warp-wide load covers 4 rows x 128 bytes (four
// full lines), and element j of the piece is the B operand of MMA j, whose column index n stands for column c0 + 4 n + j.
// So lane l ends up with vector v = l / 4 of the 8 adjacent columns c0 + 8 (l % 4) + {j, 4 + j}.  Against the column-owning
// kernel above: 1 + 1 loads, 4 conversions and 4 MMAs per 128 matrix elements instead of 54 instructions, no shared memory in
// the main loop, and half the registers -- twice the warps and four times the bytes in flight per SM.
// A CTA owns 32 kDmmaCW columns; every lane keeps kDmmaU row quads in flight, with an explicit register double buffer: the
// loads of the NEXT batch are issued before the MMAs of this one (without it ptxas schedules for minimum registers: two loads in
// flight per lane).  Measured per 4096^2 product inside a 48-matrix launch (scripts/symv_bench.py, B200): 11.4 us = 5.9 TB/s,
// 0.90 of the HBM peak, against 17.3 us for the column-owning kernel, 12.3 us without the double buffer and 11.7-12.4 us with
// 64 columns per CTA (those variants were deleted after measurement).
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ int4 ldg_stream_v4(const int32_t* p) {
  int4 v;
  asm volatile("ld.global.nc.L1::no_allocate.v4.s32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
  return v;
}
constexpr int kDmmaWarps = 8;
constexpr int kDmmaCW = 1;  // 32-column groups per warp (the A fragment is shared by them)
constexpr int kDmmaU = 4;   // row quads in flight per lane
__global__ void __launch_bounds__(32 * kDmmaWarps) symv_dmma_pipe_i32_kernel(const int32_t* __restrict__ G, int64_t ld, int64_t strideG,
                                                                            const double* __restrict__ Qt, int64_t strideQt,
                                                                            double* __restrict__ AQ, int64_t strideQ, int k,
                                                                            int rows_per_warp) {
  constexpr int CW = kDmmaCW, U = kDmmaU;
  __shared__ double red[kDmmaWarps][kKB][32 * CW];
  const int bt = blockIdx.y;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int kq = lane & 3, grp = lane >> 2;
  const int col0 = blockIdx.x * 32 * CW;
  const int32_t* Gl = G + (int64_t)bt * strideG + col0 + 4 * grp;
  const double* Ql = Qt + (int64_t)bt * strideQt + grp;
  double acc[CW][4][2];
#pragma unroll
  for (int w = 0; w < CW; ++w)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[w][j][0] = acc[w][j][1] = 0.0;
  const int row_begin = warp * rows_per_warp;
  const int row_end = min(k, row_begin + rows_per_warp);   // the row count is a multiple of 8 U (checked by the launcher)
  auto load = [&](int4 (&g)[U][CW], double (&a)[U], int r) {
    const bool on = r < row_end;
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int32_t* p = Gl + (int64_t)(r + 4 * u) * ld;
#pragma unroll
      for (int w = 0; w < CW; ++w) g[u][w] = on ? ldg_stream_v4(p + 32 * w) : make_int4(0, 0, 0, 0);
      a[u] = on ? __ldg(Ql + (int64_t)(r + 4 * u) * kKB) : 0.0;
    }
  };
  auto mul = [&](const int4 (&g)[U][CW], const double (&a)[U]) {
#pragma unroll
    for (int u = 0; u < U; ++u)
#pragma unroll
      for (int w = 0; w < CW; ++w) {
        dmma884(acc[w][0][0], acc[w][0][1], a[u], u31_to_double(g[u][w].x));
        dmma884(acc[w][1][0], acc[w][1][1], a[u], u31_to_double(g[u][w].y));
        dmma884(acc[w][2][0], acc[w][2][1], a[u], u31_to_double(g[u][w].z));
        dmma884(acc[w][3][0], acc[w][3][1], a[u], u31_to_double(g[u][w].w));
      }
  };
  int4 ga[U][CW], gb[U][CW];
  double aa[U], ab[U];
  load(ga, aa, row_begin + kq);
#pragma unroll 1
  for (int r = row_begin + kq; r < row_end; r += 8 * U) {
    load(gb, ab, r + 4 * U);
    mul(ga, aa);
    load(ga, aa, r + 8 * U);
    mul(gb, ab);
  }
#pragma unroll
  for (int w = 0; w < CW; ++w)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      red[warp][grp][32 * w + 8 * kq + j] = acc[w][j][0];
      red[warp][grp][32 * w + 8 * kq + 4 + j] = acc[w][j][1];
    }
  __syncthreads();
  double* out = AQ + (int64_t)bt * strideQ;
  for (int idx = threadIdx.x; idx < kKB * 32 * CW; idx += 32 * kDmmaWarps) {
    const int c = idx / (32 * CW), jj = idx - c * (32 * CW);
    double v = 0.0;
#pragma unroll
    for (int w = 0; w < kDmmaWarps; ++w) v += red[w][c][jj];
    out[(int64_t)c * k + col0 + jj] = v;
  }
}

inline bool symv_dmma_ok(int k, int64_t ld, const void* G) {
  return k % (kDmmaWarps * 32) == 0 && ld % 4 == 0 && reinterpret_cast<uintptr_t>(G) % 16 == 0;
}
static void launch_symv_dmma(const int32_t* G, int64_t ld, int64_t strideG, const double* Qt, int64_t strideQt, double* AQ,
                             int64_t strideQ, int k, int batch, cudaStream_t st) {
  const int rpw = k / kDmmaWarps;  // a multiple of 32 = 8 kDmmaU
  dim3 grid(k / (32 * kDmmaCW), batch);
  symv_dmma_pipe_i32_kernel<<<grid, 32 * kDmmaWarps, 0, st>>>(G, ld, strideG, Qt, strideQt, AQ, strideQ, k, rpw);
}

// AQ += C Q for the strip form of the correction (GramView).  Two deterministic passes, no atomics:
//   rows i = hr[p]:      AQ[c][i] += sum_j Cs[p][j] Q[c][j]                 (one CTA per strip row, fixed-order reduction)
//   rows i not in hr:    AQ[c][i] += sum_p Cs[p][i] Q[c][hr[p]]             (one thread per row, p ascending)
constexpr int kStripRowsPerCta = 4;  // Q is read once per CTA, so more rows per CTA = less L2 traffic
__global__ void __launch_bounds__(256) strip_rows_kernel(const GramView g, const double* __restrict__ Q, int64_t strideQ,
                                                         double* __restrict__ AQ, int k) {
  __shared__ double red[kStripRowsPerCta][kKB][8];
  const int64_t bt = blockIdx.y;
  const int p0 = blockIdx.x * kStripRowsPerCta;
  const int m = g.hm[bt];
  if (p0 >= m) return;
  const double* rows = g.Cs + (bt * g.cs_rows + p0) * g.ld;
  const double* Qb = Q + bt * strideQ;
  double acc[kStripRowsPerCta][kKB];
#pragma unroll
  for (int r = 0; r < kStripRowsPerCta; ++r)
#pragma unroll
    for (int c = 0; c < kKB; ++c) acc[r][c] = 0.0;
  for (int j = threadIdx.x; j < k; j += 256) {
    double v[kStripRowsPerCta];
    bool any = false;
#pragma unroll
    for (int r = 0; r < kStripRowsPerCta; ++r) {
      v[r] = (p0 + r < m) ? rows[(int64_t)r * g.ld + j] : 0.0;
      any |= v[r] != 0.0;
    }
    if (!any) continue;
#pragma unroll
    for (int c = 0; c < kKB; ++c) {
      const double q = Qb[(int64_t)c * k + j];
#pragma unroll
      for (int r = 0; r < kStripRowsPerCta; ++r) acc[r][c] = fma(v[r], q, acc[r][c]);
    }
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
  for (int r = 0; r < kStripRowsPerCta; ++r)
#pragma unroll
    for (int c = 0; c < kKB; ++c) {
      double v = acc[r][c];
      for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xFFFFFFFFu, v, o);
      if (lane == 0) red[r][c][warp] = v;
    }
  __syncthreads();
  if (threadIdx.x < kStripRowsPerCta * kKB) {
    const int r = threadIdx.x / kKB, c = threadIdx.x - r * kKB;
    if (p0 + r < m) {
      double v = 0.0;
#pragma unroll
      for (int w = 0; w < 8; ++w) v += red[r][c][w];
      AQ[bt * strideQ + (int64_t)c * k + g.hr[bt * g.cs_rows + p0 + r]] += v;
    }
  }
}

// The row pass on the fp64 tensor cores: Y[v][p] = sum_j Q[v][j] Cs[p][j] is an (8 x k) x (k x m) product, M = 8 vectors, N = 8
// strip rows per MMA, K = columns.  A CTA owns 64 strip rows (8 groups of 8), its 8 warps split the columns; per 16 columns a
// lane loads 4 consecutive doubles of Q[l / 4][.] (shared by all 8 groups) and of Cs[p0 + 8 g + l / 4][.] per group, element t of
// both being the k-slot l % 4 of MMA t (any pairing of k-slots with columns works as long as A and B use the same one).
// Q is read once per 64 strip rows instead of once per 4 (strip_rows_kernel: 8.6 MB of Q for a 4.3 MB strip).
constexpr int kStripDmmaRows = 64;
__global__ void __launch_bounds__(256) strip_rows_dmma_kernel(const GramView g, const double* __restrict__ Q, int64_t strideQ,
                                                              double* __restrict__ AQ, int k) {
  __shared__ double red[8][kStripDmmaRows][kKB];
  const int64_t bt = blockIdx.y;
  const int p0 = blockIdx.x * kStripDmmaRows;
  const int m = g.hm[bt];
  if (p0 >= m) return;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int kq = lane & 3, grp = lane >> 2;
  const double* Qb = Q + bt * strideQ + (int64_t)grp * k + 4 * kq;
  const double* Cb = g.Cs + (bt * g.cs_rows + p0 + grp) * g.ld + 4 * kq;
  const int ngroups = min(kStripDmmaRows / 8, (m - p0 + 7) / 8);
  double acc[kStripDmmaRows / 8][2];
#pragma unroll
  for (int gi = 0; gi < kStripDmmaRows / 8; ++gi) acc[gi][0] = acc[gi][1] = 0.0;
  const int cols_per_warp = k / 8;  // a multiple of 16 (launcher)
  const int j_end = (warp + 1) * cols_per_warp;
#pragma unroll 1
  for (int j = warp * cols_per_warp; j < j_end; j += 16) {
    const double2 a01 = __ldg(reinterpret_cast<const double2*>(Qb + j)), a23 = __ldg(reinterpret_cast<const double2*>(Qb + j + 2));
    double2 b01[kStripDmmaRows / 8], b23[kStripDmmaRows / 8];
#pragma unroll
    for (int gi = 0; gi < kStripDmmaRows / 8; ++gi) {
      const bool on = gi < ngroups && p0 + 8 * gi + grp < m;  // rows >= m of a strip are never initialised
      const double* src = Cb + (int64_t)(8 * gi) * g.ld + j;
      b01[gi] = on ? __ldg(reinterpret_cast<const double2*>(src)) : make_double2(0.0, 0.0);
      b23[gi] = on ? __ldg(reinterpret_cast<const double2*>(src + 2)) : make_double2(0.0, 0.0);
    }
#pragma unroll
    for (int gi = 0; gi < kStripDmmaRows / 8; ++gi) {
      if (gi < ngroups) {  // warp-uniform
        dmma884(acc[gi][0], acc[gi][1], a01.x, b01[gi].x);
        dmma884(acc[gi][0], acc[gi][1], a01.y, b01[gi].y);
        dmma884(acc[gi][0], acc[gi][1], a23.x, b23[gi].x);
        dmma884(acc[gi][0], acc[gi][1], a23.y, b23[gi].y);
      }
    }
  }
#pragma unroll
  for (int gi = 0; gi < kStripDmmaRows / 8; ++gi) {  // lane: vector grp, strip rows 8 gi + 2 kq + {0, 1}
    red[warp][8 * gi + 2 * kq][grp] = acc[gi][0];
    red[warp][8 * gi + 2 * kq + 1][grp] = acc[gi][1];
  }
  __syncthreads();
  for (int idx = threadIdx.x; idx < kStripDmmaRows * kKB; idx += 256) {
    const int pr = idx / kKB, c = idx - pr * kKB;
    if (p0 + pr < m) {
      double v = 0.0;
#pragma unroll
      for (int w = 0; w < 8; ++w) v += red[w][pr][c];
      AQ[bt * strideQ + (int64_t)c * k + g.hr[bt * g.cs_rows + p0 + pr]] += v;
    }
  }
}

constexpr int kStripChunk = 128;  // strip rows staged per pass
__global__ void __launch_bounds__(256) strip_cols_kernel(const GramView g, const double* __restrict__ Q, int64_t strideQ,
                                                         double* __restrict__ AQ, int k) {
  __shared__ double s_q[kStripChunk][kKB];
  const int64_t bt = blockIdx.y;
  const int m = g.hm[bt];
  if (m == 0) return;
  const int i = blockIdx.x * 256 + threadIdx.x;
  const bool mine = i < k && g.pos[bt * g.ld + i] < 0;
  const double* Cs = g.Cs + bt * g.cs_rows * g.ld;
  const double* Qb = Q + bt * strideQ;
  const int32_t* hr = g.hr + bt * g.cs_rows;
  double acc[kKB];
#pragma unroll
  for (int c = 0; c < kKB; ++c) acc[c] = 0.0;
  for (int p0 = 0; p0 < m; p0 += kStripChunk) {
    const int len = min(kStripChunk, m - p0);
    __syncthreads();
    for (int t = threadIdx.x; t < len * kKB; t += 256) {
      const int pp = t / kKB, c = t - pp * kKB;
      s_q[pp][c] = Qb[(int64_t)c * k + hr[p0 + pp]];
    }
    __syncthreads();
    if (mine) {
      for (int pp = 0; pp < len; ++pp) {
        const double v = Cs[(int64_t)(p0 + pp) * g.ld + i];
        if (v != 0.0) {
#pragma unroll
          for (int c = 0; c < kKB; ++c) acc[c] = fma(v, s_q[pp][c], acc[c]);
        }
      }
    }
  }
  if (mine) {
#pragma unroll
    for (int c = 0; c < kKB; ++c) AQ[bt * strideQ + (int64_t)c * k + i] += acc[c];
  }
}

__global__ void copy_block_kernel(const double* src, int64_t strideS, double* dst, int64_t strideD, int64_t elems) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < elems) dst[blockIdx.y * strideD + i] = src[blockIdx.y * strideS + i];
}

// W[c][pos] -= sum_r C[r][c] * Q[r][pos],  r < rows
__global__ void __launch_bounds__(256) krylov_subtract_kernel(double* W, int64_t strideW, const double* __restrict__ Q,
                                                              int64_t strideQ, const double* __restrict__ C, int64_t strideCm,
                                                              int rows, int k) {
  __shared__ double sC[kKDim * kKB];
  const int64_t bt = blockIdx.y;
  for (int i = threadIdx.x; i < rows * kKB; i += blockDim.x) sC[i] = C[bt * strideCm + i];
  __syncthreads();
  int pos = blockIdx.x * blockDim.x + threadIdx.x;
  if (pos >= k) return;
  double w[kKB];
  double* Wb = W + bt * strideW;
  const double* Qb = Q + bt * strideQ;
#pragma unroll
  for (int c = 0; c < kKB; ++c) w[c] = Wb[(int64_t)c * k + pos];
  for (int r = 0; r < rows; ++r) {
    double q = Qb[(int64_t)r * k + pos];
#pragma unroll
    for (int c = 0; c < kKB; ++c) w[c] = fma(-sC[r * kKB + c], q, w[c]);
  }
#pragma unroll
  for (int c = 0; c < kKB; ++c) Wb[(int64_t)c * k + pos] = w[c];
}

// SVQB orthonormalisation of a block, in two kernels.  factor: S = W W^T (8 x 8, given) is scaled to unit diagonal
// and eigen-decomposed ONCE per matrix; U = Lambda^{-1/2} V^T D (8 x 8) goes to global memory.  Directions with
// lambda <= 1e-13 * lambda_max are dropped (zero vectors).  apply: W <- U W, one thread per column of W.
__global__ void __launch_bounds__(64) krylov_svqb_factor_kernel(const double* __restrict__ S, int64_t strideS, double* __restrict__ U) {
  __shared__ double sS[kKB * (kKB + 1)], sV[kKB * (kKB + 1)], sD[kKB];
  __shared__ JacobiScratchT<kKB> js;
  const int64_t bt = blockIdx.x;
  const int tid = threadIdx.x;
  const int ld = kKB + 1;
  const double* Sb = S + bt * strideS;
  if (tid < kKB) {
    double d = Sb[tid * kKB + tid];
    sD[tid] = d > 0.0 ? rsqrt(d) : 0.0;
  }
  __syncthreads();
  for (int i = tid; i < kKB * kKB; i += blockDim.x) {
    int r = i / kKB, c = i - r * kKB;
    sS[r * ld + c] = 0.5 * (Sb[r * kKB + c] + Sb[c * kKB + r]) * sD[r] * sD[c];
    sV[r * ld + c] = (r == c) ? 1.0 : 0.0;
  }
  __syncthreads();
  jacobi_eig_smem(sS, ld, kKB, sV, ld, &js);
  __syncthreads();
  if (tid < kKB) {
    double lmax = 0.0;
    for (int i = 0; i < kKB; ++i) lmax = fmax(lmax, sS[i * ld + i]);
    double lam = sS[tid * ld + tid];
    double sc = (lam > 1e-13 * lmax && lam > 0.0) ? rsqrt(lam) : 0.0;
    // new vector `tid` = sum_c U[tid][c] W_c, U[tid][c] = sc * V[c][tid] * D[c]
    for (int c = 0; c < kKB; ++c) U[bt * kKB * kKB + tid * kKB + c] = sc * sV[c * ld + tid] * sD[c];
  }
}

__global__ void __launch_bounds__(256) krylov_svqb_apply_kernel(double* W, int64_t strideW, const double* __restrict__ U, int k) {
  __shared__ double sU[kKB * kKB];
  const int64_t bt = blockIdx.y;
  if (threadIdx.x < kKB * kKB) sU[threadIdx.x] = U[bt * kKB * kKB + threadIdx.x];
  __syncthreads();
  double* Wb = W + bt * strideW;
  const int pos = blockIdx.x * blockDim.x + threadIdx.x;
  if (pos >= k) return;
  double w[kKB], o[kKB];
#pragma unroll
  for (int c = 0; c < kKB; ++c) w[c] = Wb[(int64_t)c * k + pos];
#pragma unroll
  for (int v = 0; v < kKB; ++v) {
    double s = 0.0;
#pragma unroll
    for (int c = 0; c < kKB; ++c) s = fma(sU[v * kKB + c], w[c], s);
    o[v] = s;
  }
#pragma unroll
  for (int v = 0; v < kKB; ++v) Wb[(int64_t)v * k + pos] = o[v];
}

// Rayleigh-Ritz of T (dim x dim): Jacobi with eigenvectors in shared memory; writes the coefficients of the top-8
// Ritz vectors (Vtop [dim][8]), their Ritz values (theta [8]), zeroes the residual accumulators and updates
// info = {top4, trace(G), residual (filled by ritz_kernel), dim, cycles, |top4 - previous top4| / trace}.
__global__ void __launch_bounds__(256) krylov_rr_kernel(const double* __restrict__ T, int64_t strideT, int dim,
                                                        const double* __restrict__ diag, int k, double* Vtop, double* theta,
                                                        double* res2, double* info) {
  extern __shared__ __align__(16) double s_A[];  // A [dim][dim|1], V [dim][dim|1]
  __shared__ JacobiScratch js;
  __shared__ double lam[kJacobiMaxK], tmp[kJacobiMaxK];
  __shared__ int order[kKB];
  __shared__ double red[256];
  const int64_t bt = blockIdx.x;
  const int tid = threadIdx.x;
  const int lda = dim | 1;
  double* s_V = s_A + dim * lda;
  const double* Tb = T + bt * strideT;
  const double* db = diag + bt * k;
  double tr = 0.0;
  for (int i = tid; i < k; i += blockDim.x) tr += db[i];
  red[tid] = tr;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) { if (tid < o) red[tid] += red[tid + o]; __syncthreads(); }
  tr = red[0];
  for (int idx = tid; idx < dim * dim; idx += blockDim.x) {
    int r = idx / dim, c = idx - r * dim;
    s_A[r * lda + c] = 0.5 * (Tb[r * kKDim + c] + Tb[c * kKDim + r]);
    s_V[r * lda + c] = (r == c) ? 1.0 : 0.0;
  }
  __syncthreads();
  jacobi_eig_smem(s_A, lda, dim, s_V, lda, &js);
  sort_diag_desc(s_A, lda, dim, tmp, lam);
  // column index of the i-th largest eigenvalue, i < 8 (same rank rule as sort_diag_desc)
  for (int i = tid; i < dim; i += blockDim.x) {
    double v = tmp[i];
    int rank = 0;
    for (int j = 0; j < dim; ++j) rank += (tmp[j] > v || (tmp[j] == v && j < i)) ? 1 : 0;
    if (rank < kKB) order[rank] = i;
  }
  __syncthreads();
  double* Vb = Vtop + bt * kKDim * kKB;
  for (int idx = tid; idx < dim * kKB; idx += blockDim.x) {
    int d = idx / kKB, c = idx - d * kKB;
    Vb[idx] = s_V[d * lda + order[c]];
  }
  if (tid < kKB) theta[bt * kKB + tid] = lam[tid];
  if (tid < 4) res2[bt * 4 + tid] = 0.0;
  if (tid == 0) {
    double top = lam[0] + lam[1] + lam[2] + lam[3];
    double* inf = info + bt * kInfo;
    double prev = inf[0];
    inf[5] = tr > 0.0 ? fabs(top - prev) / tr : 0.0;
    inf[0] = top;
    inf[1] = tr;
    inf[3] = (double)dim;
    inf[4] += 1.0;
    inf[6] = lam[3];
    inf[7] = lam[4];
  }
}

// Ritz vectors Y = Vtop^T Q written in place of Q_0 (every thread owns one column `pos`), and the squared
// residual norms of the top 4: || Vtop_i^T AQ - theta_i Y_i ||^2 accumulated with one atomic per warp.
__global__ void __launch_bounds__(256) krylov_ritz_kernel(double* Q, const double* __restrict__ AQ, int64_t strideQ,
                                                          const double* __restrict__ Vtop, const double* __restrict__ theta,
                                                          double* res2, int dim, int k) {
  __shared__ double sV[kKDim * kKB], sT[kKB];
  const int64_t bt = blockIdx.y;
  for (int i = threadIdx.x; i < dim * kKB; i += blockDim.x) sV[i] = Vtop[bt * kKDim * kKB + i];
  if (threadIdx.x < kKB) sT[threadIdx.x] = theta[bt * kKB + threadIdx.x];
  __syncthreads();
  const int pos = blockIdx.x * blockDim.x + threadIdx.x;
  double y[kKB], gy[4];
#pragma unroll
  for (int c = 0; c < kKB; ++c) y[c] = 0.0;
#pragma unroll
  for (int c = 0; c < 4; ++c) gy[c] = 0.0;
  if (pos < k) {
    double* Qb = Q + bt * strideQ;
    const double* Ab = AQ + bt * strideQ;
    for (int d = 0; d < dim; ++d) {
      double q = Qb[(int64_t)d * k + pos], a = Ab[(int64_t)d * k + pos];
#pragma unroll
      for (int c = 0; c < kKB; ++c) y[c] = fma(sV[d * kKB + c], q, y[c]);
#pragma unroll
      for (int c = 0; c < 4; ++c) gy[c] = fma(sV[d * kKB + c], a, gy[c]);
    }
#pragma unroll
    for (int c = 0; c < kKB; ++c) Qb[(int64_t)c * k + pos] = y[c];
  }
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    double r = gy[c] - sT[c] * y[c];
    double v = r * r;
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
    if ((threadIdx.x & 31) == 0 && v != 0.0) atomicAdd(res2 + bt * 4 + c, v);
  }
}

__global__ void krylov_finish_kernel(const double* __restrict__ theta, const double* __restrict__ res2, double* info, double* scores,
                                     int64_t batch) {
  int64_t bt = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (bt >= batch) return;
  double* inf = info + bt * kInfo;
  double t0 = theta[bt * kKB];
  double r = 0.0;
  for (int c = 0; c < 4; ++c) r = fmax(r, res2[bt * 4 + c]);
  inf[2] = t0 > 0.0 ? sqrt(r) / t0 : 0.0;
  double tr = inf[1];
  scores[bt] = tr > 0.0 ? sqrt(fmax(1.0 - inf[0] / tr, 0.0)) : nan("");
}

thread_local int g_last_unconverged = 0;  // spb_score_last_unconverged()

struct KrylovWs {
  double *Q, *AQ, *C, *S, *U, *T, *Vtop, *theta, *res2, *info, *part, *idx, *diag, *Qt;
  int64_t sQ, sC, sS, sT, part_elems;
  double *W, *sp_part;  // sparse operator only: F^T Q [ncols][8] and the segment partial sums (sparse.cu)
};

static int64_t krylov_layout(int64_t k, int64_t batch, double* base, KrylovWs* w) {
  int64_t off = 0;
  auto take = [&](int64_t n) { double* p = base ? base + off : nullptr; off += (n + 1) / 2 * 2; return p; };
  w->sQ = (int64_t)kKDim * k;
  w->Q = take(batch * w->sQ);
  w->AQ = take(batch * w->sQ);
  w->sC = (int64_t)kKDim * kKB;
  w->C = take(batch * w->sC);
  w->sS = (int64_t)kKB * kKB;
  w->S = take(batch * w->sS);
  w->U = take(batch * w->sS);
  w->sT = (int64_t)kKDim * kKDim;
  w->T = take(batch * w->sT);
  w->Vtop = take(batch * kKDim * kKB);
  w->theta = take(batch * kKB);
  w->res2 = take(batch * 4);
  w->info = take(batch * kInfo);
  w->idx = take(batch * kKB);  // int[8] per matrix (start rows), stored in double-sized slots
  w->diag = take(batch * k);   // diagonal of G (start-row choice, trace)
  w->Qt = take(batch * (int64_t)symv_k_pad((int)k) * kKB);  // transposed, zero-padded copy of the block being multiplied (int32 route)
  // partial sums of the inner-product kernel: ceil(k / 128) chunks of the largest (96 x 96) product
  w->part_elems = batch * ((k + kDotChunk - 1) / kDotChunk) * (int64_t)kKDim * kKDim;
  w->part = take(w->part_elems);
  return off;
}

// Sparse operator: W and the segment partials after the dense layout
static int64_t sparse_layout(const SparseBatch& f, double* base, KrylovWs* w) {
  const int64_t off = krylov_layout(f.k, f.batch, base, w);
  const int64_t nw = (f.ncols * 8 + 1) / 2 * 2;
  w->W = base ? base + off : nullptr;
  w->sp_part = base ? base + off + nw : nullptr;
  return off + nw + sparse_part_doubles(f);
}

// AQ = F (F^T Q) for one block of 8 vectors: Q transposed into Qt [batch * k][8] (krylov_transpose_kernel with no padding),
// then the two segment products of sparse.cu
static int sparse_apply(const SparseBatch& f, const double* Q, int64_t strideQ, double* AQ, double* Qt, double* W, double* part,
                        cudaStream_t st) {
  dim3 tg((f.k + 255) / 256, f.batch);
  krylov_transpose_kernel<<<tg, 256, 0, st>>>(Q, strideQ, Qt, (int64_t)f.k * kKB, f.k, f.k);
  SPB_LAUNCH_CHECK();
  return sparse_product_launch(f, Qt, W, AQ, strideQ, part, st);
}

}  // namespace

extern "C" int64_t spb_gram_f64_ws(int64_t R, int64_t C, int64_t batch) {
  int ks = choose_ksplit((int)R, (int)R, (int)C, (int)batch);
  return ks > 1 ? batch * ks * R * R : 0;
}

extern "C" int spb_gram_f64(const double* d_A, int64_t R, int64_t C, int64_t batch, double* d_G, double* d_ws, void* stream) {
  SPB_REQUIRE(d_A && d_G && R >= 1 && C >= 1 && batch >= 1 && R < (1 << 30) && C < (1 << 30), "spb_gram_f64: bad arguments");
  int ks = choose_ksplit((int)R, (int)R, (int)C, (int)batch);
  SPB_REQUIRE(ks == 1 || d_ws, "spb_gram_f64: workspace required (spb_gram_f64_ws)");
  GemmArgs g{d_A, C, R * C, d_A, C, R * C, d_G, R, R * R, (int)R, (int)R, (int)C, (int)batch};
  return gemm_nt(g, ks, d_ws, (cudaStream_t)stream);
}

extern "C" int spb_score_gram_small(const double* d_G, int64_t k, int64_t ld, int64_t batch, double* d_scores, double* d_eig,
                                    void* stream) {
  SPB_REQUIRE(d_G && d_scores && k >= 1 && k <= kJacobiMaxK && ld >= k && batch >= 0,
              "spb_score_gram_small: need 1 <= k <= %d (got %lld)", kJacobiMaxK, (long long)k);
  if (batch == 0) return SPB_OK;
  // Score only (no eigenvalue list), 4 < k <= 64: warp-per-matrix Householder + 9-section (pairs.cu) instead of the Jacobi sweep
  if (!d_eig && k > 4 && k <= 64) return score_gram_warp_launch(d_G, (int)k, ld, batch, d_scores, (cudaStream_t)stream);
  size_t smem = (size_t)jacobi_dim((int)k) * jacobi_ld((int)k) * sizeof(double);
  SPB_CUDA(cudaFuncSetAttribute(score_small_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int threads = k <= 32 ? 128 : 256;
  int occ = 1;
  SPB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, score_small_kernel, threads, smem));
  if (occ < 1) occ = 1;
  int64_t grid = (int64_t)sm_count() * occ;
  if (grid > batch) grid = batch;
  score_small_kernel<<<(unsigned)grid, threads, smem, (cudaStream_t)stream>>>(d_G, (int)k, ld, batch, d_scores, d_eig);
  SPB_LAUNCH_CHECK();
  return SPB_OK;
}

extern "C" int64_t spb_score_gram_large_ws(int64_t k, int64_t batch) {
  KrylovWs w;
  return krylov_layout(k, batch, nullptr, &w);
}

static bool accept_matrix(const double* inf, int cycle) {
  // Convergence of the sum of the 4 largest Ritz values.  Kato-Temple: |theta - lambda| <= res^2 / gap with
  // gap = separation of the wanted cluster from the rest of the spectrum, estimated by (theta_4 - theta_5) /
  // theta_1.  The error that matters is relative to the radicand 1 - top4 / trace (it becomes the score), so a
  // matrix is accepted when res^2 <= 1e-11 * gap * radicand (100x below the 1e-9 parity tolerance), or when its
  // residual is at rounding level, or when the Ritz values have stopped moving at a residual that rounding can
  // explain (res <= 1e-9; the looser 1e-6 of round 1 accepted residuals far above the stated bound).
  const double top = inf[0], tr = inf[1], res = inf[2], delta = inf[5];
  if (!(tr > 0.0)) return true;
  const double radicand = fmax(1.0 - top / tr, 1e-12);
  const double t1 = fmax(top, 1e-300);
  const double gap = fmin(fmax((inf[6] - inf[7]) / t1, 1e-6), 1.0);
  return res <= 1e-13 || res * res <= 1e-11 * gap * radicand || (cycle > 0 && delta <= 1e-16 && res <= 1e-9);
}

// One Krylov cycle with `nb` blocks (dim = 8 nb).  first = 1 starts from the heaviest rows of G plus pseudo-random
// vectors (krylov_start_rows_kernel), otherwise from the Ritz vectors the previous cycle left in Q_0.
static int krylov_cycle(const GramView& gv, int k, int batch, int nb, bool first, const KrylovWs& w, cudaStream_t st,
                        const SparseBatch* sf = nullptr) {
  const int64_t ld = gv.ld;
  const int64_t blk = (int64_t)kKB * k;
  const int dim = nb * kKB;
  int rc;
  auto ortho_block = [&](double* W, int passes) -> int {  // SVQB
    for (int pass = 0; pass < passes; ++pass) {
      int r = dot_product(W, w.sQ, W, w.sQ, kKB, kKB, k, batch, w.S, kKB, w.sS, w.part, st);
      if (r) return r;
      krylov_svqb_factor_kernel<<<batch, 64, 0, st>>>(w.S, w.sS, w.U);
      SPB_LAUNCH_CHECK();
      dim3 grid((k + 255) / 256, batch);
      krylov_svqb_apply_kernel<<<grid, 256, 0, st>>>(W, w.sQ, w.U, k);
      SPB_LAUNCH_CHECK();
    }
    return SPB_OK;
  };
  if (first && sf) {
    dim3 grid((k + 255) / 256, batch);
    if ((rc = sparse_diag_launch(*sf, w.diag, st))) return rc;
    krylov_top8_kernel<<<batch, 256, 0, st>>>(w.diag, k, reinterpret_cast<int*>(w.idx));
    SPB_LAUNCH_CHECK();
    krylov_start_sparse_kernel<<<grid, 256, 0, st>>>(reinterpret_cast<const int*>(w.idx), w.Q, w.sQ, k);
    SPB_LAUNCH_CHECK();
    if ((rc = sparse_apply(*sf, w.Q, w.sQ, w.AQ, w.Qt, w.W, w.sp_part, st))) return rc;
    dim3 cg((unsigned)((kHeavyStart * (int64_t)k + 255) / 256), batch);  // G e_j in place of e_j
    copy_block_kernel<<<cg, 256, 0, st>>>(w.AQ, w.sQ, w.Q, w.sQ, kHeavyStart * (int64_t)k);
    SPB_LAUNCH_CHECK();
    if ((rc = ortho_block(w.Q, 2))) return rc;
  } else if (first) {
    dim3 grid((k + 255) / 256, batch);
    gram_diag_kernel<<<grid, 256, 0, st>>>(gv, k, w.diag);
    SPB_LAUNCH_CHECK();
    krylov_top8_kernel<<<batch, 256, 0, st>>>(w.diag, k, reinterpret_cast<int*>(w.idx));
    SPB_LAUNCH_CHECK();
    krylov_start_rows_kernel<<<grid, 256, 0, st>>>(gv, reinterpret_cast<const int*>(w.idx), w.Q, w.sQ, k);
    SPB_LAUNCH_CHECK();
    if ((rc = ortho_block(w.Q, 2))) return rc;
  } else {
    if ((rc = ortho_block(w.Q, 1))) return rc;  // Ritz vectors are orthonormal up to rounding: one clean-up pass
  }
  const size_t symv_smem = (size_t)kKB * kSymvChunk * sizeof(double);
  SPB_CUDA(cudaFuncSetAttribute(symv_block_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)symv_smem));
  const size_t cols_smem = (size_t)kColsWarps * 2 * kColsQRows * kKB * sizeof(double);
  SPB_CUDA(cudaFuncSetAttribute(symv_cols_i32_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cols_smem));
  SPB_CUDA(cudaFuncSetAttribute(symv_cols_i32_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cols_smem));
  const bool cols_vec = gv.Gi && (ld % 2 == 0) && (k % 2 == 0) && (reinterpret_cast<uintptr_t>(gv.Gi) % 8 == 0);
  const int rpw = symv_rows_per_warp(k), k_pad = symv_k_pad(k);
  for (int j = 0; j < nb; ++j) {
    double* Qj = w.Q + (int64_t)j * blk;
    double* AQj = w.AQ + (int64_t)j * blk;
    if (sf) {
      if ((rc = sparse_apply(*sf, Qj, w.sQ, AQj, w.Qt, w.W, w.sp_part, st))) return rc;
    } else {
      dim3 grid((k + kSymvRows - 1) / kSymvRows, batch);
      if (gv.Gf) symv_block_kernel<<<grid, 256, symv_smem, st>>>(gv.Gf, ld, ld * ld, Qj, w.sQ, AQj, k);
      else {
        dim3 tg((k_pad + 255) / 256, batch);
        krylov_transpose_kernel<<<tg, 256, 0, st>>>(Qj, w.sQ, w.Qt, (int64_t)k_pad * kKB, k, k_pad);
        SPB_LAUNCH_CHECK();
        dim3 gi((k + kColsPerCta - 1) / kColsPerCta, batch);
        if (symv_dmma_ok(k, ld, gv.Gi))
          launch_symv_dmma(gv.Gi, ld, ld * ld, w.Qt, (int64_t)k_pad * kKB, AQj, w.sQ, k, batch, st);
        else if (cols_vec) symv_cols_i32_kernel<true><<<gi, 32 * kColsWarps, cols_smem, st>>>(gv.Gi, ld, ld * ld, w.Qt, (int64_t)k_pad * kKB, AQj, w.sQ, k, rpw);
        else symv_cols_i32_kernel<false><<<gi, 32 * kColsWarps, cols_smem, st>>>(gv.Gi, ld, ld * ld, w.Qt, (int64_t)k_pad * kKB, AQj, w.sQ, k, rpw);
      }
      SPB_LAUNCH_CHECK();
      if (!gv.Gf && gv.cs_rows) {
        if (k % 128 == 0 && ld % 2 == 0 && reinterpret_cast<uintptr_t>(gv.Cs) % 16 == 0 &&
            reinterpret_cast<uintptr_t>(Qj) % 16 == 0 && w.sQ % 2 == 0) {
          dim3 rg((unsigned)((gv.cs_rows + kStripDmmaRows - 1) / kStripDmmaRows), batch);
          strip_rows_dmma_kernel<<<rg, 256, 0, st>>>(gv, Qj, w.sQ, AQj, k);
        } else {
          dim3 rg((unsigned)((gv.cs_rows + kStripRowsPerCta - 1) / kStripRowsPerCta), batch);
          strip_rows_kernel<<<rg, 256, 0, st>>>(gv, Qj, w.sQ, AQj, k);
        }
        SPB_LAUNCH_CHECK();
        dim3 cg((k + 255) / 256, batch);
        strip_cols_kernel<<<cg, 256, 0, st>>>(gv, Qj, w.sQ, AQj, k);
        SPB_LAUNCH_CHECK();
      }
    }
    if (j == nb - 1) break;
    double* Wn = w.Q + (int64_t)(j + 1) * blk;
    {
      dim3 grid((unsigned)((blk + 255) / 256), batch);
      copy_block_kernel<<<grid, 256, 0, st>>>(AQj, w.sQ, Wn, w.sQ, blk);
      SPB_LAUNCH_CHECK();
    }
    const int rows = (j + 1) * kKB;
    for (int pass = 0; pass < 2; ++pass) {
      if ((rc = dot_product(w.Q, w.sQ, Wn, w.sQ, rows, kKB, k, batch, w.C, kKB, w.sC, w.part, st))) return rc;
      dim3 grid((k + 255) / 256, batch);
      krylov_subtract_kernel<<<grid, 256, 0, st>>>(Wn, w.sQ, w.Q, w.sQ, w.C, w.sC, rows, k);
      SPB_LAUNCH_CHECK();
    }
    if ((rc = ortho_block(Wn, 2))) return rc;
  }
  {
    if ((rc = dot_product(w.Q, w.sQ, w.AQ, w.sQ, dim, dim, k, batch, w.T, kKDim, w.sT, w.part, st))) return rc;
  }
  size_t smem = (size_t)2 * dim * (dim | 1) * sizeof(double);
  SPB_CUDA(cudaFuncSetAttribute(krylov_rr_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  krylov_rr_kernel<<<batch, 256, smem, st>>>(w.T, w.sT, dim, w.diag, k, w.Vtop, w.theta, w.res2, w.info);
  SPB_LAUNCH_CHECK();
  {
    dim3 grid((k + 255) / 256, batch);
    krylov_ritz_kernel<<<grid, 256, 0, st>>>(w.Q, w.AQ, w.sQ, w.Vtop, w.theta, w.res2, dim, k);
    SPB_LAUNCH_CHECK();
  }
  return SPB_OK;
}

static int score_gram_large(const GramView& gv, int64_t k64, int64_t batch64, double* d_scores, double* d_info, double* d_ws,
                            void* stream, int max_cycles = 40, const SparseBatch* sf = nullptr) {
  SPB_REQUIRE((gv.Gf || gv.Gi || sf) && d_scores && d_ws && k64 > kJacobiMaxK && gv.ld >= k64 && batch64 >= 1 && k64 < (1 << 24) &&
                  batch64 <= 65535,
              "spb_score_gram_large: need k > %d and a workspace", kJacobiMaxK);
  const int k = (int)k64, batch = (int)batch64;
  cudaStream_t st = (cudaStream_t)stream;
  KrylovWs w;
  if (sf) sparse_layout(*sf, d_ws, &w);
  else krylov_layout(k, batch, d_ws, &w);
  SPB_CUDA(cudaMemsetAsync(w.info, 0, (size_t)batch * kInfo * sizeof(double), st));
  static thread_local std::vector<double> h_info;
  static thread_local std::vector<double> h_flag;
  h_info.resize((size_t)batch * kInfo);
  h_flag.assign((size_t)batch, 0.0);
  SPB_REQUIRE(max_cycles >= 1 && max_cycles <= 40, "spb_score_gram_large: the cycle budget must be 1..40 (got %d)", max_cycles);
  const int kMaxCycles = max_cycles;
  int rc;
  bool done = false;
  for (int cycle = 0; cycle < kMaxCycles && !done; ++cycle) {
    const int nb = cycle < 2 ? 2 : (cycle < 4 ? 4 : kKMaxBlocks);
    if ((rc = krylov_cycle(gv, k, batch, nb, cycle == 0, w, st, sf))) return rc;
    krylov_finish_kernel<<<(batch + 127) / 128, 128, 0, st>>>(w.theta, w.res2, w.info, d_scores, batch);
    SPB_LAUNCH_CHECK();
    SPB_CUDA(cudaMemcpyAsync(h_info.data(), w.info, (size_t)batch * kInfo * sizeof(double), cudaMemcpyDeviceToHost, st));
    SPB_CUDA(cudaStreamSynchronize(st));
    done = true;
    for (int b = 0; b < batch; ++b) {
      const bool ok = accept_matrix(h_info.data() + (size_t)b * kInfo, cycle);
      h_flag[b] = ok ? 1.0 : 0.0;
      if (!ok) done = false;
    }
  }
  // per-matrix converged flag (info[8]): a matrix that exhausted the cycle budget keeps its last score but is reported
  // (engine.score_gram warns); spb_last_error names the count
  int bad = 0;
  for (int b = 0; b < batch; ++b) bad += h_flag[b] == 0.0 ? 1 : 0;
  SPB_CUDA(cudaMemcpy2DAsync(w.info + 8, kInfo * sizeof(double), h_flag.data(), sizeof(double), sizeof(double), (size_t)batch,
                             cudaMemcpyHostToDevice, st));
  g_last_unconverged = bad;
  if (bad && kMaxCycles == 40) set_error("spb_score_gram_large: %d of %d matrices did not converge within %d cycles", bad, batch, kMaxCycles);
  if (d_info) SPB_CUDA(cudaMemcpyAsync(d_info, w.info, (size_t)batch * kInfo * sizeof(double), cudaMemcpyDeviceToDevice, st));
  return SPB_OK;
}

extern "C" int spb_score_last_unconverged(void) { return g_last_unconverged; }

extern "C" int spb_score_gram_large(const double* d_G, int64_t k, int64_t ld, int64_t batch, double* d_scores, double* d_info,
                                    double* d_ws, void* stream) {
  GramView gv{d_G, nullptr, ld, nullptr, 0, nullptr, nullptr, nullptr};
  return score_gram_large(gv, k, batch, d_scores, d_info, d_ws, stream);
}

// The same solvers with a cycle budget: the whole batch stays in the cycle until its last matrix is accepted, and the cycles grow
// (2, 2, 4, 4, 12, ... blocks), so a caller with a large batch runs the first cycles with a small budget, then calls again with the
// few matrices that report converged = 0 (engine.score_gram / CountScorer._score_i32).
extern "C" int spb_score_gram_large_n(const double* d_G, int64_t k, int64_t ld, int64_t batch, double* d_scores, double* d_info,
                                      double* d_ws, int max_cycles, void* stream) {
  GramView gv{d_G, nullptr, ld, nullptr, 0, nullptr, nullptr, nullptr};
  return score_gram_large(gv, k, batch, d_scores, d_info, d_ws, stream, max_cycles);
}

extern "C" int spb_score_gram_large_i32_n(const int32_t* d_Gi, int64_t k, int64_t ld, int64_t batch, const double* d_Cs, int64_t cs_rows,
                                          const int32_t* d_pos, const int32_t* d_hr, const int32_t* d_hm, double* d_scores,
                                          double* d_info, double* d_ws, int max_cycles, void* stream) {
  SPB_REQUIRE(cs_rows >= 0 && cs_rows <= 65535 && (cs_rows == 0 || (d_Cs && d_pos && d_hr && d_hm)),
              "spb_score_gram_large_i32: bad correction strip");
  GramView gv{nullptr, d_Gi, ld, d_Cs, cs_rows, d_pos, d_hr, d_hm};
  return score_gram_large(gv, k, batch, d_scores, d_info, d_ws, stream, max_cycles);
}

extern "C" int spb_score_gram_large_i32(const int32_t* d_Gi, int64_t k, int64_t ld, int64_t batch, const double* d_Cs,
                                        int64_t cs_rows, const int32_t* d_pos, const int32_t* d_hr, const int32_t* d_hm,
                                        double* d_scores, double* d_info, double* d_ws, void* stream) {
  SPB_REQUIRE(cs_rows >= 0 && cs_rows <= 65535 && (cs_rows == 0 || (d_Cs && d_pos && d_hr && d_hm)),
              "spb_score_gram_large_i32: bad correction strip");
  GramView gv{nullptr, d_Gi, ld, d_Cs, cs_rows, d_pos, d_hr, d_hm};
  return score_gram_large(gv, k, batch, d_scores, d_info, d_ws, stream);
}

// Diagnostic entry: AQ = G0 Q for a batch of int32 Gram matrices through one chosen kernel, launched exactly as krylov_cycle
// launches it: variant 0 = column-owning FMA kernel, 1 = DMMA kernel (needs k % 256 == 0, ld % 4 == 0).  d_Q, d_AQ:
// [batch][8][k]; d_Qt: spb_symv_i32_ws(k, batch) doubles of scratch.  Used by tests/test_gpu_parity_r2.py and
// scripts/symv_bench.py, not by the product path.
extern "C" int64_t spb_symv_i32_ws(int64_t k, int64_t batch) { return (int64_t)symv_k_pad((int)k) * kKB * batch; }

extern "C" int spb_symv_i32(const int32_t* d_Gi, int64_t k64, int64_t ld, int64_t batch64, const double* d_Q, double* d_AQ, double* d_Qt,
                            int variant, void* stream) {
  SPB_REQUIRE(d_Gi && d_Q && d_AQ && d_Qt && k64 > 0 && k64 <= (1 << 20) && ld >= k64 && batch64 > 0 && batch64 <= 65535 &&
              (variant == 0 || variant == 1), "spb_symv_i32: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  const int k = (int)k64, batch = (int)batch64;
  const int rpw = symv_rows_per_warp(k), k_pad = symv_k_pad(k);
  const int64_t sQ = (int64_t)kKB * k;
  dim3 tg((k_pad + 255) / 256, batch);
  krylov_transpose_kernel<<<tg, 256, 0, st>>>(d_Q, sQ, d_Qt, (int64_t)k_pad * kKB, k, k_pad);
  SPB_LAUNCH_CHECK();
  if (variant == 1) {
    SPB_REQUIRE(symv_dmma_ok(k, ld, d_Gi), "spb_symv_i32: the DMMA kernel needs k % 256 == 0, ld % 4 == 0");
    launch_symv_dmma(d_Gi, ld, ld * ld, d_Qt, (int64_t)k_pad * kKB, d_AQ, sQ, k, batch, st);
  } else {
    const size_t cols_smem = (size_t)kColsWarps * 2 * kColsQRows * kKB * sizeof(double);
    SPB_CUDA(cudaFuncSetAttribute(symv_cols_i32_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cols_smem));
    SPB_CUDA(cudaFuncSetAttribute(symv_cols_i32_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cols_smem));
    const bool vec = (ld % 2 == 0) && (k % 2 == 0) && (reinterpret_cast<uintptr_t>(d_Gi) % 8 == 0);
    dim3 gi((k + kColsPerCta - 1) / kColsPerCta, batch);
    if (vec) symv_cols_i32_kernel<true><<<gi, 32 * kColsWarps, cols_smem, st>>>(d_Gi, ld, ld * ld, d_Qt, (int64_t)k_pad * kKB, d_AQ, sQ, k, rpw);
    else symv_cols_i32_kernel<false><<<gi, 32 * kColsWarps, cols_smem, st>>>(d_Gi, ld, ld * ld, d_Qt, (int64_t)k_pad * kKB, d_AQ, sQ, k, rpw);
  }
  SPB_LAUNCH_CHECK();
  return SPB_OK;
}

// ---- sparse flattenings (sparse.cu): the same solver with G Q = F (F^T Q) ----
static SparseBatch sparse_batch(const int64_t* row_off, const int32_t* row_col, const double* row_val, const int64_t* col_off,
                                const int32_t* col_row, const double* col_val, int64_t ncols, int64_t nnz, int64_t k, int64_t batch) {
  return SparseBatch{row_off, row_col, row_val, col_off, col_row, col_val, ncols, nnz, (int)k, (int)batch};
}

extern "C" int64_t spb_score_sparse_large_ws(int64_t k, int64_t batch, int64_t ncols, int64_t nnz) {
  KrylovWs w;
  return sparse_layout(sparse_batch(nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, ncols, nnz, k, batch), nullptr, &w);
}

extern "C" int spb_score_sparse_large_n(const int64_t* d_row_off, const int32_t* d_row_col, const double* d_row_val, const int64_t* d_col_off,
                                        const int32_t* d_col_row, const double* d_col_val, int64_t ncols, int64_t nnz, int64_t k, int64_t batch,
                                        double* d_scores, double* d_info, double* d_ws, int max_cycles, void* stream) {
  SPB_REQUIRE(k > kJacobiMaxK && k < (1 << 24), "spb_score_sparse_large: need %d < k < 2^24 (got %lld)", kJacobiMaxK, (long long)k);
  const SparseBatch f = sparse_batch(d_row_off, d_row_col, d_row_val, d_col_off, d_col_row, d_col_val, ncols, nnz, k, batch);
  int rc = sparse_check(f);
  if (rc) return rc;
  GramView gv{nullptr, nullptr, k, nullptr, 0, nullptr, nullptr, nullptr};
  return score_gram_large(gv, k, batch, d_scores, d_info, d_ws, stream, max_cycles, &f);
}

// Diagnostic entry: d_AQ = F (F^T d_Q) for a batch of sparse flattenings, launched exactly as the solver launches it.
// d_Q, d_AQ: [batch][8][k]; d_ws: spb_sparse_product_ws(k, batch, ncols, nnz) doubles.
extern "C" int64_t spb_sparse_product_ws(int64_t k, int64_t batch, int64_t ncols, int64_t nnz) {
  const SparseBatch f = sparse_batch(nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, ncols, nnz, k, batch);
  return batch * k * kKB + (ncols * 8 + 1) / 2 * 2 + sparse_part_doubles(f);
}

extern "C" int spb_sparse_product(const int64_t* d_row_off, const int32_t* d_row_col, const double* d_row_val, const int64_t* d_col_off,
                                  const int32_t* d_col_row, const double* d_col_val, int64_t ncols, int64_t nnz, int64_t k, int64_t batch,
                                  const double* d_Q, double* d_AQ, double* d_ws, void* stream) {
  SPB_REQUIRE(d_Q && d_AQ && d_ws, "spb_sparse_product: bad arguments");
  const SparseBatch f = sparse_batch(d_row_off, d_row_col, d_row_val, d_col_off, d_col_row, d_col_val, ncols, nnz, k, batch);
  int rc = sparse_check(f);
  if (rc) return rc;
  double* Qt = d_ws;
  double* W = Qt + batch * k * kKB;
  double* part = W + (ncols * 8 + 1) / 2 * 2;
  return sparse_apply(f, d_Q, (int64_t)kKB * k, d_AQ, Qt, W, part, (cudaStream_t)stream);
}

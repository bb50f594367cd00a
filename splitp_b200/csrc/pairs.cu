// Kernel 3: subflattening.  Replaces splitp/constructions.py:108-198.
//
// A subflattening depends on the alignment only through the pairwise 4x4 joint tables N_ij of the taxa
// (SURVEY.md section 0): entry (3i+c, 3j+d) = (H N_{A_i B_j} H^T)[c,d] with H the +-1 sign table of
// constructions.py:143-161.  So the alignment is read ONCE (pair_kernel: bit-plane AND + POPC), the
// Hadamard-type basis change is n^2 batched 4x4x4 products (finalize / transform kernels) and each
// split is a gather + a small Gram + Jacobi in shared memory (subflatten_score_kernel).
#include "common.cuh"
#include "jacobi.cuh"

using namespace spb;

namespace {

__constant__ int c_H[16] = {1, -1, -1, 1, 1, 1, -1, -1, 1, -1, 1, -1, 1, 1, 1, 1};

constexpr int kPThreads = 256;
constexpr int kPW = 64;  // plane words per tile (2048 sites)

template <int PPT>
__global__ void __launch_bounds__(kPThreads) pair_kernel(const uint32_t* __restrict__ planes, const uint32_t* __restrict__ valid,
                                                         int n, int64_t Wp, int64_t word_begin, int64_t word_end,
                                                         unsigned long long* raw) {
  extern __shared__ uint32_t s_mem[];
  const int Wpad = kPW + 1;
  uint32_t* s_mask = s_mem;                       // [n*3][Wpad]
  uint32_t* s_valid = s_mask + n * 3 * Wpad;      // [kPW]
  uint8_t* s_ij = reinterpret_cast<uint8_t*>(s_valid + kPW);  // [npairs][2]
  const int tid = threadIdx.x;
  const int npairs = n * (n - 1) / 2;
  for (int p = tid; p < npairs; p += kPThreads) {
    // invert p = i*(2n-i-1)/2 + (j-i-1)
    int i = 0, rem = p;
    while (rem >= n - 1 - i) { rem -= n - 1 - i; ++i; }
    s_ij[2 * p] = (uint8_t)i;
    s_ij[2 * p + 1] = (uint8_t)(i + 1 + rem);
  }
  uint32_t cnt[PPT][9];
#pragma unroll
  for (int q = 0; q < PPT; ++q)
#pragma unroll
    for (int e = 0; e < 9; ++e) cnt[q][e] = 0;
  uint32_t marg = 0, total = 0;
  const int64_t tile0 = word_begin / kPW, tile1 = (word_end + kPW - 1) / kPW;
  for (int64_t tile = tile0 + blockIdx.x; tile < tile1; tile += gridDim.x) {
    __syncthreads();
    const int64_t wbase = tile * kPW;
    for (int idx = tid; idx < n * kPW; idx += kPThreads) {
      int j = idx / kPW, w = idx - j * kPW;
      int64_t gw = wbase + w;
      uint32_t lo = 0, hi = 0, v = 0;
      if (gw >= word_begin && gw < word_end) {
        v = __ldg(valid + gw);
        lo = __ldg(planes + ((int64_t)j * 2) * Wp + gw);
        hi = __ldg(planes + ((int64_t)j * 2 + 1) * Wp + gw);
      }
      s_mask[(j * 3 + 0) * Wpad + w] = ~hi & ~lo & v;
      s_mask[(j * 3 + 1) * Wpad + w] = ~hi & lo & v;
      s_mask[(j * 3 + 2) * Wpad + w] = hi & ~lo & v;
      if (j == 0) s_valid[w] = v;
    }
    __syncthreads();
    if (tid < n * 3) {
      const uint32_t* m = s_mask + tid * Wpad;
#pragma unroll 8
      for (int w = 0; w < kPW; ++w) marg += __popc(m[w]);
    } else if (tid == kPThreads - 1) {
#pragma unroll 8
      for (int w = 0; w < kPW; ++w) total += __popc(s_valid[w]);
    }
#pragma unroll
    for (int q = 0; q < PPT; ++q) {
      int p = tid + q * kPThreads;
      if (p < npairs) {
        const uint32_t* mi = s_mask + (int)s_ij[2 * p] * 3 * Wpad;
        const uint32_t* mj = s_mask + (int)s_ij[2 * p + 1] * 3 * Wpad;
#pragma unroll 4
        for (int w = 0; w < kPW; ++w) {
          uint32_t a0 = mi[w], a1 = mi[Wpad + w], a2 = mi[2 * Wpad + w];
          uint32_t b0 = mj[w], b1 = mj[Wpad + w], b2 = mj[2 * Wpad + w];
          cnt[q][0] += __popc(a0 & b0); cnt[q][1] += __popc(a0 & b1); cnt[q][2] += __popc(a0 & b2);
          cnt[q][3] += __popc(a1 & b0); cnt[q][4] += __popc(a1 & b1); cnt[q][5] += __popc(a1 & b2);
          cnt[q][6] += __popc(a2 & b0); cnt[q][7] += __popc(a2 & b1); cnt[q][8] += __popc(a2 & b2);
        }
      }
    }
  }
  // flush: one 64-bit atomic per counter per CTA
#pragma unroll
  for (int q = 0; q < PPT; ++q) {
    int p = tid + q * kPThreads;
    if (p < npairs) {
      int i = s_ij[2 * p], j = s_ij[2 * p + 1];
#pragma unroll
      for (int e = 0; e < 9; ++e)
        if (cnt[q][e]) atomicAdd(raw + ((int64_t)i * n + j) * 9 + e, (unsigned long long)cnt[q][e]);
    }
  }
  if (tid < n * 3 && marg) atomicAdd(raw + (int64_t)n * n * 9 + tid, (unsigned long long)marg);
  if (tid == kPThreads - 1 && total) atomicAdd(raw + (int64_t)n * n * 9 + n * 3, (unsigned long long)total);
}

// raw pair statistics -> full joint tables N[i][j][4][4] and T = H N H^T, one thread per ordered (i, j)
__global__ void finalize_kernel(const unsigned long long* __restrict__ raw, int n, double divisor, double* Nout, double* Tout,
                                double* total_out) {
  int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n * n) return;
  int i = idx / n, j = idx - i * n;
  const unsigned long long* marg = raw + (int64_t)n * n * 9;
  long long tot = (long long)marg[n * 3];
  if (divisor < 0.0) divisor = (double)tot;  // probabilities = count / usable sites (fasta.py:66-70) without a host round trip
  long long N[4][4];
  if (i == j) {
    long long s = 0;
    for (int x = 0; x < 4; ++x) for (int y = 0; y < 4; ++y) N[x][y] = 0;
    for (int x = 0; x < 3; ++x) { N[x][x] = (long long)marg[i * 3 + x]; s += N[x][x]; }
    N[3][3] = tot - s;
  } else {
    int lo = i < j ? i : j, hi = i < j ? j : i;
    const unsigned long long* r = raw + ((int64_t)lo * n + hi) * 9;
    long long M[4][4];
    long long all = 0;
    for (int x = 0; x < 3; ++x) {
      long long rs = 0;
      for (int y = 0; y < 3; ++y) { M[x][y] = (long long)r[x * 3 + y]; rs += M[x][y]; }
      M[x][3] = (long long)marg[lo * 3 + x] - rs;
      all += rs + M[x][3];
    }
    for (int y = 0; y < 3; ++y) {
      long long cs = M[0][y] + M[1][y] + M[2][y];
      M[3][y] = (long long)marg[hi * 3 + y] - cs;
      all += M[3][y];
    }
    M[3][3] = tot - all;
    for (int x = 0; x < 4; ++x) for (int y = 0; y < 4; ++y) N[x][y] = (i < j) ? M[x][y] : M[y][x];
  }
  long long HN[4][4];
  for (int c = 0; c < 4; ++c) for (int y = 0; y < 4; ++y) {
    long long s = 0;
    for (int x = 0; x < 4; ++x) s += c_H[c * 4 + x] * N[x][y];
    HN[c][y] = s;
  }
  for (int c = 0; c < 4; ++c) for (int d = 0; d < 4; ++d) {
    long long s = 0;
    for (int y = 0; y < 4; ++y) s += HN[c][y] * c_H[d * 4 + y];
    double t = (double)s;
    Tout[(int64_t)idx * 16 + c * 4 + d] = divisor > 0.0 ? t / divisor : t;
    if (Nout) {
      double v = (double)N[c][d];
      Nout[(int64_t)idx * 16 + c * 4 + d] = divisor > 0.0 ? v / divisor : v;
    }
  }
  if (idx == 0 && total_out) *total_out = divisor > 0.0 ? (double)tot / divisor : (double)tot;
}

__global__ void weighted_kernel(const uint64_t* __restrict__ keys, const double* __restrict__ vals, int64_t num, int n,
                                double* Nout) {
  int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t pat = g / n;
  int i = (int)(g - pat * n);
  if (pat >= num) return;
  uint64_t k = keys[pat];
  double v = vals[pat];
  if (v == 0.0) return;
  int x = (int)((k >> (2 * (n - 1 - i))) & 3ull);
  for (int j = 0; j < n; ++j) {
    int y = (int)((k >> (2 * (n - 1 - j))) & 3ull);
    atomicAdd(Nout + ((int64_t)i * n + j) * 16 + x * 4 + y, v);
  }
}

__global__ void transform_kernel(const double* __restrict__ Nin, int n, double* Tout, double* total_out) {
  int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n * n) return;
  const double* N = Nin + (int64_t)idx * 16;
  double HN[4][4];
  for (int c = 0; c < 4; ++c) for (int y = 0; y < 4; ++y) {
    double s = 0;
    for (int x = 0; x < 4; ++x) s += c_H[c * 4 + x] * N[x * 4 + y];
    HN[c][y] = s;
  }
  for (int c = 0; c < 4; ++c) for (int d = 0; d < 4; ++d) {
    double s = 0;
    for (int y = 0; y < 4; ++y) s += HN[c][y] * c_H[d * 4 + y];
    Tout[(int64_t)idx * 16 + c * 4 + d] = s;
  }
  if (idx == 0 && total_out) *total_out = N[0] + N[5] + N[10] + N[15];  // diagonal marginal of taxon 0
}

__device__ __forceinline__ double subflat_entry(const double* __restrict__ T, double total, int n, const uint8_t* la, int a,
                                                const uint8_t* lb, int b, int r, int c) {
  if (r < 3 * a) {
    int i = r / 3, ci = r - 3 * i, ta = la[i];
    if (c < 3 * b) {
      int j = c / 3, dj = c - 3 * j;
      return T[((int64_t)ta * n + lb[j]) * 16 + ci * 4 + dj];
    }
    return T[((int64_t)ta * n + ta) * 16 + ci * 4 + 3];
  }
  if (c < 3 * b) {
    int j = c / 3, dj = c - 3 * j, tb = lb[j];
    return T[((int64_t)tb * n + tb) * 16 + 12 + dj];
  }
  return total;
}

__global__ void subflatten_kernel(const double* __restrict__ T, const double* __restrict__ total, int n, SplitDev sp,
                                  double* out) {
  __shared__ uint8_t la[SPB_MAX_TAXA], lb[SPB_MAX_TAXA];
  if (threadIdx.x < sp.a) la[threadIdx.x] = (uint8_t)(n - 1 - sp.sh_a[threadIdx.x] / 2);
  if (threadIdx.x < sp.b) lb[threadIdx.x] = (uint8_t)(n - 1 - sp.sh_b[threadIdx.x] / 2);
  __syncthreads();
  int rows = 3 * sp.a + 1, cols = 3 * sp.b + 1;
  double tot = *total;
  for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < rows * cols; idx += gridDim.x * blockDim.x) {
    int r = idx / cols, c = idx - r * cols;
    out[idx] = subflat_entry(T, tot, n, la, sp.a, lb, sp.b, r, c);
  }
}

constexpr int kSThreads = 128;

// Score of split s of the mask lists against the pair tables T / total, by the whole CTA (staged matrix + Jacobi): the
// per-split body of subflatten_score_kernel and subflatten_score_multi_kernel.
__device__ __forceinline__ void staged_split_score(const double* __restrict__ T, double tot, int n, const uint64_t* __restrict__ masks_a,
                                                   const uint64_t* __restrict__ masks_b, int64_t s, double* M, double* G,
                                                   double* scores) {
  __shared__ JacobiScratchT<3 * (SPB_MAX_TAXA / 2) + 2> js;  // k = min(3a, 3b) + 1 <= 97
  __shared__ double lam[kJacobiMaxK], tmp[kJacobiMaxK];
  __shared__ uint8_t la[SPB_MAX_TAXA], lb[SPB_MAX_TAXA];
  __shared__ int s_a, s_b;
  const int tid = threadIdx.x;
  const uint64_t full = (n == 64) ? ~0ull : ((1ull << n) - 1ull);
  __syncthreads();
  if (tid == 0) {
    uint64_t ma = masks_a[s] & full;
    uint64_t mb = masks_b ? (masks_b[s] & full & ~ma) : (full & ~ma);
    int a = 0, b = 0;
    while (ma) { la[a++] = (uint8_t)(__ffsll((long long)ma) - 1); ma &= ma - 1; }
    while (mb) { lb[b++] = (uint8_t)(__ffsll((long long)mb) - 1); mb &= mb - 1; }
    s_a = a; s_b = b;
  }
  __syncthreads();
  const int a = s_a, b = s_b;
  const int rows = 3 * a + 1, cols = 3 * b + 1;
  const bool tr = rows > cols;          // orient so that k = smaller dimension
  const int k = tr ? cols : rows, L = tr ? rows : cols;
  const int ldm = (L + 1) | 1, ldg = jacobi_ld(k);  // odd strides: rows of M / G start on different banks
  for (int idx = tid; idx < k * L; idx += kSThreads) {
    int r = idx / L, c = idx - r * L;
    M[r * ldm + c] = tr ? subflat_entry(T, tot, n, la, a, lb, b, c, r) : subflat_entry(T, tot, n, la, a, lb, b, r, c);
  }
  __syncthreads();
  for (int idx = tid; idx < k * k; idx += kSThreads) {
    int r1 = idx / k, r2 = idx - r1 * k;
    if (r2 < r1) continue;
    const double* x = M + r1 * ldm;
    const double* y = M + r2 * ldm;
    double acc = 0.0;
    for (int c = 0; c < L; ++c) acc = fma(x[c], y[c], acc);
    G[r1 * ldg + r2] = acc;
    G[r2 * ldg + r1] = acc;
  }
  if ((k & 1) && tid <= k) { G[k * ldg + tid] = 0.0; G[tid * ldg + k] = 0.0; }  // zero padding of the odd dimension
  __syncthreads();
  jacobi_eig_smem(G, ldg, k, nullptr, 0, &js);
  sort_diag_desc(G, ldg, k, tmp, lam);
  if (tid == 0) scores[s] = (k <= 4) ? 0.0 : score_from_sorted(lam, k);
}

__global__ void __launch_bounds__(kSThreads) subflatten_score_kernel(const double* __restrict__ T, const double* __restrict__ total,
                                                                     int n, const uint64_t* __restrict__ masks_a,
                                                                     const uint64_t* __restrict__ masks_b, int64_t num,
                                                                     double* scores, int m_elems) {
  extern __shared__ __align__(16) double s_d[];
  double* M = s_d;                 // k x (L+1)
  double* G = M + m_elems;         // k x (k|1)
  const double tot = *total;
  for (int64_t s = blockIdx.x; s < num; s += gridDim.x) staged_split_score(T, tot, n, masks_a, masks_b, s, M, G, scores);
}

// Split s against the pair tables T + (s / per_table) n^2 16, totals[s / per_table]: many tables in one launch.
__global__ void __launch_bounds__(kSThreads) subflatten_score_multi_kernel(const double* __restrict__ T, const double* __restrict__ totals,
                                                                           int n, const uint64_t* __restrict__ masks_a,
                                                                           const uint64_t* __restrict__ masks_b, int64_t num,
                                                                           int64_t per_table, double* scores, int m_elems) {
  extern __shared__ __align__(16) double s_d[];
  double* M = s_d;
  double* G = M + m_elems;
  for (int64_t s = blockIdx.x; s < num; s += gridDim.x) {
    const int64_t t = s / per_table;
    staged_split_score(T + t * n * n * 16, totals[t], n, masks_a, masks_b, s, M, G, scores);
  }
}

// ---------------------------------------------------------------------------------------------------
// One WARP per split (n <= 21 taxa: k <= 31 rows, staging matrix <= 1085 doubles).  No CTA barriers at all:
//   gather M (k x L) -> Gram G = M M^T (lane r owns row r) -> Householder tridiagonalisation of G in the warp's
//   shared-memory tile (lane i owns row i; v and q are exchanged through two 32-entry arrays) -> the 4 largest
//   eigenvalues by 9-section with Sturm counts (8 lanes per eigenvalue, 18 rounds) -> score = sqrt((trace - top4) / trace).
// About 10x fewer warp instructions than the block-wide Jacobi of subflatten_score_kernel; numerics checked on the CPU
// in scripts/prototype_tridiag_top4.py (worst error 0.04 x the parity tolerance on 317 splits of a 20-taxon alignment).
// ---------------------------------------------------------------------------------------------------
constexpr int kWarpMaxTaxa = 21;
constexpr int kWarpLdg = 33;
constexpr int kWarpMElems = 1120;
constexpr int kWarpsPerCta = 4;
struct WarpScratch {
  double M[kWarpMElems];
  double G[32 * kWarpLdg];
  double v[32], q[32], d[32], e[32];
  uint8_t la[SPB_MAX_TAXA], lb[SPB_MAX_TAXA];
};

__device__ __forceinline__ double warp_sum_all(double x) {  // butterfly: every lane ends with the same bits
  for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xFFFFFFFFu, x, o);
  return x;
}
__device__ __forceinline__ double warp_min_all(double x) {
  for (int o = 16; o > 0; o >>= 1) x = fmin(x, __shfl_xor_sync(0xFFFFFFFFu, x, o));
  return x;
}
__device__ __forceinline__ double warp_max_all(double x) {
  for (int o = 16; o > 0; o >>= 1) x = fmax(x, __shfl_xor_sync(0xFFFFFFFFu, x, o));
  return x;
}

__global__ void __launch_bounds__(32 * kWarpsPerCta) subflatten_score_warp_kernel(const double* __restrict__ T, const double* __restrict__ total,
                                                                                   int n, const uint64_t* __restrict__ masks_a,
                                                                                   const uint64_t* __restrict__ masks_b, int64_t num,
                                                                                   double* scores) {
  extern __shared__ __align__(16) unsigned char s_warp_raw[];
  WarpScratch& ws = reinterpret_cast<WarpScratch*>(s_warp_raw)[threadIdx.x >> 5];
  const int lane = threadIdx.x & 31;
  const uint64_t full = (n == 64) ? ~0ull : ((1ull << n) - 1ull);
  const double tot = *total;
  const int64_t nwarps = (int64_t)gridDim.x * kWarpsPerCta;
  for (int64_t s = (int64_t)blockIdx.x * kWarpsPerCta + (threadIdx.x >> 5); s < num; s += nwarps) {
    __syncwarp();
    const uint64_t ma = masks_a[s] & full;
    const uint64_t mb = masks_b ? (masks_b[s] & full & ~ma) : (full & ~ma);
    const int a = __popcll(ma), b = __popcll(mb);
    for (int t = lane; t < 64; t += 32) {  // position lists in ascending taxon order, as the block-wide kernel builds them
      const uint64_t below = (1ull << t) - 1ull;
      if ((ma >> t) & 1ull) ws.la[__popcll(ma & below)] = (uint8_t)t;
      if ((mb >> t) & 1ull) ws.lb[__popcll(mb & below)] = (uint8_t)t;
    }
    __syncwarp();
    const int rows = 3 * a + 1, cols = 3 * b + 1;
    const bool tr = rows > cols;
    const int k = tr ? cols : rows, L = tr ? rows : cols;
    if (k <= 4) {  // at most 4 singular values: the score vanishes (phylogenetics.py:293-300)
      if (lane == 0) scores[s] = 0.0;
      continue;
    }
    const int ldm = L | 1;
    for (int idx = lane; idx < k * L; idx += 32) {
      const int r = idx / L, c = idx - r * L;
      ws.M[r * ldm + c] = tr ? subflat_entry(T, tot, n, ws.la, a, ws.lb, b, c, r) : subflat_entry(T, tot, n, ws.la, a, ws.lb, b, r, c);
    }
    __syncwarp();
    if (lane < k) {
      const double* x = ws.M + lane * ldm;
      for (int c = 0; c < k; ++c) {
        const double* y = ws.M + c * ldm;
        double acc = 0.0;
        for (int l = 0; l < L; ++l) acc = fma(x[l], y[l], acc);
        ws.G[lane * kWarpLdg + c] = acc;  // G[r][c] and G[c][r] are the same fma chain: bitwise symmetric
      }
    }
    __syncwarp();
    const double trace = warp_sum_all(lane < k ? ws.G[lane * kWarpLdg + lane] : 0.0);
    // ---- Householder tridiagonalisation: after step j, column j of the trailing block is (alpha_j, 0, ..., 0) ----
    for (int j = 0; j + 2 < k; ++j) {
      const bool below = lane > j && lane < k;
      const double x = below ? ws.G[lane * kWarpLdg + j] : 0.0;
      const double s2 = warp_sum_all(x * x);
      const double aj = __shfl_sync(0xFFFFFFFFu, x, j + 1);
      double alpha = 0.0;
      if (s2 > 0.0) {  // uniform: every lane holds the same s2
        alpha = aj > 0.0 ? -sqrt(s2) : sqrt(s2);
        const double v = (lane == j + 1) ? aj - alpha : ((lane > j + 1 && lane < k) ? x : 0.0);
        const double vn2 = warp_sum_all(v * v);
        if (vn2 > 0.0) {
          const double beta = 2.0 / vn2;
          ws.v[lane] = v;
          __syncwarp();
          double p = 0.0;
          if (below) {
            const double* row = ws.G + lane * kWarpLdg;
            for (int l = j + 1; l < k; ++l) p = fma(row[l], ws.v[l], p);
            p *= beta;
          }
          const double K = 0.5 * beta * warp_sum_all(v * p);
          const double qv = p - K * v;
          ws.q[lane] = qv;
          __syncwarp();
          if (below) {
            double* row = ws.G + lane * kWarpLdg;
            for (int l = j + 1; l < k; ++l) row[l] -= v * ws.q[l] + qv * ws.v[l];
          }
          __syncwarp();
        }
      }
      if (lane == 0) ws.e[j] = alpha;
    }
    __syncwarp();
    if (lane < k) ws.d[lane] = ws.G[lane * kWarpLdg + lane];
    if (lane == 0) ws.e[k - 2] = ws.G[(k - 1) * kWarpLdg + (k - 2)];
    __syncwarp();
    // ---- Gershgorin interval, then 9-section with Sturm counts: 8 lanes per wanted eigenvalue ----
    double lo, hi;
    {
      const double dd = lane < k ? ws.d[lane] : 0.0;
      const double e1 = (lane < k - 1) ? fabs(ws.e[lane]) : 0.0;
      const double e0 = (lane > 0 && lane < k) ? fabs(ws.e[lane - 1]) : 0.0;
      lo = warp_min_all(lane < k ? dd - e1 - e0 : 1.0e300);
      hi = warp_max_all(lane < k ? dd + e1 + e0 : -1.0e300);
    }
    const int grp = lane >> 3, m = lane & 7;
    const int want = k - 1 - grp;  // ascending index of this group's eigenvalue (k >= 5, so want >= 1)
    double glo = lo, ghi = hi;
    for (int round = 0; round < 18; ++round) {
      const double w = (ghi - glo) / 9.0;
      const double xm = glo + w * (double)(m + 1);
      int cnt = 0;
      double piv = ws.d[0] - xm;
      cnt += piv < 0.0;
      for (int i = 1; i < k; ++i) {
        if (piv == 0.0) piv = -1.0e-300;
        const double ee = ws.e[i - 1];
        piv = ws.d[i] - xm - ee * ee / piv;
        cnt += piv < 0.0;
      }
      const unsigned bal = __ballot_sync(0xFFFFFFFFu, cnt <= want);  // eigenvalue `want` is >= xm
      const int t = __popc((bal >> (grp * 8)) & 0xFFu);               // sample points at or below it (prefix property)
      const double nlo = glo + w * (double)t;
      if (t < 8) ghi = glo + w * (double)(t + 1);
      glo = nlo;
    }
    const double lam = 0.5 * (glo + ghi);
    const double l0 = __shfl_sync(0xFFFFFFFFu, lam, 0), l1 = __shfl_sync(0xFFFFFFFFu, lam, 8);
    const double l2 = __shfl_sync(0xFFFFFFFFu, lam, 16), l3 = __shfl_sync(0xFFFFFFFFu, lam, 24);
    if (lane == 0) {
      const double top = ((fmax(l0, 0.0) + fmax(l1, 0.0)) + fmax(l2, 0.0)) + fmax(l3, 0.0);
      scores[s] = trace > 0.0 ? sqrt(fmax(trace - top, 0.0) / trace) : nan("");
    }
  }
}

// ---------------------------------------------------------------------------------------------------
// Round-2 scorer: one warp per split, Gram matrix from TRIPLE tables, k = 3 min(a, b) + 1 up to 64.
//
// The first warp kernel staged the k x L subflattening in shared memory (8.7 KB of its 18.5 KB per warp -> 12 warps per
// SM) and took its Gram from it (k L / 32 dependent fma chains of length L per lane, two shared-memory loads per fma);
// ncu: ~190 k cycles per split for ~25 k warp instructions, i.e. latency-bound.  But S S^T has block structure: with
// row taxa A, column taxa B and T[x][y] = H N_xy H^T (4 x 4),
//     G[(i,c), (i',c')] = sum_{y in B} P[A_i][A_i'][y][c][c'] + m[A_i][c] m[A_i'][c'],   P[x][x'][y] = T3[x][y] T3[x'][y]^T  (3 x 3)
//     G[(i,c), last]    = sum_{y in B} R[A_i][y][c] + m[A_i][c] total,                    R[x][y][c] = sum_{d<3} T[x][y][c][d] T[y][y][3][d]
//     G[last, last]     = sum_{y in B} D[y] + total^2,        D[y] = sum_{d<3} T[y][y][3][d]^2,   m[x][c] = T[x][x][c][3]
// so after ONE pass that tabulates P, R, D, m (n^3 3x3 blocks: 576 KB at 20 taxa, 2.4 MB at 32, L2-resident), a split needs
// a b gathers of 3 doubles per row instead of the staged matrix.  Without the staging tile a warp needs k (k|1) + 4 k
// doubles (8.7 KB at k = 31), a lane owns rows i and i + 32 (k <= 64: sides up to 21 taxa, all of BASELINE config 5), and the
// Sturm counts of the bisection use the determinant recurrence p_i = (d_i - x) p_{i-1} - e_{i-1}^2 p_{i-2} (one dependent
// fma per step, rescaled by powers of two) instead of the pivot recurrence with its fp64 division per step.
// The arithmetic is modelled lane by lane in tests/warp_scorer_model.py (score_warp2_model) and checked against LAPACK.
// ---------------------------------------------------------------------------------------------------
struct TripleTables {
  const double* P;  // [n][n][n][3][3]
  const double* R;  // [n][n][3]
  const double* D;  // [n]
  const double* m;  // [n][3]
  int n;
};

__global__ void triple_tables_kernel(const double* __restrict__ T, int n, double* P, double* R, double* D, double* m) {
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t n3 = (int64_t)n * n * n;
  if (g >= n3) return;
  const int y = (int)(g % n), xp = (int)((g / n) % n), x = (int)(g / ((int64_t)n * n));
  if (x <= xp) {
    const double* Tx = T + ((int64_t)x * n + y) * 16;
    const double* Tp = T + ((int64_t)xp * n + y) * 16;
    double* out = P + (((int64_t)x * n + xp) * n + y) * 9;
    double* mir = P + (((int64_t)xp * n + x) * n + y) * 9;
    for (int c = 0; c < 3; ++c)
      for (int cp = 0; cp < 3; ++cp) {
        double acc = 0.0;
        for (int d = 0; d < 3; ++d) acc = acc + Tx[c * 4 + d] * Tp[cp * 4 + d];
        out[c * 3 + cp] = acc;
        mir[cp * 3 + c] = acc;  // the mirrored copy makes the Gram matrices bitwise symmetric
      }
  }
  if (xp == 0) {  // (x, y) pairs: R
    const double* Tx = T + ((int64_t)x * n + y) * 16;
    const double* Ty = T + ((int64_t)y * n + y) * 16;
    for (int c = 0; c < 3; ++c) {
      double acc = 0.0;
      for (int d = 0; d < 3; ++d) acc = acc + Tx[c * 4 + d] * Ty[12 + d];
      R[((int64_t)x * n + y) * 3 + c] = acc;
    }
    if (x == 0) {
      double acc = 0.0;
      for (int d = 0; d < 3; ++d) acc = acc + Ty[12 + d] * Ty[12 + d];
      D[y] = acc;
      for (int c = 0; c < 3; ++c) m[y * 3 + c] = Ty[c * 4 + 3];
    }
  }
}

constexpr int kW2MaxK = 64;
constexpr int kW2WarpsPerCta = 4;

// Householder tridiagonalisation of the symmetric k x k matrix G (leading dimension ldg, warp-private shared memory;
// lane owns rows lane + 32 t) followed by the 4 largest eigenvalues by 9-section; returns their clamped sum.
template <int ROWS>
__device__ __forceinline__ double warp2_top4(double* G, int ldg, int k, double* sv, double* sq, double* sd, double* se, int lane) {
  for (int j = 0; j + 2 < k; ++j) {
    double x[ROWS], v[ROWS];
    double part = 0.0;
#pragma unroll
    for (int t = 0; t < ROWS; ++t) {
      const int r = lane + 32 * t;
      x[t] = (r > j && r < k) ? G[r * ldg + j] : 0.0;
      part = fma(x[t], x[t], part);
    }
    const double s2 = warp_sum_all(part);
    double aj = 0.0;
#pragma unroll
    for (int t = 0; t < ROWS; ++t) {
      const double cand = __shfl_sync(0xFFFFFFFFu, x[t], (j + 1) & 31);
      if (((j + 1) >> 5) == t) aj = cand;
    }
    double alpha = 0.0;
    if (s2 > 0.0) {  // uniform: every lane holds the same s2
      alpha = aj > 0.0 ? -sqrt(s2) : sqrt(s2);
      part = 0.0;
#pragma unroll
      for (int t = 0; t < ROWS; ++t) {
        const int r = lane + 32 * t;
        v[t] = (r == j + 1) ? aj - alpha : ((r > j + 1 && r < k) ? x[t] : 0.0);
        part = fma(v[t], v[t], part);
      }
      const double vn2 = warp_sum_all(part);
      if (vn2 > 0.0) {
        const double beta = 2.0 / vn2;
#pragma unroll
        for (int t = 0; t < ROWS; ++t) sv[lane + 32 * t] = v[t];
        __syncwarp();
        double pr[ROWS];
        part = 0.0;
#pragma unroll
        for (int t = 0; t < ROWS; ++t) {
          const int r = lane + 32 * t;
          double acc = 0.0;
          if (r > j && r < k) {
            const double* row = G + r * ldg;
            for (int l = j + 1; l < k; ++l) acc = fma(row[l], sv[l], acc);
            acc *= beta;
          }
          pr[t] = acc;
          part = fma(v[t], acc, part);
        }
        const double K = 0.5 * beta * warp_sum_all(part);
        double qv[ROWS];
#pragma unroll
        for (int t = 0; t < ROWS; ++t) {
          qv[t] = pr[t] - K * v[t];
          sq[lane + 32 * t] = qv[t];
        }
        __syncwarp();
#pragma unroll
        for (int t = 0; t < ROWS; ++t) {
          const int r = lane + 32 * t;
          if (r > j && r < k) {
            double* row = G + r * ldg;
            for (int l = j + 1; l < k; ++l) row[l] -= v[t] * sq[l] + qv[t] * sv[l];
          }
        }
        __syncwarp();
      }
    }
    if (lane == 0) se[j] = alpha;
  }
  __syncwarp();
#pragma unroll
  for (int t = 0; t < ROWS; ++t) {
    const int r = lane + 32 * t;
    if (r < k) sd[r] = G[r * ldg + r];
  }
  if (lane == 0) se[k - 2] = G[(k - 1) * ldg + (k - 2)];
  __syncwarp();
  // Gershgorin interval
  double lo = 1.0e300, hi = -1.0e300;
#pragma unroll
  for (int t = 0; t < ROWS; ++t) {
    const int r = lane + 32 * t;
    if (r < k) {
      const double e1 = (r < k - 1) ? fabs(se[r]) : 0.0;
      const double e0 = (r > 0) ? fabs(se[r - 1]) : 0.0;
      lo = fmin(lo, sd[r] - e1 - e0);
      hi = fmax(hi, sd[r] + e1 + e0);
    }
  }
  lo = warp_min_all(lo);
  hi = warp_max_all(hi);
  __syncwarp();
  // The Sturm recurrence runs on the matrix scaled by 1 / max(|lo|, |hi|) (|d_i - x| <= 2, e_i^2 <= 1: at most a factor 3 of
  // growth per step, so overflow is impossible for k <= 64), with e squared once.
  const double nrm = fmax(fabs(lo), fabs(hi));
  const double inv = nrm > 0.0 ? 1.0 / nrm : 1.0;
#pragma unroll
  for (int t = 0; t < ROWS; ++t) {
    const int r = lane + 32 * t;
    if (r < k) sd[r] *= inv;
    if (r < k - 1) se[r] = (se[r] * inv) * (se[r] * inv);
  }
  __syncwarp();
  // 9-section with Sturm counts, 8 lanes per wanted eigenvalue.  Count = sign changes of the determinant sequence
  // p_{-1} = 1, p_i = (d_i - x) p_{i-1} - e_{i-1}^2 p_{i-2}.  Every 4 steps the pair (p_i, p_{i-1}) is multiplied by the power
  // of two that brings max(|p_i|, |p_{i-1}|) back to [1, 2) (exponent arithmetic, no branch): underflow -- the recurrence
  // shrinks by |d_i - x| per step -- can then never reach the denormal range (4 steps lose at most 4 x 53 + ... bits of a
  // value that starts in [1, 2)); signs are unaffected.  An exact zero p_i counts as positive (measure-zero event: x is
  // then an eigenvalue of a leading block and either side of it is a correct answer for the bisection).
  const int grp = lane >> 3, mm = lane & 7;
  const int want = k - 1 - grp;
  double glo = lo * inv, ghi = hi * inv;
  for (int round = 0; round < 18; ++round) {
    const double w = (ghi - glo) / 9.0;
    const double xm = glo + w * (double)(mm + 1);
    double pm = 1.0, p = sd[0] - xm;
    int cnt = __double2hiint(p) < 0 ? 1 : 0;
    int i = 1;
    for (; i + 3 < k; i += 4) {
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const double pn = fma(sd[i + u] - xm, p, -(se[i + u - 1] * pm));
        cnt += (int)(((unsigned)__double2hiint(pn) ^ (unsigned)__double2hiint(p)) >> 31);
        pm = p;
        p = pn;
      }
      const int ex = (__double2hiint(fmax(fabs(p), fabs(pm))) >> 20) & 0x7FF;        // biased exponent of the larger one
      const double sc = __hiloint2double((2046 - (ex > 0 ? ex : 1023)) << 20, 0);     // 2^(1023 - ex); 1 when both are zero
      p *= sc;
      pm *= sc;
    }
    for (; i < k; ++i) {
      const double pn = fma(sd[i] - xm, p, -(se[i - 1] * pm));
      cnt += (int)(((unsigned)__double2hiint(pn) ^ (unsigned)__double2hiint(p)) >> 31);
      pm = p;
      p = pn;
    }
    const unsigned bal = __ballot_sync(0xFFFFFFFFu, cnt <= want);  // eigenvalue `want` is >= xm
    const int t = __popc((bal >> (grp * 8)) & 0xFFu);               // sample points at or below it (prefix property)
    const double nlo = glo + w * (double)t;
    if (t < 8) ghi = glo + w * (double)(t + 1);
    glo = nlo;
  }
  glo *= nrm;
  ghi *= nrm;
  const double lam = 0.5 * (glo + ghi);
  const double l0 = __shfl_sync(0xFFFFFFFFu, lam, 0), l1 = __shfl_sync(0xFFFFFFFFu, lam, 8);
  const double l2 = __shfl_sync(0xFFFFFFFFu, lam, 16), l3 = __shfl_sync(0xFFFFFFFFu, lam, 24);
  return ((fmax(l0, 0.0) + fmax(l1, 0.0)) + fmax(l2, 0.0)) + fmax(l3, 0.0);
}

// Score of split s of the mask lists against one set of triple tables, by one warp (its shared-memory tile at `base`): the
// per-split body of subflatten_score_warp2_kernel and subflatten_score_warp2_multi_kernel.
__device__ __forceinline__ void warp2_split_score(const TripleTables& tt, double tot, const uint64_t* __restrict__ masks_a,
                                                  const uint64_t* __restrict__ masks_b, int64_t s, double* scores, int kcap,
                                                  uint64_t full, double* base, int lane) {
  const int ldg = kcap | 1;
  double* G = base;                       // [kcap][ldg]
  double* sv = G + (size_t)kcap * ldg;    // 4 x 64
  double* sq = sv + 64;
  double* sd = sq + 64;
  double* se = sd + 64;
  uint8_t* la = reinterpret_cast<uint8_t*>(se + 64);  // row-side taxa (<= 21), then column-side taxa (<= 64)
  uint8_t* lb = la + 32;
  const int n = tt.n;
  {
    uint64_t ma = masks_a[s] & full;
    uint64_t mb = masks_b ? (masks_b[s] & full & ~ma) : (full & ~ma);
    if (__popcll(ma) > __popcll(mb)) { const uint64_t t = ma; ma = mb; mb = t; }  // rows = the smaller side (S S^T and S^T S share
    const int a = __popcll(ma), b = __popcll(mb);                                 // their non-zero eigenvalues)
    const int k = 3 * a + 1;
    if (k <= 4 || b == 0) {  // at most 4 singular values: the score vanishes (phylogenetics.py:293-300)
      if (lane == 0) scores[s] = 0.0;
      return;
    }
    if (k > kcap) {  // not reachable through spb_subflatten_score_tables (the host routes such batches elsewhere)
      if (lane == 0) scores[s] = nan("");
      return;
    }
    for (int t = lane; t < 64; t += 32) {  // position lists in ascending taxon order
      const uint64_t below = (1ull << t) - 1ull;
      if ((ma >> t) & 1ull) la[__popcll(ma & below)] = (uint8_t)t;
      if ((mb >> t) & 1ull) lb[__popcll(mb & below)] = (uint8_t)t;
    }
    __syncwarp();
    // ---- Gram matrix from the triple tables.  Work items (i, i' >= i, c) = 3 entries G[3i + c][3i' .. 3i' + 2], dealt round-robin
    // to the lanes and written to both triangles (bitwise symmetric by construction); then the last row / column. ----
    {
      const int npairs = a * (a + 1) / 2;
      for (int t = lane; t < 3 * npairs; t += 32) {
        const int q = t / 3, c = t - 3 * q;
        int i = 0, rem = q;
        while (rem >= a - i) { rem -= a - i; ++i; }  // row-major over the upper triangle: row i holds i' = i .. a - 1
        const int ip = i + rem;
        const int x = la[i], xp = la[ip];
        const double* src = tt.P + (((int64_t)x * n + xp) * n) * 9 + c * 3;
        double a0 = 0.0, a1 = 0.0, a2 = 0.0;
        int jj = 0;
        for (; jj + 1 < b; jj += 2) {  // two column taxa per iteration: six independent loads in flight
          const double* q0 = src + (int)lb[jj] * 9;
          const double* q1 = src + (int)lb[jj + 1] * 9;
          const double u0 = __ldg(q0), u1 = __ldg(q0 + 1), u2 = __ldg(q0 + 2);
          const double v0 = __ldg(q1), v1 = __ldg(q1 + 1), v2 = __ldg(q1 + 2);
          a0 = (a0 + u0) + v0; a1 = (a1 + u1) + v1; a2 = (a2 + u2) + v2;
        }
        if (jj < b) {
          const double* q0 = src + (int)lb[jj] * 9;
          a0 = a0 + __ldg(q0); a1 = a1 + __ldg(q0 + 1); a2 = a2 + __ldg(q0 + 2);
        }
        const double mxc = tt.m[x * 3 + c];
        const double g0 = fma(mxc, tt.m[xp * 3], a0), g1 = fma(mxc, tt.m[xp * 3 + 1], a1), g2 = fma(mxc, tt.m[xp * 3 + 2], a2);
        const int r = 3 * i + c, cc = 3 * ip;
        G[r * ldg + cc] = g0; G[r * ldg + cc + 1] = g1; G[r * ldg + cc + 2] = g2;
        G[cc * ldg + r] = g0; G[(cc + 1) * ldg + r] = g1; G[(cc + 2) * ldg + r] = g2;
      }
      for (int r = lane; r < 3 * a; r += 32) {  // last column / row
        const int i = r / 3, c = r - 3 * i;
        const int x = la[i];
        double acc = 0.0;
        for (int jj = 0; jj < b; ++jj) acc = acc + __ldg(tt.R + ((int64_t)x * n + lb[jj]) * 3 + c);
        const double g = fma(tt.m[x * 3 + c], tot, acc);
        G[r * ldg + 3 * a] = g;
        G[3 * a * ldg + r] = g;
      }
      if (lane == 0) {
        double acc = 0.0;
        for (int jj = 0; jj < b; ++jj) acc = acc + __ldg(tt.D + lb[jj]);
        G[3 * a * ldg + 3 * a] = fma(tot, tot, acc);
      }
    }
    __syncwarp();
    double part = 0.0;
    for (int r = lane; r < k; r += 32) part += G[r * ldg + r];
    const double trace = warp_sum_all(part);
    const double top = (k <= 32) ? warp2_top4<1>(G, ldg, k, sv, sq, sd, se, lane) : warp2_top4<2>(G, ldg, k, sv, sq, sd, se, lane);
    if (lane == 0) scores[s] = trace > 0.0 ? sqrt(fmax(trace - top, 0.0) / trace) : nan("");
  }
}

__global__ void __launch_bounds__(32 * kW2WarpsPerCta) subflatten_score_warp2_kernel(const TripleTables tt, const double* __restrict__ total,
                                                                                    const uint64_t* __restrict__ masks_a,
                                                                                    const uint64_t* __restrict__ masks_b, int64_t num,
                                                                                    double* scores, int kcap, int warp_doubles) {
  extern __shared__ __align__(16) double s_w2[];
  double* base = s_w2 + (size_t)(threadIdx.x >> 5) * warp_doubles;
  const int lane = threadIdx.x & 31;
  const uint64_t full = (tt.n == 64) ? ~0ull : ((1ull << tt.n) - 1ull);
  const double tot = *total;
  const int64_t nwarps = (int64_t)gridDim.x * kW2WarpsPerCta;
  for (int64_t s = (int64_t)blockIdx.x * kW2WarpsPerCta + (threadIdx.x >> 5); s < num; s += nwarps) {
    __syncwarp();
    warp2_split_score(tt, tot, masks_a, masks_b, s, scores, kcap, full, base, lane);
  }
}

// Split s against the triple tables at tables + (s / per_table) table_doubles (layout of spb_subflatten_score_tables) and
// totals[s / per_table]: many tables in one launch.  No __launch_bounds__: with it ptxas holds the kernel to 64 registers and
// spills 4 bytes; without it it takes 66 registers, which still fit 7 CTAs of 4 warps on an SM.
__global__ void subflatten_score_warp2_multi_kernel(
    const double* __restrict__ tables, int64_t table_doubles, const double* __restrict__ totals, int n,
    const uint64_t* __restrict__ masks_a, const uint64_t* __restrict__ masks_b, int64_t num, int64_t per_table, double* scores,
    int kcap, int warp_doubles) {
  extern __shared__ __align__(16) double s_w2[];
  double* base = s_w2 + (size_t)(threadIdx.x >> 5) * warp_doubles;
  const int lane = threadIdx.x & 31;
  const int64_t nn = n;
  const uint64_t full = (n == 64) ? ~0ull : ((1ull << n) - 1ull);
  const int64_t nwarps = (int64_t)gridDim.x * kW2WarpsPerCta;
  for (int64_t s = (int64_t)blockIdx.x * kW2WarpsPerCta + (threadIdx.x >> 5); s < num; s += nwarps) {
    const int64_t t = s / per_table;
    const double* P = tables + t * table_doubles;
    const double* R = P + nn * nn * nn * 9;
    const double* D = R + nn * nn * 3;
    const TripleTables tt{P, R, D, D + nn, n};
    __syncwarp();
    warp2_split_score(tt, totals[t], masks_a, masks_b, s, scores, kcap, full, base, lane);
  }
}

// The same eigen stage for symmetric k x k matrices that already exist in global memory (k <= 64): the Gram matrices of the
// thin size classes of a count flattening (2|10, 3|9 of 12 taxa: k = 16, 64).  One warp per matrix: copy to the warp-private tile,
// trace, Householder + 9-section.  Replaces the cyclic Jacobi kernel (score.cu: 0.58 ms per launch whatever the batch, two
// barriers per rotation round) where only the score is wanted.
__global__ void __launch_bounds__(32 * kW2WarpsPerCta) gram_score_warp_kernel(const double* __restrict__ Gin, int k, int64_t ld, int64_t batch,
                                                                             double* __restrict__ scores, int warp_doubles) {
  extern __shared__ __align__(16) double s_w2[];
  double* base = s_w2 + (size_t)(threadIdx.x >> 5) * warp_doubles;
  const int ldg = k | 1;
  double* G = base;                    // [k][ldg]
  double* sv = G + (size_t)k * ldg;    // 4 x 64
  double* sq = sv + 64;
  double* sd = sq + 64;
  double* se = sd + 64;
  const int lane = threadIdx.x & 31;
  const int64_t nwarps = (int64_t)gridDim.x * kW2WarpsPerCta;
  for (int64_t s = (int64_t)blockIdx.x * kW2WarpsPerCta + (threadIdx.x >> 5); s < batch; s += nwarps) {
    __syncwarp();
    const double* src = Gin + s * ld * ld;
    for (int t = lane; t < k * k; t += 32) {
      const int r = t / k, c = t - r * k;
      G[r * ldg + c] = (c >= r) ? src[(int64_t)r * ld + c] : src[(int64_t)c * ld + r];  // upper triangle, mirrored: bitwise symmetric
    }
    __syncwarp();
    double part = 0.0;
    for (int r = lane; r < k; r += 32) part += G[r * ldg + r];
    const double trace = warp_sum_all(part);
    const double top = (k <= 32) ? warp2_top4<1>(G, ldg, k, sv, sq, sd, se, lane) : warp2_top4<2>(G, ldg, k, sv, sq, sd, se, lane);
    if (lane == 0) scores[s] = trace > 0.0 ? sqrt(fmax(trace - top, 0.0) / trace) : nan("");
  }
}

inline size_t subflat_smem(int n, int* m_elems) {
  // the widest staging matrix over ALL side sizes: k x ((L + 1) | 1) with k = 3 min(a, b) + 1, L = 3 max(a, b) + 1.  It is
  // NOT maximised at the balanced split (22 taxa: 10|12 needs 31 x 39 = 1209 doubles, 11|11 only 34 x 35 = 1190: round 1
  // sized the buffer from the balanced split and the 10|12 matrices ran 19 doubles into G -- found by
  // tests/test_gpu_parity_r2.py::test_subflatten_score_stratified[22]); the Jacobi tile is largest at the balanced split
  int worst = 0;
  for (int a = 1; a <= n / 2; ++a) {
    const int k = 3 * a + 1, L = 3 * (n - a) + 1;
    const int m = k * ((L + 1) | 1);
    if (m > worst) worst = m;
  }
  if (worst < 4 * 7) worst = 4 * 7;
  *m_elems = worst;
  const int kmax = 3 * (n / 2) + 1;
  return ((size_t)*m_elems + (size_t)jacobi_dim(kmax) * jacobi_ld(kmax)) * sizeof(double);
}

}  // namespace

extern "C" int64_t spb_pair_raw_words(int n_taxa) { return (int64_t)n_taxa * n_taxa * 9 + (int64_t)n_taxa * 3 + 1; }

extern "C" int spb_pair_tables(const uint32_t* d_planes, const uint32_t* d_valid, int n_taxa, int64_t plane_words,
                               int64_t word_begin, int64_t word_end, uint64_t* d_raw, void* stream) {
  SPB_REQUIRE(d_planes && d_valid && d_raw, "spb_pair_tables: NULL buffer");
  SPB_REQUIRE(n_taxa >= 1 && n_taxa <= SPB_MAX_TAXA, "spb_pair_tables: n_taxa out of range");
  SPB_REQUIRE(word_begin >= 0 && word_end <= plane_words && word_begin <= word_end, "spb_pair_tables: bad word range");
  if (word_end == word_begin) return SPB_OK;
  cudaStream_t st = (cudaStream_t)stream;
  int npairs = n_taxa * (n_taxa - 1) / 2;
  size_t smem = ((size_t)n_taxa * 3 * (kPW + 1) + kPW) * 4 + (size_t)(npairs > 0 ? npairs : 1) * 2 + 16;
  int64_t tiles = (word_end + kPW - 1) / kPW - word_begin / kPW;
  int64_t grid = (int64_t)sm_count() * 2;
  if (grid > tiles) grid = tiles;
#define SPB_PAIR_LAUNCH(PPT)                                                                                          \
  do {                                                                                                                \
    SPB_CUDA(cudaFuncSetAttribute(pair_kernel<PPT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));          \
    pair_kernel<PPT><<<(unsigned)grid, kPThreads, smem, st>>>(d_planes, d_valid, n_taxa, plane_words, word_begin,     \
                                                              word_end, (unsigned long long*)d_raw);                  \
  } while (0)
  if (npairs <= kPThreads) SPB_PAIR_LAUNCH(1);
  else if (npairs <= 2 * kPThreads) SPB_PAIR_LAUNCH(2);
  else if (npairs <= 4 * kPThreads) SPB_PAIR_LAUNCH(4);
  else SPB_PAIR_LAUNCH(8);
#undef SPB_PAIR_LAUNCH
  SPB_LAUNCH_CHECK();
  return SPB_OK;
}

extern "C" int spb_pair_finalize(const uint64_t* d_raw, int n_taxa, double divisor, double* d_N, double* d_T, double* d_total,
                                 void* stream) {
  SPB_REQUIRE(d_raw && d_T && n_taxa >= 1 && n_taxa <= SPB_MAX_TAXA, "spb_pair_finalize: bad arguments");
  int nn = n_taxa * n_taxa;
  finalize_kernel<<<(nn + 127) / 128, 128, 0, (cudaStream_t)stream>>>((const unsigned long long*)d_raw, n_taxa, divisor, d_N, d_T,
                                                                     d_total);
  SPB_LAUNCH_CHECK();
  return SPB_OK;
}

extern "C" int spb_pair_tables_weighted(const uint64_t* d_keys, const double* d_vals, int64_t num, int n_taxa, double* d_N,
                                        void* stream) {
  SPB_REQUIRE(d_N && n_taxa >= 1 && n_taxa <= 31, "spb_pair_tables_weighted: uint64 keys need n_taxa <= 31");
  if (num <= 0) return SPB_OK;
  SPB_REQUIRE(d_keys && d_vals, "spb_pair_tables_weighted: NULL buffer");
  int64_t work = num * n_taxa;
  weighted_kernel<<<(unsigned)((work + 255) / 256), 256, 0, (cudaStream_t)stream>>>(d_keys, d_vals, num, n_taxa, d_N);
  SPB_LAUNCH_CHECK();
  return SPB_OK;
}

extern "C" int spb_pair_transform(const double* d_N, int n_taxa, double* d_T, double* d_total, void* stream) {
  SPB_REQUIRE(d_N && d_T && n_taxa >= 1 && n_taxa <= SPB_MAX_TAXA, "spb_pair_transform: bad arguments");
  int nn = n_taxa * n_taxa;
  transform_kernel<<<(nn + 127) / 128, 128, 0, (cudaStream_t)stream>>>(d_N, n_taxa, d_T, d_total);
  SPB_LAUNCH_CHECK();
  return SPB_OK;
}

extern "C" int spb_subflatten(const double* d_T, const double* d_total, int n_taxa, const spb_split* split, double* d_out,
                              void* stream) {
  SplitDev sp;
  int rc = make_split_dev(split, &sp, false);
  if (rc) return rc;
  SPB_REQUIRE(d_T && d_total && d_out && sp.n == n_taxa, "spb_subflatten: bad arguments");
  int cells = (3 * sp.a + 1) * (3 * sp.b + 1);
  int blocks = (cells + 127) / 128;
  if (blocks > 64) blocks = 64;
  subflatten_kernel<<<blocks, 128, 0, (cudaStream_t)stream>>>(d_T, d_total, n_taxa, sp, d_out);
  SPB_LAUNCH_CHECK();
  return SPB_OK;
}

extern "C" int64_t spb_subflatten_tables_doubles(int n_taxa) {
  const int64_t n = n_taxa;
  return n * n * n * 9 + n * n * 3 + n + n * 3 + 8;
}

// Scores through the triple-table warp kernel (header: spb_subflatten_score_tables).
extern "C" int spb_subflatten_score_tables(const double* d_T, const double* d_total, int n_taxa, const uint64_t* d_masks_a,
                                           const uint64_t* d_masks_b, int64_t num, double* d_scores, double* d_tables,
                                           int tables_ready, void* stream) {
  SPB_REQUIRE(d_T && d_total && d_tables && n_taxa >= 2 && n_taxa <= SPB_MAX_TAXA, "spb_subflatten_score_tables: bad arguments");
  const int kcap = 3 * (n_taxa / 2) + 1;  // largest k = 3 min(a, b) + 1 over all splits of n taxa
  SPB_REQUIRE(kcap <= kW2MaxK, "spb_subflatten_score_tables: handles sides of up to %d taxa (n <= %d); use spb_subflatten_score",
              (kW2MaxK - 1) / 3, 2 * ((kW2MaxK - 1) / 3) + 1);
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t n = n_taxa;
  double* P = d_tables;
  double* R = P + n * n * n * 9;
  double* D = R + n * n * 3;
  double* m = D + n;
  if (!tables_ready) {
    const int64_t n3 = n * n * n;
    triple_tables_kernel<<<(unsigned)((n3 + 127) / 128), 128, 0, st>>>(d_T, n_taxa, P, R, D, m);
    SPB_LAUNCH_CHECK();
  }
  if (num <= 0) return SPB_OK;
  SPB_REQUIRE(d_masks_a && d_scores, "spb_subflatten_score_tables: NULL buffer");
  const int ldg = kcap | 1;
  const int warp_doubles = kcap * ldg + 4 * 64 + 16;  // G, v / q / d / e, 96 bytes of taxon lists (padded to 128)
  const size_t smem = (size_t)kW2WarpsPerCta * warp_doubles * sizeof(double);
  SPB_CUDA(cudaFuncSetAttribute(subflatten_score_warp2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int occ = 1;
  SPB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, subflatten_score_warp2_kernel, 32 * kW2WarpsPerCta, smem));
  if (occ < 1) occ = 1;
  int64_t grid = (int64_t)sm_count() * occ;
  const int64_t need = (num + kW2WarpsPerCta - 1) / kW2WarpsPerCta;
  if (grid > need) grid = need;
  TripleTables tt{P, R, D, m, n_taxa};
  subflatten_score_warp2_kernel<<<(unsigned)grid, 32 * kW2WarpsPerCta, smem, st>>>(tt, d_total, d_masks_a, d_masks_b, num, d_scores, kcap,
                                                                               warp_doubles);
  SPB_LAUNCH_CHECK();
  return SPB_OK;
}

// Many tables per launch through the triple-table warp kernel (header: spb_subflatten_score_tables_multi).
extern "C" int spb_subflatten_score_tables_multi(const double* d_tables, const double* d_totals, int n_taxa, const uint64_t* d_masks_a,
                                                 const uint64_t* d_masks_b, int64_t num, int64_t per_table, double* d_scores,
                                                 void* stream) {
  SPB_REQUIRE(n_taxa >= 2 && n_taxa <= SPB_MAX_TAXA && per_table >= 1, "spb_subflatten_score_tables_multi: bad arguments");
  const int kcap = 3 * (n_taxa / 2) + 1;
  SPB_REQUIRE(kcap <= kW2MaxK, "spb_subflatten_score_tables_multi: handles up to %d taxa; use spb_subflatten_score_multi",
              2 * ((kW2MaxK - 1) / 3) + 1);
  if (num <= 0) return SPB_OK;
  SPB_REQUIRE(d_tables && d_totals && d_masks_a && d_scores, "spb_subflatten_score_tables_multi: NULL buffer");
  const int ldg = kcap | 1;
  const int warp_doubles = kcap * ldg + 4 * 64 + 16;
  const size_t smem = (size_t)kW2WarpsPerCta * warp_doubles * sizeof(double);
  SPB_CUDA(cudaFuncSetAttribute(subflatten_score_warp2_multi_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int occ = 1;
  SPB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, subflatten_score_warp2_multi_kernel, 32 * kW2WarpsPerCta, smem));
  if (occ < 1) occ = 1;
  int64_t grid = (int64_t)sm_count() * occ;
  const int64_t need = (num + kW2WarpsPerCta - 1) / kW2WarpsPerCta;
  if (grid > need) grid = need;
  subflatten_score_warp2_multi_kernel<<<(unsigned)grid, 32 * kW2WarpsPerCta, smem, (cudaStream_t)stream>>>(
      d_tables, spb_subflatten_tables_doubles(n_taxa), d_totals, n_taxa, d_masks_a, d_masks_b, num, per_table, d_scores, kcap, warp_doubles);
  SPB_LAUNCH_CHECK();
  return SPB_OK;
}

namespace spb {
int score_gram_warp_launch(const double* d_G, int k, int64_t ld, int64_t batch, double* d_scores, cudaStream_t st) {
  const int warp_doubles = k * (k | 1) + 4 * 64;
  const size_t smem = (size_t)kW2WarpsPerCta * warp_doubles * sizeof(double);
  SPB_CUDA(cudaFuncSetAttribute(gram_score_warp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int occ = 1;
  SPB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, gram_score_warp_kernel, 32 * kW2WarpsPerCta, smem));
  if (occ < 1) occ = 1;
  int64_t grid = (int64_t)sm_count() * occ;
  const int64_t need = (batch + kW2WarpsPerCta - 1) / kW2WarpsPerCta;
  if (grid > need) grid = need;
  gram_score_warp_kernel<<<(unsigned)grid, 32 * kW2WarpsPerCta, smem, st>>>(d_G, k, ld, batch, d_scores, warp_doubles);
  SPB_LAUNCH_CHECK();
  return SPB_OK;
}
}  // namespace spb

extern "C" int spb_subflatten_score(const double* d_T, const double* d_total, int n_taxa, const uint64_t* d_masks_a,
                                    const uint64_t* d_masks_b, int64_t num, double* d_scores, void* stream) {
  SPB_REQUIRE(d_T && d_total && n_taxa >= 2 && n_taxa <= SPB_MAX_TAXA, "spb_subflatten_score: bad arguments");
  if (num <= 0) return SPB_OK;
  SPB_REQUIRE(d_masks_a && d_scores, "spb_subflatten_score: NULL buffer");
  if (n_taxa <= kWarpMaxTaxa) {
    const size_t wsmem = (size_t)kWarpsPerCta * sizeof(WarpScratch);
    SPB_CUDA(cudaFuncSetAttribute(subflatten_score_warp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)wsmem));
    int wocc = 1;
    SPB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&wocc, subflatten_score_warp_kernel, 32 * kWarpsPerCta, wsmem));
    if (wocc < 1) wocc = 1;
    int64_t wgrid = (int64_t)sm_count() * wocc;
    const int64_t need = (num + kWarpsPerCta - 1) / kWarpsPerCta;
    if (wgrid > need) wgrid = need;
    subflatten_score_warp_kernel<<<(unsigned)wgrid, 32 * kWarpsPerCta, wsmem, (cudaStream_t)stream>>>(d_T, d_total, n_taxa, d_masks_a,
                                                                                                   d_masks_b, num, d_scores);
    SPB_LAUNCH_CHECK();
    return SPB_OK;
  }
  int m_elems = 0;
  size_t smem = subflat_smem(n_taxa, &m_elems);
  SPB_CUDA(cudaFuncSetAttribute(subflatten_score_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int occ = 1;
  SPB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, subflatten_score_kernel, kSThreads, smem));
  if (occ < 1) occ = 1;
  int64_t grid = (int64_t)sm_count() * occ;
  if (grid > num) grid = num;
  subflatten_score_kernel<<<(unsigned)grid, kSThreads, smem, (cudaStream_t)stream>>>(d_T, d_total, n_taxa, d_masks_a, d_masks_b,
                                                                                    num, d_scores, m_elems);
  SPB_LAUNCH_CHECK();
  return SPB_OK;
}

// Many tables per launch through the staged CTA kernel (header: spb_subflatten_score_multi).
extern "C" int spb_subflatten_score_multi(const double* d_T, const double* d_totals, int n_taxa, const uint64_t* d_masks_a,
                                          const uint64_t* d_masks_b, int64_t num, int64_t per_table, double* d_scores, void* stream) {
  SPB_REQUIRE(n_taxa > kWarpMaxTaxa && n_taxa <= SPB_MAX_TAXA && per_table >= 1, "spb_subflatten_score_multi: bad arguments");
  if (num <= 0) return SPB_OK;
  SPB_REQUIRE(d_T && d_totals && d_masks_a && d_scores, "spb_subflatten_score_multi: NULL buffer");
  int m_elems = 0;
  size_t smem = subflat_smem(n_taxa, &m_elems);
  SPB_CUDA(cudaFuncSetAttribute(subflatten_score_multi_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int occ = 1;
  SPB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, subflatten_score_multi_kernel, kSThreads, smem));
  if (occ < 1) occ = 1;
  int64_t grid = (int64_t)sm_count() * occ;
  if (grid > num) grid = num;
  subflatten_score_multi_kernel<<<(unsigned)grid, kSThreads, smem, (cudaStream_t)stream>>>(d_T, d_totals, n_taxa, d_masks_a, d_masks_b,
                                                                                          num, per_table, d_scores, m_elems);
  SPB_LAUNCH_CHECK();
  return SPB_OK;
}

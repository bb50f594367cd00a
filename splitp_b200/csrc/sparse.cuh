// Sparse flattenings as an operator of the block-Krylov solver (sparse.cu, used by score.cu).
//
// A batch of `batch` flattenings F_b (k_b x C_b, k_b <= k) is stored twice, both over GLOBAL indices:
//   rows    r_glob = b * k + r      (r < k; rows k_b <= r < k of a matrix are empty: they add zero eigenvalues only)
//   columns c_glob = base_b + c     (the columns of all matrices concatenated, ncols in all)
//   CSR: row_off [batch * k + 1], row_col [nnz] (global column), row_val [nnz], entries grouped by global row
//   CSC: col_off [ncols + 1],     col_row [nnz] (global row),    col_val [nnz], entries grouped by global column
// G Q = F (F^T Q) is applied in two gathers: W = F^T Q (one 8-vector per column) from the transposed block
// Qt [batch * k][8], then AQ = F W into the solver's [8][k] layout.
#pragma once
#include "common.cuh"

namespace spb {

struct SparseBatch {
  const int64_t* row_off;
  const int32_t* row_col;
  const double* row_val;
  const int64_t* col_off;
  const int32_t* col_row;
  const double* col_val;
  int64_t ncols, nnz;
  int k, batch;
};

// Entries per piece of a segment sum (see sparse.cu): a segment of L entries is cut into about L / kSparsePiece pieces.
constexpr int kSparsePiece = 16;

// doubles of partial sums one product needs (pieces of the larger of the two segment lists, 8 doubles each)
inline int64_t sparse_part_doubles(const SparseBatch& f) {
  const int64_t nseg = (int64_t)f.batch * f.k > f.ncols ? (int64_t)f.batch * f.k : f.ncols;
  return 8 * (nseg + f.nnz / kSparsePiece + 1);
}

int sparse_check(const SparseBatch& f);
// W [ncols][8] = F^T Q and AQ [b][c][r] (stride strideQ per matrix, [8][k] inside) = F W; Qt [batch * k][8]
int sparse_product_launch(const SparseBatch& f, const double* Qt, double* W, double* AQ, int64_t strideQ, double* part,
                          cudaStream_t st);
// diag [batch * k]: sum of v^2 over every CSR row (the diagonal of G = F F^T)
int sparse_diag_launch(const SparseBatch& f, double* diag, cudaStream_t st);

}  // namespace spb

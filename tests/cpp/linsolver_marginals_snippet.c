/* Compiled (never run) by tests/test_linsolver_marginals_host.py with a plain C compiler: the
 * s3o_linsolver_solve_pattern declaration must be valid C, and the two call forms of a g2o LinearSolver adapter
 * (solveBlocks: every diagonal block; solvePattern: chosen block pairs) must type-check against it. */
#include <stddef.h>
#include <stdint.h>

#include "sim3opt_b200.h"

int covariances_of_a(s3o_linsolver *s, int n, const int32_t *colptr, const int32_t *rowidx,
                     const double *blocks /* colptr[n] x 7 x 7, column-major (Eigen) */, double *diag /* n x 7 x 7 */,
                     int n_pairs, const int32_t *rows, const int32_t *cols, double *out /* n_pairs x 7 x 7 */) {
    int rc = s3o_linsolver_solve_pattern(s, n, colptr, rowidx, blocks, 1, n, NULL, NULL, diag);
    if (rc == S3O_ERR_SOLVE) return 1;          /* A is not positive definite: g2o's solvePattern returns false */
    if (rc != S3O_OK) return rc;
    return s3o_linsolver_solve_pattern(s, n, colptr, rowidx, blocks, 1, n_pairs, rows, cols, out);
}

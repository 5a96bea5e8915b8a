/* Compiled (never run) by tests/test_marginals_host.py with a plain C compiler: the s3o_compute_marginals declaration
 * must be valid C, and the two call forms (every diagonal block / chosen pairs) must type-check against it. */
#include <stddef.h>
#include <stdint.h>

#include "sim3opt_b200.h"

int marginals_after_optimize(s3o_problem *prob, int n_free, double *diag /* n_free x 7 x 7 */, const int32_t *rows,
                             const int32_t *cols, int n_pairs, double *blocks /* n_pairs x 7 x 7 */) {
    int iters = 0;
    double chi2 = 0, lambda = 0;
    if (s3o_optimize(prob, 20, 0.0, &iters, &chi2, &lambda, NULL, 0) != S3O_OK) return -1;
    int rc = s3o_compute_marginals(prob, n_free, NULL, NULL, diag);
    if (rc == S3O_ERR_SOLVE) return 1;          /* a connected component without a fixed vertex */
    if (rc != S3O_OK) return rc;
    return s3o_compute_marginals(prob, n_pairs, rows, cols, blocks);
}

/* Compiled (never run) by tests/test_ba_marginals_host.py with a plain C compiler: the s3o_ba_compute_marginals
 * declaration must be valid C, and the two call forms (every diagonal block / chosen pairs) must type-check against it. */
#include <stddef.h>
#include <stdint.h>

#include "sim3opt_b200.h"

int ba_marginals_after_optimize(s3o_problem *prob, double *diag /* 36 ncf + 9 npf */, const int32_t *rows,
                                const int32_t *cols, int n_pairs, double *blocks) {
    int iters = 0, ncf = 0, npf = 0, nb = 0;
    int64_t ncon = 0;
    double chi2 = 0, lambda = 0;
    if (s3o_optimize(prob, 20, 0.0, &iters, &chi2, &lambda, NULL, 0) != S3O_OK) return -1;
    if (s3o_ba_get_sizes(prob, &ncf, &npf, &nb, &ncon) != S3O_OK) return -1;
    int rc = s3o_ba_compute_marginals(prob, ncf + npf, NULL, NULL, diag);
    if (rc == S3O_ERR_SOLVE) return 1;          /* a free gauge or a point seen by one camera */
    if (rc != S3O_OK) return rc;
    return s3o_ba_compute_marginals(prob, n_pairs, rows, cols, blocks);
}

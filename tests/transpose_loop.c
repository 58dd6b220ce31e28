/*
 * tests/transpose_loop.c -- TEST INFRASTRUCTURE ONLY: the sequential transposed CSR loop, y = A^T x,
 *
 *     for r: for j in row r: y[col_ind[j]] += val[j] * x[r]        (y zeroed first)
 *
 * written the way oracle/smvp_oracle.c writes the forward loop (main-cli.c:410-416) and compiled like it
 * (-ffp-contract=off: every product is rounded before it is added).  Column c of y receives its terms in
 * ascending row order, each added to the running sum from +0.0.  tests/test_transpose.py compiles it.
 */
#include <stdint.h>

void oracle_csr_mult_transpose(int32_t rows, int32_t cols, const int32_t *row_ptr, const int32_t *col_ind,
                               const double *val, const double *x, double *y)
{
    int32_t r, j, c;
    for (c = 0; c < cols; c++)
        y[c] = 0.0;
    for (r = 0; r < rows; r++)
        for (j = row_ptr[r]; j < row_ptr[r + 1]; j++)
            y[col_ind[j]] += val[j] * x[r];
}

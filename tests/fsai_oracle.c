/*
 * Test oracle of the FSAI kernel (csrc/fsai.cu, dp_fsai_f64): a plain sequential C restatement of its arithmetic,
 * loaded by tests/fsai_oracle.py. Compiled with -ffp-contract=off: every product, difference, quotient and square root
 * is rounded separately, as the kernel rounds them with __dmul_rn / __dsub_rn / __ddiv_rn / __dsqrt_rn, so the two
 * agree bit for bit.
 */
#include <math.h>

/* FSAI factor on a given pattern, the arithmetic order of csrc/fsai.cu (dp_fsai_f64, DESIGN §3.6). A: full symmetric
 * CSR, sorted rows. u_rowptr / u_col: CSR of U = L^T, row i = (i < j_1 < ... < j_{k-1}), k <= 32. Row i of U gets
 * y_p / sqrt(y_0) with A[J,J] y = e_0, by a Cholesky factor R of A[J,J] (left-looking by columns), forward and backward
 * substitution, every sum subtracted term by term in ascending index, every operation rounded separately.
 * fp32: values rounded once to fp32. Returns 0, 5 (structure: see dp_fsai_f64) or 7 (a pivot that is not positive)
 * for the first row that fails. */
int oracle_fsai(int n, const int* a_rowptr, const int* a_col, const double* a_val, const int* u_rowptr,
                const int* u_col, int fp32, double* u_val) {
    double r[32][32], w[32], y[32];
    for (int i = 0; i < n; ++i) {
        const int rs = u_rowptr[i], k = u_rowptr[i + 1] - rs;
        const int* J = u_col + rs;
        if (k < 1 || k > 32 || J[0] != i) return 5;
        for (int p = 1; p < k; ++p)
            if (J[p] <= J[p - 1] || J[p] >= n) return 5;
        for (int p = 0; p < k; ++p) { /* S_pq = A[j_p, j_q], q <= p */
            int diag = 0, a = a_rowptr[J[p]], q = 0;
            for (int t = 0; t <= p; ++t) r[p][t] = 0.0;
            while (a < a_rowptr[J[p] + 1] && q <= p) {
                if (a_col[a] == J[q]) {
                    r[p][q] = a_val[a];
                    diag = q == p;
                    ++a; ++q;
                } else if (a_col[a] < J[q]) ++a; else ++q;
            }
            if (!diag) return 5;
        }
        for (int q = 0; q < k; ++q) { /* Cholesky, column q */
            double d = r[q][q];
            for (int t = 0; t < q; ++t) {
                double m = r[q][t] * r[q][t];
                d = d - m;
            }
            if (!(d > 0.0)) return 7;
            double rqq = sqrt(d);
            for (int p = q + 1; p < k; ++p) {
                double s = r[p][q];
                for (int t = 0; t < q; ++t) {
                    double m = r[p][t] * r[q][t];
                    s = s - m;
                }
                r[p][q] = s / rqq;
            }
            r[q][q] = rqq;
        }
        w[0] = 1.0 / r[0][0];
        for (int p = 1; p < k; ++p) {
            double s = 0.0;
            for (int t = 0; t < p; ++t) {
                double m = r[p][t] * w[t];
                s = s - m;
            }
            w[p] = s / r[p][p];
        }
        for (int p = k - 1; p >= 0; --p) {
            double s = w[p];
            for (int t = p + 1; t < k; ++t) {
                double m = r[t][p] * y[t];
                s = s - m;
            }
            y[p] = s / r[p][p];
        }
        if (!(y[0] > 0.0)) return 7;
        double g = sqrt(y[0]);
        for (int p = 0; p < k; ++p) {
            double v = y[p] / g;
            u_val[rs + p] = fp32 ? (double)(float)v : v;
        }
    }
    return 0;
}

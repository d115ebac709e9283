/* TEST INFRASTRUCTURE ONLY -- plain-C statement of the STR window search (DESIGN.md section 4.5), the
 * checker of the locate kernel (warpstr_b200/csrc/locate.cu).  Never linked into the product library.
 * Same arithmetic conventions as dp_oracle.c: float64, sums left to right, strict '<'.
 * Pinned by tests/test_locate_oracle.py against an enumeration of every path on tiny inputs. */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>

/* STR window search in a whole read (DESIGN.md section 4.5): the caller's DP rules (no mask, so back = m
 * on every row; no end band) with the cost c_t(j) = |x_t - v_j| - lam, a free start in state 0 on every
 * row and a free end.  Candidates of L[i][j], first strict minimum wins:
 *   stay        L[i-1][j] + c_i(j)
 *   incoming p  ((L[i-m][p] + c_{i-m+1}(p)) + ... + c_{i-1}(p)) + c_i(j), in list order
 *   start       c_i(0), state 0 only
 * Each cell carries the start row of its winner.  E = min_i L[i][endstate] (first i on ties); the
 * window is [start, i_E].  Returns 0 (found: E < 0), 1 (E >= 0) or 2 (no path: E = +inf), the
 * WSTR_LOCATE_* codes; *lo / *hi are -1 when there is no path.  Keeps the last m + 1 rows only and
 * sums every skip candidate from its definition (not from running sums, as the kernel does). */
int wso_locate(const double *x, int64_t N, const double *v, const int32_t *in_ptr, const int32_t *in_idx,
               int S, int endstate, int m, double lam, int64_t *lo, int64_t *hi, double *score)
{
    const double inf = INFINITY;
    const int R = m + 1;                     /* rows kept: i-m .. i */
    double *L = (double *)malloc(sizeof(double) * (size_t)R * S);
    int64_t *G = (int64_t *)malloc(sizeof(int64_t) * (size_t)R * S);
    if (!L || !G) { free(L); free(G); return 3; }
    double E = inf;
    int64_t e_lo = -1, e_hi = -1;
    for (int64_t i = 0; i < N; ++i) {
        double *row = L + (size_t)(i % R) * S;
        int64_t *tag = G + (size_t)(i % R) * S;
        const double *up = i >= 1 ? L + (size_t)((i - 1) % R) * S : NULL;
        const int64_t *up_tag = i >= 1 ? G + (size_t)((i - 1) % R) * S : NULL;
        const double *far = i >= m ? L + (size_t)((i - m) % R) * S : NULL;
        const int64_t *far_tag = i >= m ? G + (size_t)((i - m) % R) * S : NULL;
        for (int j = 0; j < S; ++j) {
            const double cj = fabs(x[i] - v[j]) - lam;
            double best = inf;
            int64_t bt = -1;
            if (up) {
                double c = up[j] + cj;
                if (c < best) { best = c; bt = up_tag[j]; }
            }
            if (far) {
                for (int e = in_ptr[j]; e < in_ptr[j + 1]; ++e) {
                    int p = in_idx[e];
                    double c = far[p];
                    for (int64_t t = i - m + 1; t < i; ++t) c += fabs(x[t] - v[p]) - lam;
                    c += cj;
                    if (c < best) { best = c; bt = far_tag[p]; }
                }
            }
            if (j == 0 && cj < best) { best = cj; bt = i; }
            row[j] = best;
            tag[j] = bt;
        }
        if (row[endstate] < E) { E = row[endstate]; e_lo = tag[endstate]; e_hi = i; }
    }
    free(L);
    free(G);
    *score = E;
    *lo = e_lo;
    *hi = e_hi;
    if (E == inf) return 2;
    return E < 0.0 ? 0 : 1;
}

/*
 * chain_oracle.c -- CPU restatement (plain C, IEEE fp64) of the reference's Fabrik.calculate (fabrik.py:19-67) for
 * chains of J points, the checker of csrc/fabrik_chain.cu (tests/test_fabrik_chain.py builds and loads it).
 *
 *   while (se > tol or ge > tol) and max_iter > k:
 *       b = T; for j = J-2 .. 0: b = PB(b, P[j], d[j]); P[j] = b         backward, d[J-2..0]
 *       se = |P[0] - S|; P[0] = S
 *       for j = 1 .. J-1: P[j] = PB(P[j-1], (j == J-1 ? T : P[j]), d[j])  forward, d[1..J-1]
 *       ge = |P[J-1] - T|; k += 1
 *   PB(a, b, L) = a + (L / |b - a|) * (b - a) per axis (point.py:32-45)
 *
 * Operation order follows the Python source.  Build with -ffp-contract=off and without -ffast-math.  A zero-length
 * segment is not an early exit here (ZeroDivisionError upstream): the division by 0 propagates as on the GPU, the
 * chain becomes non-finite, the loop ends, and the row is reported in *first_zero.
 */
#include <math.h>
#include <stdint.h>
#include <string.h>

static double dist(const double a[3], const double b[3])
{
    double dx = a[0] - b[0], dy = a[1] - b[1], dz = a[2] - b[2];
    return sqrt(dx * dx + dy * dy + dz * dz);
}

static void point_between(const double s[3], const double e[3], double distance, double out[3])
{
    double t = distance / dist(s, e), o[3];
    for (int i = 0; i < 3; ++i)
        o[i] = s[i] + t * (e[i] - s[i]);
    memcpy(out, o, sizeof o);
}

/* init: n_init x J x 3 (n_init is 1 or n), goals: n x 3, out: n x J x 3, iters: n.  Returns the number of rows that
 * stopped on max_iter with an error above tol after at least one pass; *first_zero = lowest row whose chain is not
 * finite although its goal is, or -1. */
int64_t ico_fabrik_chain(int J, const double *d, double tol, int max_iter, const double *init, int64_t n_init,
                         const double *goals, int64_t n, double *out, int32_t *iters, int64_t *first_zero)
{
    int64_t capped = 0;
    *first_zero = -1;
    for (int64_t r = 0; r < n; ++r) {
        double (*P)[3] = (double (*)[3])(out + (int64_t)3 * J * r);
        memcpy(P, init + (n_init == 1 ? 0 : (int64_t)3 * J * r), sizeof(double) * 3 * J);
        const double *T = goals + 3 * r;
        double S[3], b[3];
        memcpy(S, P[0], sizeof S);
        double se = 1.0, ge = 1.0;
        int k = 0;
        while ((se > tol || ge > tol) && max_iter > k) {
            memcpy(b, T, sizeof b);
            for (int j = J - 2; j >= 0; --j) {
                point_between(b, P[j], d[j], P[j]);
                memcpy(b, P[j], sizeof b);
            }
            se = dist(P[0], S);
            memcpy(P[0], S, sizeof S);
            for (int j = 1; j < J; ++j)
                point_between(P[j - 1], j == J - 1 ? T : P[j], d[j], P[j]);
            ge = dist(P[J - 1], T);
            ++k;
        }
        iters[r] = k;
        capped += (se > tol || ge > tol) && k > 0;
        int bad = 0;
        for (int j = 0; j < 3 * J; ++j)
            bad |= !isfinite(P[0][j]);
        if (bad && isfinite(T[0]) && isfinite(T[1]) && isfinite(T[2]) && *first_zero < 0)
            *first_zero = r;
    }
    return capped;
}

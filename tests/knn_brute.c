/*
 * knn_brute.c -- TEST INFRASTRUCTURE ONLY: the fp64 brute force the kNN tests compare pc_knn_batch with
 * (compiled on first use by tests/knn_brute.py with gcc -O2 -ffp-contract=off -fopenmp).
 * d2 is the reference's expression, accumulated from 0.0 in the order x, y, z (kdtree.c:379-382), un-fused.
 */
#include <stdint.h>
#include <math.h>
#ifdef _OPENMP
#include <omp.h>
#endif

static inline double sq(double v) { return v * v; }

/* Per query the k smallest (d2, original index); max_range >= 0 keeps only points with d2 <= max_range * max_range (the
 * inclusive range test).  Rows with fewer than k points are padded with idx -1, d2 +inf.  idx / d2: m * k entries,
 * row-major. */
int knn_brute_batch(const float *xyz, int64_t n, int64_t pstride,
                    const float *q, int64_t m, int64_t qstride, int k, double max_range,
                    int64_t *idx, double *d2, int nthreads)
{
    if (k < 1) return -1;
#ifdef _OPENMP
    if (nthreads <= 0) nthreads = omp_get_max_threads();
#else
    (void)nthreads;
#endif
    const int bounded = max_range >= 0.0;
    const double r2 = max_range * max_range;
#pragma omp parallel for schedule(dynamic, 16) num_threads(nthreads)
    for (int64_t j = 0; j < m; j++) {
        const float *qq = q + j * qstride;
        const double qx = qq[0], qy = qq[1], qz = qq[2];
        int64_t *ri = idx + j * k;
        double *rd = d2 + j * k;
        for (int t = 0; t < k; t++) { ri[t] = -1; rd[t] = INFINITY; }
        for (int64_t i = 0; i < n; i++) {
            const float *p = xyz + i * pstride;
            double s = 0.0;
            s += sq((double)p[0] - qx);
            s += sq((double)p[1] - qy);
            s += sq((double)p[2] - qz);
            if (bounded && !(s <= r2)) continue;
            /* i grows, so a point tied with the k-th entry never displaces it */
            if (!(s < rd[k - 1]) && !(ri[k - 1] < 0 && s <= rd[k - 1])) continue;
            int t = k - 1;
            while (t > 0 && (ri[t - 1] < 0 || rd[t - 1] > s)) { rd[t] = rd[t - 1]; ri[t] = ri[t - 1]; t--; }
            rd[t] = s; ri[t] = i;
        }
    }
    return 0;
}

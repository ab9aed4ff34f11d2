/*
 * range_sorted_brute.c -- TEST INFRASTRUCTURE ONLY: the fp64 brute force the sorted-range tests compare
 * pc_range_sorted_batch with (compiled on first use by tests/range_sorted_brute.py with gcc -O2 -ffp-contract=off -fopenmp).
 * d2 is the reference's expression, accumulated from 0.0 in the order x, y, z (kdtree.c:379-382), un-fused.
 */
#include <stdint.h>
#include <stdlib.h>
#include <math.h>
#ifdef _OPENMP
#include <omp.h>
#endif

static inline double sq(double v) { return v * v; }

typedef struct { double d2; int64_t idx; } rs_hit;

static int rs_cmp(const void *a, const void *b)
{
    const rs_hit *x = (const rs_hit *)a, *y = (const rs_hit *)b;
    if (x->d2 != y->d2) return x->d2 < y->d2 ? -1 : 1;
    return (x->idx > y->idx) - (x->idx < y->idx);
}

/* Per query every point with d2 <= range * range (inclusive; one range, or one per query when range_is_scalar == 0), sorted
 * by (d2, original index) and cut to max_nn entries (0 keeps all).  Two calls: with idx == NULL it writes the row lengths to
 * counts[m]; given offsets[m + 1] of those lengths it writes the rows to idx / d2. */
int range_sorted_brute(const float *xyz, int64_t n, int64_t pstride,
                       const float *q, int64_t m, int64_t qstride, const double *range, int range_is_scalar, int64_t max_nn,
                       int64_t *counts, const int64_t *offsets, int64_t *idx, double *d2, int nthreads)
{
    if (max_nn < 0) return -1;
#ifdef _OPENMP
    if (nthreads <= 0) nthreads = omp_get_max_threads();
#else
    (void)nthreads;
#endif
    int fail = 0;
#pragma omp parallel num_threads(nthreads) reduction(|: fail)
    {
        rs_hit *buf = NULL;
        int64_t buf_cap = 0;
#pragma omp for schedule(dynamic, 16)
        for (int64_t j = 0; j < m; j++) {
            const float *qq = q + j * qstride;
            const double qx = qq[0], qy = qq[1], qz = qq[2];
            const double r = range[range_is_scalar ? 0 : j];
            const double r2 = r * r;
            int64_t cnt = 0;
            for (int64_t i = 0; i < n; i++) {
                const float *p = xyz + i * pstride;
                double s = 0.0;
                s += sq((double)p[0] - qx);
                s += sq((double)p[1] - qy);
                s += sq((double)p[2] - qz);
                if (!(s <= r2)) continue;
                if (idx) {
                    if (cnt == buf_cap) {
                        buf_cap = buf_cap ? 2 * buf_cap : 1024;
                        rs_hit *nb = (rs_hit *)realloc(buf, (size_t)buf_cap * sizeof(rs_hit));
                        if (!nb) { fail = 1; break; }
                        buf = nb;
                    }
                    buf[cnt].d2 = s;
                    buf[cnt].idx = i;
                }
                cnt++;
            }
            const int64_t keep = max_nn > 0 && max_nn < cnt ? max_nn : cnt;
            if (!idx) { counts[j] = keep; continue; }
            if (fail || offsets[j + 1] - offsets[j] != keep) { fail = 1; continue; }
            qsort(buf, (size_t)cnt, sizeof(rs_hit), rs_cmp);
            for (int64_t t = 0; t < keep; t++) { idx[offsets[j] + t] = buf[t].idx; d2[offsets[j] + t] = buf[t].d2; }
        }
        free(buf);
    }
    return fail ? -1 : 0;
}

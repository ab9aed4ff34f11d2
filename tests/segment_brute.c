/*
 * segment_brute.c -- TEST INFRASTRUCTURE ONLY: the fp64 brute force the segment tests compare pc_segment_nearest_batch with
 * (compiled on first use by tests/segment_brute.py with gcc -O2 -ffp-contract=off -fopenmp).
 * d2 is the contract's expression (include/pc_index.h), operation for operation, un-fused.
 */
#include <stdint.h>
#include <math.h>
#ifdef _OPENMP
#include <omp.h>
#endif

/* the reference's point expression: s = 0; s += dx^2; s += dy^2; s += dz^2 */
static inline double point_d2(double px, double py, double pz, double qx, double qy, double qz)
{
    const double dx = px - qx, dy = py - qy, dz = pz - qz;
    double s = dx * dx;
    s = s + dy * dy;
    s = s + dz * dz;
    return s;
}

double segment_d2(const float *p, const float *a, const float *b)
{
    const double Px = p[0], Py = p[1], Pz = p[2], Ax = a[0], Ay = a[1], Az = a[2], Bx = b[0], By = b[1], Bz = b[2];
    const double Dx = Bx - Ax, Dy = By - Ay, Dz = Bz - Az;
    const double Wx = Px - Ax, Wy = Py - Ay, Wz = Pz - Az;
    const double L2 = (Dx * Dx + Dy * Dy) + Dz * Dz;
    const double s = (Wx * Dx + Wy * Dy) + Wz * Dz;
    if (s <= 0.0 || L2 == 0.0) return point_d2(Px, Py, Pz, Ax, Ay, Az);
    if (s >= L2) return point_d2(Px, Py, Pz, Bx, By, Bz);
    const double t = s / L2;
    const double Ex = Wx - t * Dx, Ey = Wy - t * Dy, Ez = Wz - t * Dz;
    return (Ex * Ex + Ey * Ey) + Ez * Ez;
}

/* Per segment j (a + j * sstride, b + j * sstride) the smallest (d2, original index); max_range >= 0 keeps only points with
 * d2 <= max_range * max_range.  No point: idx -1, d2 +inf.  A non-finite endpoint coordinate: idx -1, d2 NaN. */
int segment_brute_batch(const float *xyz, int64_t n, int64_t pstride, const float *a, const float *b, int64_t m, int64_t sstride,
                        double max_range, int64_t *idx, double *d2, int nthreads)
{
#ifdef _OPENMP
    if (nthreads <= 0) nthreads = omp_get_max_threads();
#else
    (void)nthreads;
#endif
    const int bounded = max_range >= 0.0;
    const double r2 = max_range * max_range;
#pragma omp parallel for schedule(dynamic, 16) num_threads(nthreads)
    for (int64_t j = 0; j < m; j++) {
        const float *aa = a + j * sstride, *bb = b + j * sstride;
        int finite = 1;
        for (int c = 0; c < 3; c++) finite &= isfinite(aa[c]) && isfinite(bb[c]);
        idx[j] = -1;
        d2[j] = finite ? INFINITY : NAN;
        if (!finite) continue;
        for (int64_t i = 0; i < n; i++) {
            const double s = segment_d2(xyz + i * pstride, aa, bb);
            if (bounded && !(s <= r2)) continue;
            if (s < d2[j]) { d2[j] = s; idx[j] = i; }       /* i grows: a tie keeps the lower index */
        }
    }
    return 0;
}

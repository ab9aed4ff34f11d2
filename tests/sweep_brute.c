/*
 * sweep_brute.c -- TEST INFRASTRUCTURE ONLY: the fp64 brute force the sphere-sweep tests compare pc_sphere_sweep_batch with
 * (compiled on first use by tests/sweep_brute.py with gcc -O2 -ffp-contract=off -fopenmp).
 * t(p) is the contract's expression (include/pc_index.h), operation for operation, un-fused; sqrt and / are IEEE.
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

/* t(p) in [0, 1], or +inf where p makes no contact */
double sweep_t(const float *p, const float *a, const float *b, double r2)
{
    const double Px = p[0], Py = p[1], Pz = p[2], Ax = a[0], Ay = a[1], Az = a[2], Bx = b[0], By = b[1], Bz = b[2];
    const double c0 = point_d2(Px, Py, Pz, Ax, Ay, Az);
    if (c0 <= r2) return 0.0;
    const double Dx = Bx - Ax, Dy = By - Ay, Dz = Bz - Az;
    const double Wx = Px - Ax, Wy = Py - Ay, Wz = Pz - Az;
    const double L2 = (Dx * Dx + Dy * Dy) + Dz * Dz;
    const double s = (Wx * Dx + Wy * Dy) + Wz * Dz;
    if (L2 != 0.0 && s > 0.0) {
        const double h = c0 - r2;
        const double disc = s * s - L2 * h;
        if (disc >= 0.0) {
            const double t = h / (s + sqrt(disc));
            if (t <= 1.0) return t;
        }
    }
    return point_d2(Px, Py, Pz, Bx, By, Bz) <= r2 ? 1.0 : INFINITY;
}

/* Per segment j (a + j * sstride, b + j * sstride) the smallest (t, original index) for a sphere of radius `radius`
 * (r2 = radius * radius).  No contact: idx -1, t +inf.  A non-finite endpoint coordinate: idx -1, t NaN. */
int sweep_brute_batch(const float *xyz, int64_t n, int64_t pstride, const float *a, const float *b, int64_t m, int64_t sstride,
                      double radius, int64_t *idx, double *t, int nthreads)
{
#ifdef _OPENMP
    if (nthreads <= 0) nthreads = omp_get_max_threads();
#else
    (void)nthreads;
#endif
    const double r2 = radius * radius;
#pragma omp parallel for schedule(dynamic, 16) num_threads(nthreads)
    for (int64_t j = 0; j < m; j++) {
        const float *aa = a + j * sstride, *bb = b + j * sstride;
        int finite = 1;
        for (int c = 0; c < 3; c++) finite &= isfinite(aa[c]) && isfinite(bb[c]);
        idx[j] = -1;
        t[j] = finite ? INFINITY : NAN;
        if (!finite) continue;
        for (int64_t i = 0; i < n; i++) {
            const double e = sweep_t(xyz + i * pstride, aa, bb, r2);
            if (e < t[j]) { t[j] = e; idx[j] = i; }         /* i grows: a tie keeps the lower index */
        }
    }
    return 0;
}

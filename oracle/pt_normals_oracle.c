/*
 * pt_normals_oracle.c -- CPU statement of the normal estimation (DESIGN.md section 8, "Normal
 * estimation"), which csrc/pt_normals.cu must equal bit for bit.
 *
 * TEST INFRASTRUCTURE ONLY, like the rest of oracle/.  Built with -ffp-contract=off (no FMA), fp64
 * throughout, every operation rounded on its own in the order written here; no transcendental
 * function other than sqrt.  The neighbour lists come from the caller (pto.knn_bruteforce or
 * pto.KdTree: ascending (d2, id), padded with -1).
 */
#include <math.h>
#include <stdint.h>
#include <string.h>

#define NORMALS_MAX_SWEEPS 50

typedef struct { double x, y, z; } d3;

static double dot3(d3 a, d3 b) { return (a.x * b.x + a.y * b.y) + a.z * b.z; }
static int usable3(d3 a) { return isfinite(a.x) && isfinite(a.y) && isfinite(a.z) && dot3(a, a) > 0.0; }

/* Numerical Recipes' ROTATE */
static void rotate(double *gr, double *hr, double s, double tau)
{
    const double g = *gr, h = *hr;
    *gr = g - s * (h + g * tau);
    *hr = h + s * (g - h * tau);
}

/* Cyclic Jacobi (Numerical Recipes' jacobi) on the symmetric 3 x 3 with upper triangle
 * c = (c00, c01, c02, c11, c12, c22): eigenvalues d, eigenvectors in the columns of v. */
static void jacobi3(const double c[6], double d[3], double v[3][3])
{
    double a[3][3] = {{c[0], c[1], c[2]}, {0.0, c[3], c[4]}, {0.0, 0.0, c[5]}};
    double b[3] = {c[0], c[3], c[5]}, z[3] = {0.0, 0.0, 0.0};
    static const int PQ[3][2] = {{0, 1}, {0, 2}, {1, 2}};
    for (int i = 0; i < 3; ++i) {
        d[i] = b[i];
        for (int j = 0; j < 3; ++j) v[i][j] = i == j ? 1.0 : 0.0;
    }
    for (int sweep = 1; sweep <= NORMALS_MAX_SWEEPS; ++sweep) {
        const double sm = (fabs(a[0][1]) + fabs(a[0][2])) + fabs(a[1][2]);
        if (sm == 0.0) break;
        const double tresh = sweep < 4 ? (0.2 * sm) / 9.0 : 0.0;
        for (int e = 0; e < 3; ++e) {
            const int p = PQ[e][0], q = PQ[e][1];
            const double apq = a[p][q];
            const double g = 100.0 * fabs(apq);
            if (sweep > 4 && fabs(d[p]) + g == fabs(d[p]) && fabs(d[q]) + g == fabs(d[q])) {
                a[p][q] = 0.0;
                continue;
            }
            if (!(fabs(apq) > tresh)) continue;
            double h = d[q] - d[p], t;
            if (fabs(h) + g == fabs(h)) {
                t = apq / h;
            } else {
                const double theta = (0.5 * h) / apq;
                t = 1.0 / (fabs(theta) + sqrt(1.0 + theta * theta));
                if (theta < 0.0) t = -t;
            }
            const double cc = 1.0 / sqrt(1.0 + t * t);
            const double s = t * cc;
            const double tau = s / (1.0 + cc);
            h = t * apq;
            z[p] -= h; z[q] += h;
            d[p] -= h; d[q] += h;
            a[p][q] = 0.0;
            /* the other two off-diagonal elements of the upper triangle */
            if (p == 0 && q == 1) rotate(&a[0][2], &a[1][2], s, tau);
            if (p == 0 && q == 2) rotate(&a[0][1], &a[1][2], s, tau);
            if (p == 1 && q == 2) rotate(&a[0][1], &a[0][2], s, tau);
            for (int j = 0; j < 3; ++j) rotate(&v[j][p], &v[j][q], s, tau);
        }
        for (int i = 0; i < 3; ++i) {
            b[i] += z[i];
            d[i] = b[i];
            z[i] = 0.0;
        }
    }
}

/* Row r: point rows[r] (r when rows is NULL) with neighbour list idx[r*k ...].  xyz: n x 3,
 * nrm: n x 3 fp32 input normals (NULL: none), view: 3 doubles or NULL.  Outputs per row: normal
 * (3 floats, 0 without an estimate), variation (quiet NaN 0x7fc00000 without) and, when fp64_out is
 * not NULL, the same before the rounding to fp32 (4 doubles: n xyz, variation).  Returns the number
 * of rows with an estimate, -1 on bad arguments. */
int64_t pto_estimate_normals(const double *xyz, const float *nrm, int64_t n, const int32_t *rows, int64_t m,
                             const int32_t *idx, int k, const double *view, float *normal_out, float *variation_out,
                             double *fp64_out)
{
    if ((!xyz && n) || (!idx && m) || !normal_out || !variation_out || k < 1) return -1;
    const uint32_t nan_bits = 0x7fc00000u;
    float qnan;
    memcpy(&qnan, &nan_bits, sizeof qnan);
    int64_t estimated = 0;
#pragma omp parallel for schedule(dynamic, 1024) reduction(+ : estimated)
    for (int64_t r = 0; r < m; ++r) {
        const int64_t i = rows ? rows[r] : r;
        const int32_t *list = idx + r * (int64_t)k;
        int cnt = 0;
        while (cnt < k && list[cnt] >= 0 && list[cnt] < n) ++cnt;
        d3 sum = {0.0, 0.0, 0.0};
        for (int j = 0; j < cnt; ++j) {
            const double *p = xyz + 3 * (int64_t)list[j];
            sum.x += p[0]; sum.y += p[1]; sum.z += p[2];
        }
        const d3 mu = {sum.x / (double)cnt, sum.y / (double)cnt, sum.z / (double)cnt};
        double c[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
        for (int j = 0; j < cnt; ++j) {
            const double *p = xyz + 3 * (int64_t)list[j];
            const double ex = p[0] - mu.x, ey = p[1] - mu.y, ez = p[2] - mu.z;
            c[0] += ex * ex; c[1] += ex * ey; c[2] += ex * ez;
            c[3] += ey * ey; c[4] += ey * ez; c[5] += ez * ez;
        }
        const double trace = (c[0] + c[3]) + c[5];
        int est = cnt >= 3 && trace > 0.0 && trace < INFINITY;
        d3 nv = {0.0, 0.0, 0.0};
        double lam0 = 0.0;
        if (est) {
            double d[3], v[3][3];
            jacobi3(c, d, v);
            int i0 = 0;
            if (d[1] < d[i0]) i0 = 1;
            if (d[2] < d[i0]) i0 = 2;
            lam0 = d[i0];
            const d3 col = {v[0][i0], v[1][i0], v[2][i0]};
            const double l = sqrt(dot3(col, col));
            nv = (d3){col.x / l, col.y / l, col.z / l};
            est = usable3(nv);
        }
        if (est) {
            int flip;
            const d3 mi = nrm ? (d3){(double)nrm[3 * i], (double)nrm[3 * i + 1], (double)nrm[3 * i + 2]} : (d3){0.0, 0.0, 0.0};
            if (nrm && usable3(mi)) {
                flip = dot3(nv, mi) < 0.0;
            } else if (view) {
                const double *p = xyz + 3 * i;
                const d3 w = {view[0] - p[0], view[1] - p[1], view[2] - p[2]};
                flip = dot3(nv, w) < 0.0;
            } else {
                const double ax = fabs(nv.x), ay = fabs(nv.y), az = fabs(nv.z);
                flip = (ax >= ay && ax >= az) ? nv.x < 0.0 : (ay >= az ? nv.y < 0.0 : nv.z < 0.0);
            }
            if (flip) nv = (d3){-nv.x, -nv.y, -nv.z};
            ++estimated;
        }
        normal_out[3 * r] = (float)nv.x;
        normal_out[3 * r + 1] = (float)nv.y;
        normal_out[3 * r + 2] = (float)nv.z;
        const double var = est ? (lam0 > 0.0 ? lam0 : 0.0) / trace : (double)qnan;
        variation_out[r] = (float)var;
        if (fp64_out) {
            double *o = fp64_out + 4 * r;
            o[0] = nv.x; o[1] = nv.y; o[2] = nv.z; o[3] = var;
        }
    }
    return estimated;
}

/*
 * pt_bake_oracle.c -- CPU statement of the per-texel bake (DESIGN.md section 8, "Per-texel bake").
 * TEST INFRASTRUCTURE ONLY, like the rest of oracle/.  The reference has no per-texel path; this
 * file states the project's own frozen definition, which csrc/pt_texture.cu must equal bit for bit
 * (tests/test_bake.py).  Built on its own into libpt_bake_oracle.so by oracle/pto_bake.py, which
 * takes the neighbour lists, the blend and the padding from libpt_oracle.so (pto.KdTree,
 * pto.blend, pto.texture_pad).
 *
 *   Texel (col, row) of a res x res image, row 0 on top, samples p = (col + 0.5, res - row - 0.5)
 *   in UV * res units.  Face f covers it iff the barycentrics of p in (U * res, V * res) are all
 *   >= 0 (inv = 1 / area2, bc2 = 1 - bc0 - bc1, as tri_coords of pt_texture_oracle.c); a degenerate
 *   UV triangle gives NaN and covers nothing, faces with an out-of-range vertex index are skipped.
 *   Faces are visited in index order and later ones overwrite: the highest covering face wins.
 *   Sample position x = (bc0 * X0 + bc1 * X1) + bc2 * X2 per axis, fp64, no FMA
 *   (-ffp-contract=off, the flags of oracle/Makefile).
 */
#include "pt_oracle.h"

#include <math.h>
#include <stdlib.h>

/* texel_out[res*res] (uint32 ids row * res + col, ascending), xyz_out[res*res*3]; returns the
 * number of covered texels, or -1 when out of memory */
int64_t pto_bake_texels(const pto_point *v, int64_t nv, const int32_t *faces, int64_t nf, int res,
                        uint32_t *texel_out, double *xyz_out);
/* the normal-map byte of one fp32 component */
int pto_bake_encode(float n);
/* samples -> the three unpadded maps (res*res each, zeroed here; any may be NULL) */
int pto_bake_compose(const uint32_t *texels, int64_t count, const uint8_t *rgba, const float *normal,
                     int res, uint8_t *bgra, uint8_t *normal_bgra, float *normal_out);

typedef struct { double a, b; } bv2;

static double bake_area2(bv2 p, bv2 q, bv2 r)
{
    return (q.a - p.a) * (r.b - p.b) - (q.b - p.b) * (r.a - p.a);
}

static void bake_coords(const bv2 t[3], bv2 x, double bc[3])
{
    const double inv = 1.0 / bake_area2(t[0], t[1], t[2]);
    bc[0] = bake_area2(t[1], t[2], x) * inv;
    bc[1] = bake_area2(t[2], t[0], x) * inv;
    bc[2] = 1.0 - bc[0] - bc[1];
}

static int face_uv(const pto_point *v, int64_t nv, const int32_t *face, int res, bv2 t[3])
{
    for (int j = 0; j < 3; ++j) {
        if (face[j] < 0 || face[j] >= nv) return 0;
        t[j].a = v[face[j]].U * res;
        t[j].b = v[face[j]].V * res;
    }
    return 1;
}

static bv2 texel_point(int res, int col, int row)
{
    const bv2 p = {(double)col + 0.5, (double)(res - row) - 0.5};
    return p;
}

/* texel_out[res*res] (uint32 ids row * res + col, ascending), xyz_out[res*res*3].  Returns the
 * number of covered texels, or -1 when out of memory. */
int64_t pto_bake_texels(const pto_point *v, int64_t nv, const int32_t *faces, int64_t nf, int res,
                        uint32_t *texel_out, double *xyz_out)
{
    const size_t n_pix = (size_t)res * res;
    int64_t *owner = (int64_t *)malloc(sizeof(int64_t) * n_pix);
    if (!owner) return -1;
    for (size_t i = 0; i < n_pix; ++i) owner[i] = -1;
    for (int64_t f = 0; f < nf; ++f) {
        bv2 t[3];
        if (!face_uv(v, nv, faces + 3 * f, res, t)) continue;
        /* every texel whose centre is within 2 texels of the triangle's box: a superset of the
         * covered ones */
        const double xmin = fmin(t[0].a, fmin(t[1].a, t[2].a)), xmax = fmax(t[0].a, fmax(t[1].a, t[2].a));
        const double ymin = fmin(t[0].b, fmin(t[1].b, t[2].b)), ymax = fmax(t[0].b, fmax(t[1].b, t[2].b));
        int nan_uv = 0;
        for (int j = 0; j < 3; ++j) nan_uv |= isnan(t[j].a) || isnan(t[j].b);
        if (nan_uv) continue;                      /* every barycentric is NaN */
        const double c0 = fmax(floor(xmin) - 2.0, 0.0), c1 = fmin(ceil(xmax) + 2.0, res - 1.0);
        const double r0 = fmax(floor(res - ymax) - 2.0, 0.0), r1 = fmin(ceil(res - ymin) + 2.0, res - 1.0);
        for (int row = (int)r0; row <= (int)r1 && r0 <= r1; ++row)
            for (int col = (int)c0; col <= (int)c1 && c0 <= c1; ++col) {
                double bc[3];
                bake_coords(t, texel_point(res, col, row), bc);
                if (bc[0] >= 0 && bc[1] >= 0 && bc[2] >= 0) owner[(size_t)row * res + col] = f;
            }
    }
    int64_t count = 0;
    for (size_t i = 0; i < n_pix; ++i) {
        if (owner[i] < 0) continue;
        const int32_t *face = faces + 3 * owner[i];
        bv2 t[3];
        face_uv(v, nv, face, res, t);
        double bc[3];
        bake_coords(t, texel_point(res, (int)(i % res), (int)(i / res)), bc);
        for (int a = 0; a < 3; ++a)
            xyz_out[3 * count + a] = (bc[0] * v[face[0]].ver[a] + bc[1] * v[face[1]].ver[a]) + bc[2] * v[face[2]].ver[a];
        texel_out[count++] = (uint32_t)i;
    }
    free(owner);
    return count;
}

/* e(n) = clamp(floor((n + 1) * 127.5 + 0.5), 0, 255), fp64 from the fp32 component */
int pto_bake_encode(float n)
{
    const double e = floor(((double)n + 1.0) * 127.5 + 0.5);
    return (int)fmin(fmax(e, 0.0), 255.0);
}

/* Samples -> the three unpadded maps (each res*res, zeroed here; any may be NULL).  A sample
 * whose neighbour list was empty (rgba alpha 0, pto_blend) stays 0 everywhere. */
int pto_bake_compose(const uint32_t *texels, int64_t count, const uint8_t *rgba, const float *normal,
                     int res, uint8_t *bgra, uint8_t *normal_bgra, float *normal_out)
{
    const size_t n_pix = (size_t)res * res;
    for (size_t i = 0; i < n_pix; ++i) {
        for (int c = 0; c < 4; ++c) {
            if (bgra) bgra[4 * i + c] = 0;
            if (normal_bgra) normal_bgra[4 * i + c] = 0;
        }
        if (normal_out) normal_out[3 * i] = normal_out[3 * i + 1] = normal_out[3 * i + 2] = 0.0f;
    }
    for (int64_t s = 0; s < count; ++s) {
        if (texels[s] >= n_pix) return 1;
        if (rgba[4 * s + 3] == 0) continue;
        const size_t t = texels[s];
        const float *n = normal + 3 * s;
        if (bgra) {
            bgra[4 * t] = rgba[4 * s + 2]; bgra[4 * t + 1] = rgba[4 * s + 1];
            bgra[4 * t + 2] = rgba[4 * s]; bgra[4 * t + 3] = 255;
        }
        if (normal_bgra) {
            normal_bgra[4 * t] = (uint8_t)pto_bake_encode(n[2]);
            normal_bgra[4 * t + 1] = (uint8_t)pto_bake_encode(n[1]);
            normal_bgra[4 * t + 2] = (uint8_t)pto_bake_encode(n[0]);
            normal_bgra[4 * t + 3] = 255;
        }
        if (normal_out) for (int a = 0; a < 3; ++a) normal_out[3 * t + a] = n[a];
    }
    return 0;
}

/*
 * pt_bake_oracle.c -- CPU statement of the per-texel bake (DESIGN.md section 8: "Per-texel bake",
 * "Tangent-space bake", "Height bake").  TEST INFRASTRUCTURE ONLY, like the rest of oracle/.  The
 * reference has no per-texel path; this file states the project's own frozen definitions, which
 * csrc/pt_texture.cu must equal bit for bit (tests/test_bake.py, tests/test_bake_tangent.py,
 * tests/test_bake_height.py).  Built into libpt_oracle.so with the rest of oracle/; its binding
 * oracle/pto_bake.py takes the neighbour lists, the blend and the 8-bit padding from pto.KdTree,
 * pto.blend and pto.texture_pad.  Fp64 throughout, no FMA (-ffp-contract=off, oracle/Makefile),
 * every operation in the order the definition states.
 *
 *   texels      Texel (col, row) of a res x res image, row 0 on top, samples p = (col + 0.5,
 *               res - row - 0.5) in UV * res units.  Face f covers it iff the barycentrics of p in
 *               (U * res, V * res) are all >= 0 (inv = 1 / area2, bc2 = 1 - bc0 - bc1, as tri_coords
 *               of pt_texture_oracle.c); a degenerate UV triangle gives NaN and covers nothing, faces
 *               with an out-of-range vertex index are skipped.  Faces are visited in index order and
 *               later ones overwrite: the highest covering face (the owner) wins.  Sample position
 *               x = (bc0 * X0 + bc1 * X1) + bc2 * X2 per axis.
 *   compose     the object-space maps of the blended colour and normal
 *   frames      per face T_f, B_f, G_f; per vertex the sums in face order, N, T, w
 *   tangent     per covered texel the mixed frame, made orthonormal, and the blended normal in it
 *   height      per covered texel h = (float)((sum_j w_j (p_j - x).N) / W), the blend's weights
 *   encode/pad  the height code range, the 16-bit codes and their padding
 */
#include "pt_oracle.h"

#include <math.h>
#include <stdlib.h>
#include <string.h>

/* texel_out[res*res] (uint32 ids row * res + col, ascending), xyz_out[res*res*3], face_out[res*res]
 * (the owner face of each sample; may be NULL).  Returns the number of covered texels, or -1 when
 * out of memory. */
int64_t pto_bake_texels(const pto_point *v, int64_t nv, const int32_t *faces, int64_t nf, int res,
                        uint32_t *texel_out, double *xyz_out, int32_t *face_out);
/* the normal-map byte of one fp32 component */
int pto_bake_encode(float n);
/* samples -> the three unpadded maps (res*res each, zeroed here; any may be NULL) */
int pto_bake_compose(const uint32_t *texels, int64_t count, const uint8_t *rgba, const float *normal,
                     int res, uint8_t *bgra, uint8_t *normal_bgra, float *normal_out);
/* frames_out[nv*8] = N xyz, T xyz, w, 0 (zero without a frame); tangents_out[nv*4] = (T, w) in
 * fp32 (may be NULL).  Returns -1 when out of memory. */
int pto_bake_frames(const pto_point *v, int64_t nv, const int32_t *faces, int64_t nf, double *frames_out,
                    float *tangents_out);
/* samples -> the two unpadded tangent maps (res*res each, zeroed here; either may be NULL).
 * Returns 1 on a malformed sample. */
int pto_bake_compose_tangent(const pto_point *v, int64_t nv, const double *frames, const int32_t *faces,
                             int64_t nf, const uint32_t *texels, const int32_t *sample_faces, int64_t count,
                             const uint8_t *rgba, const float *normal, int res, uint8_t *tangent_bgra,
                             float *tangent_normal);
/* height[res*res] (written here): h per covered texel with a value, NaN (0x7fc00000) elsewhere.
 * idx / d2: count x k, ascending; a list ends at its first id outside 0..n-1.  Returns 1 on a
 * malformed sample. */
int pto_bake_height(const pto_point *v, int64_t nv, const double *frames, const int32_t *faces, int64_t nf,
                    const uint32_t *texels, const int32_t *sample_faces, const double *xyz, int64_t count,
                    const pto_point *pts, int64_t n, const int32_t *idx, const double *d2, int k, int res,
                    float *height);
/* codes[res*res] without padding (0 without a value) and the range used; returns the number of
 * texels with a value */
int64_t pto_bake_height_encode(const float *height, int64_t n_pix, const double *range_in, uint16_t *codes,
                               double *range_used);
/* padded[res*res] from the unpadded codes; returns -1 when out of memory */
int pto_bake_height_pad(const float *height, const uint16_t *codes, int res, uint16_t *padded);

/* ---- texels ------------------------------------------------------------------------------------ */
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

/* the UV triangle in UV * res units; 0 for a face with an out-of-range vertex index */
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

int64_t pto_bake_texels(const pto_point *v, int64_t nv, const int32_t *faces, int64_t nf, int res,
                        uint32_t *texel_out, double *xyz_out, int32_t *face_out)
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
        bv2 t[3] = {{0, 0}, {0, 0}, {0, 0}};     /* an owner face has valid corners */
        face_uv(v, nv, face, res, t);
        double bc[3];
        bake_coords(t, texel_point(res, (int)(i % res), (int)(i / res)), bc);
        for (int a = 0; a < 3; ++a)
            xyz_out[3 * count + a] = (bc[0] * v[face[0]].ver[a] + bc[1] * v[face[1]].ver[a]) + bc[2] * v[face[2]].ver[a];
        if (face_out) face_out[count] = (int32_t)owner[i];
        texel_out[count++] = (uint32_t)i;
    }
    free(owner);
    return count;
}

/* ---- object-space maps ------------------------------------------------------------------------- */
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

/* ---- tangent-space bake ------------------------------------------------------------------------ */
typedef struct { double x, y, z; } d3;

static d3 d3_of(const double *p) { const d3 r = {p[0], p[1], p[2]}; return r; }
static d3 add3(d3 a, d3 b) { const d3 r = {a.x + b.x, a.y + b.y, a.z + b.z}; return r; }
static d3 sub3(d3 a, d3 b) { const d3 r = {a.x - b.x, a.y - b.y, a.z - b.z}; return r; }
static d3 scale3(double s, d3 a) { const d3 r = {s * a.x, s * a.y, s * a.z}; return r; }
static double dot3(d3 a, d3 b) { return (a.x * b.x + a.y * b.y) + a.z * b.z; }
static d3 cross3(d3 a, d3 b)
{
    const d3 r = {a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x};
    return r;
}
static int finite3(d3 a) { return isfinite(a.x) && isfinite(a.y) && isfinite(a.z); }
static int usable3(d3 a) { return finite3(a) && dot3(a, a) > 0.0; }
static d3 normalise3(d3 a)
{
    const double l = sqrt(dot3(a, a));
    const d3 r = {a.x / l, a.y / l, a.z / l};
    return r;
}
static d3 mix3(const double bc[3], d3 a, d3 b, d3 c)
{
    return add3(add3(scale3(bc[0], a), scale3(bc[1], b)), scale3(bc[2], c));
}
/* t - (n.t) n normalised if usable, otherwise F(n) = e_i - n_i n normalised, i = argmin |n_i|
 * (lowest i on ties) */
static d3 tangent_dir(d3 n, d3 t)
{
    const d3 r = sub3(t, scale3(dot3(n, t), n));
    if (usable3(r)) return normalise3(r);
    const double a[3] = {fabs(n.x), fabs(n.y), fabs(n.z)};
    int i = 0;
    if (a[1] < a[i]) i = 1;
    if (a[2] < a[i]) i = 2;
    const double ni = i == 0 ? n.x : (i == 1 ? n.y : n.z);
    const d3 e = {i == 0 ? 1.0 : 0.0, i == 1 ? 1.0 : 0.0, i == 2 ? 1.0 : 0.0};
    return normalise3(sub3(e, scale3(ni, n)));
}

static int face_valid(const int32_t *face, int64_t nv)
{
    for (int j = 0; j < 3; ++j)
        if (face[j] < 0 || face[j] >= nv) return 0;
    return 1;
}

/* T_f, B_f (0 when det == 0 or not finite) and G_f of a face with valid corners */
static void face_frame(const pto_point *v, const int32_t *face, d3 *T, d3 *B, d3 *G)
{
    const pto_point *a = v + face[0], *b = v + face[1], *c = v + face[2];
    const d3 xa = d3_of(a->ver);
    const d3 e1 = sub3(d3_of(b->ver), xa), e2 = sub3(d3_of(c->ver), xa);
    const double du1 = b->U - a->U, dv1 = b->V - a->V, du2 = c->U - a->U, dv2 = c->V - a->V;
    const double det = du1 * dv2 - du2 * dv1;
    const double r = 1.0 / det;
    *T = scale3(r, sub3(scale3(dv2, e1), scale3(dv1, e2)));
    *B = scale3(r, sub3(scale3(du1, e2), scale3(du2, e1)));
    if (det == 0.0 || !finite3(*T) || !finite3(*B)) {
        const d3 z = {0.0, 0.0, 0.0};
        *T = *B = z;
    }
    *G = cross3(e1, e2);
}

int pto_bake_frames(const pto_point *v, int64_t nv, const int32_t *faces, int64_t nf, double *frames_out,
                    float *tangents_out)
{
    d3 *acc = (d3 *)calloc(3 * (size_t)(nv ? nv : 1), sizeof(d3));   /* T, B, G per vertex, +0.0 */
    if (!acc) return -1;
    for (int64_t f = 0; f < nf; ++f) {                                 /* faces ascending, corners a, b, c */
        const int32_t *face = faces + 3 * f;
        if (!face_valid(face, nv)) continue;
        d3 T, B, G;
        face_frame(v, face, &T, &B, &G);
        for (int j = 0; j < 3; ++j) {
            d3 *s = acc + 3 * (size_t)face[j];
            s[0] = add3(s[0], T);
            s[1] = add3(s[1], B);
            s[2] = add3(s[2], G);
        }
    }
    for (int64_t i = 0; i < nv; ++i) {
        const d3 T = acc[3 * i], B = acc[3 * i + 1], G = acc[3 * i + 2];
        const d3 n = d3_of(v[i].normal);
        double *o = frames_out + 8 * i;
        for (int j = 0; j < 8; ++j) o[j] = 0.0;
        if (usable3(n) || usable3(G)) {
            const d3 N = normalise3(usable3(n) ? n : G);
            const d3 Th = tangent_dir(N, T);
            o[0] = N.x; o[1] = N.y; o[2] = N.z;
            o[3] = Th.x; o[4] = Th.y; o[5] = Th.z;
            o[6] = dot3(cross3(N, Th), B) < 0.0 ? -1.0 : 1.0;
        }
        if (tangents_out)
            for (int j = 0; j < 4; ++j) tangents_out[4 * i + j] = (float)o[3 + j];
    }
    free(acc);
    return 0;
}

/* The frame of texel tx on its owner face: the barycentrics of the texel centre, the corners'
 * frame rows and the unit mesh normal N (the mixed N rows, normalised).  -1: a corner index out of
 * range; 0: the mixed normal is not usable; 1: done. */
static int texel_frame(const pto_point *v, int64_t nv, const double *frames, const int32_t *face, int res,
                       size_t tx, double bc[3], const double *fr[3], d3 *N)
{
    bv2 t[3];
    if (!face_uv(v, nv, face, res, t)) return -1;
    bake_coords(t, texel_point(res, (int)(tx % res), (int)(tx / res)), bc);
    for (int j = 0; j < 3; ++j) fr[j] = frames + 8 * (size_t)face[j];
    const d3 n = mix3(bc, d3_of(fr[0]), d3_of(fr[1]), d3_of(fr[2]));
    if (!usable3(n)) return 0;
    *N = normalise3(n);
    return 1;
}

int pto_bake_compose_tangent(const pto_point *v, int64_t nv, const double *frames, const int32_t *faces,
                             int64_t nf, const uint32_t *texels, const int32_t *sample_faces, int64_t count,
                             const uint8_t *rgba, const float *normal, int res, uint8_t *tangent_bgra,
                             float *tangent_normal)
{
    const size_t n_pix = (size_t)res * res;
    if (tangent_bgra) for (size_t i = 0; i < 4 * n_pix; ++i) tangent_bgra[i] = 0;
    if (tangent_normal) for (size_t i = 0; i < 3 * n_pix; ++i) tangent_normal[i] = 0.0f;
    for (int64_t s = 0; s < count; ++s) {
        if (texels[s] >= n_pix || sample_faces[s] < 0 || sample_faces[s] >= nf) return 1;
        if (rgba[4 * s + 3] == 0) continue;
        const int32_t *face = faces + 3 * (int64_t)sample_faces[s];
        const size_t tx = texels[s];
        double bc[3];
        const double *fr[3];
        d3 N;
        const int got = texel_frame(v, nv, frames, face, res, tx, bc, fr, &N);
        if (got < 0) return 1;
        if (got == 0) continue;
        const d3 tm = mix3(bc, d3_of(fr[0] + 3), d3_of(fr[1] + 3), d3_of(fr[2] + 3));
        const d3 T = tangent_dir(N, tm);
        d3 Tf, Bf, Gf;
        face_frame(v, face, &Tf, &Bf, &Gf);
        const d3 x = cross3(N, T);
        const double w = dot3(x, Bf) < 0.0 ? -1.0 : 1.0;
        const d3 B = scale3(w, x);
        const d3 m = {(double)normal[3 * s], (double)normal[3 * s + 1], (double)normal[3 * s + 2]};
        const float ts[3] = {(float)dot3(m, T), (float)dot3(m, B), (float)dot3(m, N)};
        if (tangent_bgra) {
            tangent_bgra[4 * tx] = (uint8_t)pto_bake_encode(ts[2]);
            tangent_bgra[4 * tx + 1] = (uint8_t)pto_bake_encode(ts[1]);
            tangent_bgra[4 * tx + 2] = (uint8_t)pto_bake_encode(ts[0]);
            tangent_bgra[4 * tx + 3] = 255;
        }
        if (tangent_normal) for (int a = 0; a < 3; ++a) tangent_normal[3 * tx + a] = ts[a];
    }
    return 0;
}

/* ---- height bake ------------------------------------------------------------------------------- */
static float nan_value(void)
{
    const uint32_t u = 0x7fc00000u;
    float f;
    memcpy(&f, &u, sizeof f);
    return f;
}

int pto_bake_height(const pto_point *v, int64_t nv, const double *frames, const int32_t *faces, int64_t nf,
                    const uint32_t *texels, const int32_t *sample_faces, const double *xyz, int64_t count,
                    const pto_point *pts, int64_t n, const int32_t *idx, const double *d2, int k, int res,
                    float *height)
{
    const size_t n_pix = (size_t)res * res;
    for (size_t i = 0; i < n_pix; ++i) height[i] = nan_value();
    for (int64_t s = 0; s < count; ++s) {
        if (texels[s] >= n_pix || sample_faces[s] < 0 || sample_faces[s] >= nf) return 1;
        const size_t tx = texels[s];
        /* 1. the unit mesh normal */
        double bc[3];
        const double *fr[3];
        d3 N;
        const int got = texel_frame(v, nv, frames, faces + 3 * (int64_t)sample_faces[s], res, tx, bc, fr, &N);
        if (got < 0) return 1;
        if (got == 0) continue;
        /* 2. the list */
        const int32_t *qi = idx + s * (int64_t)k;
        const double *qd = d2 + s * (int64_t)k;
        int cnt = 0;
        while (cnt < k && qi[cnt] >= 0 && qi[cnt] < n) ++cnt;
        if (cnt == 0) continue;
        const d3 x = d3_of(xyz + 3 * s);
        /* 3. and 4. the blend's weights; S and W in neighbour order from +0.0 */
        int mode = qd[0] == 0.0 ? 1 : 0;
        double W = 0.0, S = 0.0;
        for (int pass = 0; pass < 2; ++pass) {
            W = 0.0;
            S = 0.0;
            for (int j = 0; j < cnt; ++j) {
                double w;
                if (mode == 0) w = 1.0 / qd[j];
                else if (mode == 1) w = qd[j] == 0.0 ? 1.0 : 0.0;
                else w = j == 0 ? 1.0 : 0.0;
                const double o = dot3(sub3(d3_of(pts[qi[j]].ver), x), N);
                W = W + w;
                S = S + w * o;
            }
            if (W > 0.0 && W < INFINITY) break;
            mode = 2;
        }
        const float h = (float)(S / W);
        height[tx] = isnan(h) ? nan_value() : h;
    }
    return 0;
}

/* E(h) = clamp(floor((h - lo) * s + 0.5), 0, 65535), s = 65535 / (hi - lo) */
static uint16_t height_code(float h, double lo, double hi)
{
    if (hi == lo) return 0;
    const double s = 65535.0 / (hi - lo);
    const double e = floor(((double)h - lo) * s + 0.5);
    return (uint16_t)fmin(fmax(e, 0.0), 65535.0);
}

/* -0 orders below +0, as a sign-magnitude comparison does */
static int below(float a, float b) { return a < b || (a == b && signbit(a) && !signbit(b)); }

int64_t pto_bake_height_encode(const float *height, int64_t n_pix, const double *range_in, uint16_t *codes,
                               double *range_used)
{
    int64_t valued = 0;
    float lo = 0.0f, hi = 0.0f;
    for (int64_t i = 0; i < n_pix; ++i) {
        const float h = height[i];
        if (isnan(h)) continue;
        if (valued == 0 || below(h, lo)) lo = h;
        if (valued == 0 || below(hi, h)) hi = h;
        ++valued;
    }
    double l = lo, u = hi;
    if (range_in && isfinite(range_in[0]) && isfinite(range_in[1]) && range_in[0] < range_in[1]) {
        l = range_in[0];
        u = range_in[1];
    }
    range_used[0] = l;
    range_used[1] = u;
    for (int64_t i = 0; i < n_pix; ++i) codes[i] = isnan(height[i]) ? 0 : height_code(height[i], l, u);
    return valued;
}

/* word = E + 1 with a value, else 0; 25-wide maxima along rows, then along columns; a texel
 * without a value takes the window's maximum minus one (0 if the window has no value) */
int pto_bake_height_pad(const float *height, const uint16_t *codes, int res, uint16_t *padded)
{
    const size_t n_pix = (size_t)res * res;
    uint32_t *word = (uint32_t *)malloc(sizeof(uint32_t) * (n_pix ? n_pix : 1));
    uint32_t *tmp = (uint32_t *)malloc(sizeof(uint32_t) * (n_pix ? n_pix : 1));
    if (!word || !tmp) {
        free(word);
        free(tmp);
        return -1;
    }
    for (size_t i = 0; i < n_pix; ++i) word[i] = isnan(height[i]) ? 0u : (uint32_t)codes[i] + 1u;
    for (int y = 0; y < res; ++y)
        for (int x = 0; x < res; ++x) {
            uint32_t m = 0;
            for (int xx = x - 12; xx <= x + 12; ++xx)
                if (xx >= 0 && xx < res && word[(size_t)y * res + xx] > m) m = word[(size_t)y * res + xx];
            tmp[(size_t)y * res + x] = m;
        }
    for (int y = 0; y < res; ++y)
        for (int x = 0; x < res; ++x) {
            uint32_t m = 0;
            for (int yy = y - 12; yy <= y + 12; ++yy)
                if (yy >= 0 && yy < res && tmp[(size_t)yy * res + x] > m) m = tmp[(size_t)yy * res + x];
            const uint32_t t = word[(size_t)y * res + x] ? word[(size_t)y * res + x] : m;
            padded[(size_t)y * res + x] = (uint16_t)(t ? t - 1u : 0u);
        }
    free(word);
    free(tmp);
    return 0;
}

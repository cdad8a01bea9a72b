/*
 * bake_tangent_oracle.c -- CPU statement of the tangent-space bake (DESIGN.md section 8,
 * "Tangent-space bake").  TEST INFRASTRUCTURE ONLY.  csrc/pt_texture.cu must equal it bit for bit
 * (tests/test_bake_tangent.py).  Built on its own by tests/bake_tangent_oracle.py with the flags of
 * oracle/Makefile (-ffp-contract=off: no FMA); it reads the 80-byte records through
 * oracle/pt_oracle.h and takes the texel list, positions, neighbour lists, blend and padding from
 * the existing oracle libraries.
 *
 *   owner faces : the texel stage of oracle/pt_bake_oracle.c restated, keeping the winning face of
 *                 every covered texel (texel centres, tx_tri_coords arithmetic, highest face wins)
 *   frames      : per face T_f, B_f, G_f; per vertex the sums in face order, N, T, w
 *   composition : per covered texel the mixed frame, made orthonormal, and the blended normal in it
 * Every operation in the order the definition states.
 */
#include "pt_oracle.h"

#include <math.h>
#include <stdlib.h>

/* texel_out[res*res] (ascending texel ids), face_out[res*res]; returns the number of covered
 * texels, or -1 when out of memory */
int64_t ptt_bake_owners(const pto_point *v, int64_t nv, const int32_t *faces, int64_t nf, int res,
                        uint32_t *texel_out, int32_t *face_out);
/* frames_out[nv*8] = N xyz, T xyz, w, 0 (zero without a frame); tangents_out[nv*4] = (T, w) in
 * fp32 (may be NULL).  Returns -1 when out of memory. */
int ptt_bake_frames(const pto_point *v, int64_t nv, const int32_t *faces, int64_t nf, double *frames_out,
                    float *tangents_out);
/* samples -> the two unpadded tangent maps (res*res each, zeroed here; either may be NULL) */
int ptt_bake_compose_tangent(const pto_point *v, int64_t nv, const double *frames, const int32_t *faces,
                             int64_t nf, const uint32_t *texels, const int32_t *sample_faces, int64_t count,
                             const uint8_t *rgba, const float *normal, int res, uint8_t *tangent_bgra,
                             float *tangent_normal);

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

/* e(n) = clamp(floor((n + 1) * 127.5 + 0.5), 0, 255), fp64 from the fp32 component */
static int encode(float n)
{
    const double e = floor(((double)n + 1.0) * 127.5 + 0.5);
    return (int)fmin(fmax(e, 0.0), 255.0);
}

int64_t ptt_bake_owners(const pto_point *v, int64_t nv, const int32_t *faces, int64_t nf, int res,
                        uint32_t *texel_out, int32_t *face_out)
{
    const size_t n_pix = (size_t)res * res;
    int64_t *owner = (int64_t *)malloc(sizeof(int64_t) * n_pix);
    if (!owner) return -1;
    for (size_t i = 0; i < n_pix; ++i) owner[i] = -1;
    for (int64_t f = 0; f < nf; ++f) {
        bv2 t[3] = {{0, 0}, {0, 0}, {0, 0}};
        if (!face_uv(v, nv, faces + 3 * f, res, t)) continue;
        int nan_uv = 0;
        for (int j = 0; j < 3; ++j) nan_uv |= isnan(t[j].a) || isnan(t[j].b);
        if (nan_uv) continue;                      /* every barycentric is NaN */
        /* every texel whose centre is within 2 texels of the triangle's box: a superset of the
         * covered ones */
        const double xmin = fmin(t[0].a, fmin(t[1].a, t[2].a)), xmax = fmax(t[0].a, fmax(t[1].a, t[2].a));
        const double ymin = fmin(t[0].b, fmin(t[1].b, t[2].b)), ymax = fmax(t[0].b, fmax(t[1].b, t[2].b));
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
        face_out[count] = (int32_t)owner[i];
        texel_out[count++] = (uint32_t)i;
    }
    free(owner);
    return count;
}

/* ---- tangent-space bake ---------------------------------------------------------------------- */
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

static int face_valid(const int32_t *face, int64_t nv)
{
    for (int j = 0; j < 3; ++j)
        if (face[j] < 0 || face[j] >= nv) return 0;
    return 1;
}

int ptt_bake_frames(const pto_point *v, int64_t nv, const int32_t *faces, int64_t nf, double *frames_out,
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

static d3 mix3(const double bc[3], d3 a, d3 b, d3 c)
{
    return add3(add3(scale3(bc[0], a), scale3(bc[1], b)), scale3(bc[2], c));
}

int ptt_bake_compose_tangent(const pto_point *v, int64_t nv, const double *frames, const int32_t *faces,
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
        bv2 t[3];
        if (!face_uv(v, nv, face, res, t)) return 1;
        const size_t tx = texels[s];
        double bc[3];
        bake_coords(t, texel_point(res, (int)(tx % res), (int)(tx / res)), bc);
        const double *fa = frames + 8 * (size_t)face[0], *fb = frames + 8 * (size_t)face[1], *fc = frames + 8 * (size_t)face[2];
        const d3 n = mix3(bc, d3_of(fa), d3_of(fb), d3_of(fc));
        if (!usable3(n)) continue;
        const d3 tm = mix3(bc, d3_of(fa + 3), d3_of(fb + 3), d3_of(fc + 3));
        const d3 N = normalise3(n);
        const d3 T = tangent_dir(N, tm);
        d3 Tf, Bf, Gf;
        face_frame(v, face, &Tf, &Bf, &Gf);
        const d3 x = cross3(N, T);
        const double w = dot3(x, Bf) < 0.0 ? -1.0 : 1.0;
        const d3 B = scale3(w, x);
        const d3 m = {(double)normal[3 * s], (double)normal[3 * s + 1], (double)normal[3 * s + 2]};
        const float ts[3] = {(float)dot3(m, T), (float)dot3(m, B), (float)dot3(m, N)};
        if (tangent_bgra) {
            tangent_bgra[4 * tx] = (uint8_t)encode(ts[2]);
            tangent_bgra[4 * tx + 1] = (uint8_t)encode(ts[1]);
            tangent_bgra[4 * tx + 2] = (uint8_t)encode(ts[0]);
            tangent_bgra[4 * tx + 3] = 255;
        }
        if (tangent_normal) for (int a = 0; a < 3; ++a) tangent_normal[3 * tx + a] = ts[a];
    }
    return 0;
}

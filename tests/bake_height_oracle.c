/*
 * bake_height_oracle.c -- CPU statement of the height bake (DESIGN.md section 8, "Height bake").
 * TEST INFRASTRUCTURE ONLY.  csrc/pt_texture.cu must equal it bit for bit
 * (tests/test_bake_height.py).  Built on its own by tests/bake_height_oracle.py with the flags of
 * oracle/Makefile (-ffp-contract=off: no FMA); it reads the 80-byte records through
 * oracle/pt_oracle.h.  Texels, positions, owner faces and vertex frames come from
 * tests/bake_tangent_oracle.c, the neighbour lists and their d2 from oracle/pto.
 *
 *   height   per covered texel: 1. the unit mesh normal N, 2. the neighbour list, 3. the blend's
 *            weights, 4. h = (float)((sum_j w_j (p_j - x).N) / W)
 *   encode   the code range and the 16-bit codes
 *   pad      the 16-bit padding, rows then columns as the device runs it
 * Every operation in the order the definition states.
 */
#include "pt_oracle.h"

#include <math.h>
#include <stdlib.h>
#include <string.h>

/* height[res*res] (written here): h per covered texel with a value, NaN (0x7fc00000) elsewhere.
 * idx / d2: count x k, ascending; a list ends at its first id outside 0..n-1.  Returns 1 on a
 * malformed sample. */
int pth_bake_height(const pto_point *v, int64_t nv, const double *frames, const int32_t *faces, int64_t nf,
                    const uint32_t *texels, const int32_t *sample_faces, const double *xyz, int64_t count,
                    const pto_point *pts, int64_t n, const int32_t *idx, const double *d2, int k, int res,
                    float *height);
/* codes[res*res] without padding (0 without a value) and the range used; returns the number of
 * texels with a value */
int64_t pth_bake_height_encode(const float *height, int64_t n_pix, const double *range_in, uint16_t *codes,
                               double *range_used);
/* padded[res*res] from the unpadded codes; returns -1 when out of memory */
int pth_bake_height_pad(const float *height, const uint16_t *codes, int res, uint16_t *padded);

typedef struct { double a, b; } bv2;
typedef struct { double x, y, z; } d3;

static float nan_value(void)
{
    const uint32_t u = 0x7fc00000u;
    float f;
    memcpy(&f, &u, sizeof f);
    return f;
}

static double area2(bv2 p, bv2 q, bv2 r)
{
    return (q.a - p.a) * (r.b - p.b) - (q.b - p.b) * (r.a - p.a);
}

static d3 d3_of(const double *p) { const d3 r = {p[0], p[1], p[2]}; return r; }
static d3 add3(d3 a, d3 b) { const d3 r = {a.x + b.x, a.y + b.y, a.z + b.z}; return r; }
static d3 sub3(d3 a, d3 b) { const d3 r = {a.x - b.x, a.y - b.y, a.z - b.z}; return r; }
static d3 scale3(double s, d3 a) { const d3 r = {s * a.x, s * a.y, s * a.z}; return r; }
static double dot3(d3 a, d3 b) { return (a.x * b.x + a.y * b.y) + a.z * b.z; }
static int usable3(d3 a) { return isfinite(a.x) && isfinite(a.y) && isfinite(a.z) && dot3(a, a) > 0.0; }

int pth_bake_height(const pto_point *v, int64_t nv, const double *frames, const int32_t *faces, int64_t nf,
                    const uint32_t *texels, const int32_t *sample_faces, const double *xyz, int64_t count,
                    const pto_point *pts, int64_t n, const int32_t *idx, const double *d2, int k, int res,
                    float *height)
{
    const size_t n_pix = (size_t)res * res;
    for (size_t i = 0; i < n_pix; ++i) height[i] = nan_value();
    for (int64_t s = 0; s < count; ++s) {
        if (texels[s] >= n_pix || sample_faces[s] < 0 || sample_faces[s] >= nf) return 1;
        const int32_t *face = faces + 3 * (int64_t)sample_faces[s];
        bv2 t[3];
        for (int j = 0; j < 3; ++j) {
            if (face[j] < 0 || face[j] >= nv) return 1;
            t[j].a = v[face[j]].U * res;
            t[j].b = v[face[j]].V * res;
        }
        const size_t tx = texels[s];
        /* 1. the owner face's barycentrics of the texel centre and the mixed vertex normal */
        const bv2 p = {(double)(tx % res) + 0.5, (double)(res - (int)(tx / res)) - 0.5};
        const double inv = 1.0 / area2(t[0], t[1], t[2]);
        double bc[3];
        bc[0] = area2(t[1], t[2], p) * inv;
        bc[1] = area2(t[2], t[0], p) * inv;
        bc[2] = 1.0 - bc[0] - bc[1];
        const d3 na = d3_of(frames + 8 * (size_t)face[0]), nb = d3_of(frames + 8 * (size_t)face[1]),
                 nc = d3_of(frames + 8 * (size_t)face[2]);
        const d3 nm = add3(add3(scale3(bc[0], na), scale3(bc[1], nb)), scale3(bc[2], nc));
        if (!usable3(nm)) continue;
        const double l = sqrt(dot3(nm, nm));
        const d3 N = {nm.x / l, nm.y / l, nm.z / l};
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
static uint16_t encode(float h, double lo, double hi)
{
    if (hi == lo) return 0;
    const double s = 65535.0 / (hi - lo);
    const double e = floor(((double)h - lo) * s + 0.5);
    return (uint16_t)fmin(fmax(e, 0.0), 65535.0);
}

/* -0 orders below +0, as a sign-magnitude comparison does */
static int below(float a, float b) { return a < b || (a == b && signbit(a) && !signbit(b)); }

int64_t pth_bake_height_encode(const float *height, int64_t n_pix, const double *range_in, uint16_t *codes,
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
    for (int64_t i = 0; i < n_pix; ++i) codes[i] = isnan(height[i]) ? 0 : encode(height[i], l, u);
    return valued;
}

/* word = E + 1 with a value, else 0; 25-wide maxima along rows, then along columns; a texel
 * without a value takes the window's maximum minus one (0 if the window has no value) */
int pth_bake_height_pad(const float *height, const uint16_t *codes, int res, uint16_t *padded)
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

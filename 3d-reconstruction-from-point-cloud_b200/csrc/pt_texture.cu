// pt_texture.cu -- per-face transfer and texture output on the GPU (SURVEY.md section 8 rows
// N1 / N3 / N4): everything the reference does AFTER the neighbour search,
// /root/reference src/pointsTransfer.cpp:
//   :484-537  project the neighbours of a face's corners onto the face plane, keep those inside
//   :539-581  2-D Delaunay triangulation of corners + inside points, UVs by barycentric mix
//   :66-107   draw_triangle -- rasterise every sub-triangle into the BGRA texture
//   :593-611  25 x 25 dilate, gutter = dilated & ~alpha, padded = texture + gutter
//
// One thread per face runs :484-581 start to finish (the data of a face -- <= 3 K neighbours --
// lives in its local arrays) and rasterises its sub-triangles itself.  The reference draws faces
// one after the other, later ones overwriting earlier ones where sub-triangles meet; here every
// pixel write is a 64-bit atomicMax on (face << 8 | sub-triangle rank) << 32 | BGRA, so the
// result is that same "last writer in reference order wins", independent of scheduling.
//
// CGAL is restated from memory (flagged in oracle/pt_texture_oracle.c, the CPU statement of the
// same definitions, which the tests compare this file with bit for bit): Plane_3::to_2d's
// stretched frame, Triangle_coordinates_2, and Delaunay by its definition (a non-degenerate
// triple is a face iff no other point is strictly inside its circumcircle; the in-circle sign is
// evaluated once per index-sorted quadruple).  Not reproduced: the out-of-bounds row
// `resolution - j` at j = 0 / column `resolution` (:100-103) and the uninitialised Mat (:402).
#include <algorithm>
#include <cmath>
#include <initializer_list>
#include <vector>

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <cub/device/device_select.cuh>
#include <thrust/iterator/counting_iterator.h>

#include "pt_index.cuh"

namespace pt {

constexpr int TEX_MAX_NB = 3 * PT_MAX_K;      // neighbours of one face before the union
constexpr int TEX_MAX_PTS = 3 + TEX_MAX_NB;

struct V2 { double a, b; };

struct MeshVertex {      // what a face needs of a mesh vertex (unpacked from the 80-byte Point)
    double x, y, z, u, v;
    int    r, g, b;
    int    pad;
};

struct Raw80t {
    double ver[3];
    double normal[3];
    int    color[3];
    int    pad;
    double U, V;
};

__global__ void __launch_bounds__(256)
tex_unpack_vertices_kernel(const Raw80t *raw, uint32_t n, MeshVertex *mv, double *xyz)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const Raw80t r = raw[i];
    MeshVertex m;
    m.x = r.ver[0]; m.y = r.ver[1]; m.z = r.ver[2];
    m.u = r.U; m.v = r.V;
    m.r = r.color[0]; m.g = r.color[1]; m.b = r.color[2];
    m.pad = 0;
    mv[i] = m;
    xyz[3 * (size_t)i] = r.ver[0]; xyz[3 * (size_t)i + 1] = r.ver[1]; xyz[3 * (size_t)i + 2] = r.ver[2];
}

template <typename PT>
__global__ void __launch_bounds__(256) tex_inverse_perm_kernel(const PT *pts, uint32_t n, uint32_t *inv)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) inv[pts[i].idx] = i;
}

__device__ __forceinline__ double tx_area2(V2 p, V2 q, V2 r)
{
    return (q.a - p.a) * (r.b - p.b) - (q.b - p.b) * (r.a - p.a);
}
__device__ __forceinline__ void tx_tri_coords(V2 v0, V2 v1, V2 v2, V2 x, double bc[3])
{
    const double inv = 1.0 / tx_area2(v0, v1, v2);
    bc[0] = tx_area2(v1, v2, x) * inv;
    bc[1] = tx_area2(v2, v0, x) * inv;
    bc[2] = 1.0 - bc[0] - bc[1];
}
__device__ __forceinline__ double tx_incircle(V2 a, V2 b, V2 c, V2 d)
{
    const double ax = a.a - d.a, ay = a.b - d.b, bx = b.a - d.a, by = b.b - d.b, cx = c.a - d.a, cy = c.b - d.b;
    const double al = ax * ax + ay * ay, bl = bx * bx + by * by, cl = cx * cx + cy * cy;
    return ax * (by * cl - bl * cy) - ay * (bx * cl - bl * cx) + al * (bx * cy - by * cx);
}
__device__ __forceinline__ double tx_dot3(const double *u, const double *v)
{
    return u[0] * v[0] + u[1] * v[1] + u[2] * v[2];
}
__device__ __forceinline__ V2 tx_to_2d(const double x[3], const double r[3], const double n[3],
                                       const double b1[3], const double b2[3])
{
    const double w[3] = {x[0] - r[0], x[1] - r[1], x[2] - r[2]};
    const double t = tx_dot3(w, n) / tx_dot3(n, n);
    const double pr[3] = {w[0] - t * n[0], w[1] - t * n[1], w[2] - t * n[2]};
    V2 o;
    o.a = tx_dot3(pr, b1) / tx_dot3(b1, b1);
    o.b = tx_dot3(pr, b2) / tx_dot3(b2, b2);
    return o;
}

struct TexVertex { double u, v; int r, g, b; };

// src/pointsTransfer.cpp:66-107; `order` = (face << 8 | sub-triangle rank), later wins
__device__ void tx_draw_triangle(const TexVertex &t0, const TexVertex &t1, const TexVertex &t2, int res,
                                 unsigned long long *canvas, unsigned long long order)
{
    V2 p, q, r;
    p.a = t0.u * res; p.b = t0.v * res;
    q.a = t1.u * res; q.b = t1.v * res;
    r.a = t2.u * res; r.b = t2.v * res;
    const double xmin = fmin(p.a, fmin(q.a, r.a)), xmax = fmax(p.a, fmax(q.a, r.a));
    const double ymin = fmin(p.b, fmin(q.b, r.b)), ymax = fmax(p.b, fmax(q.b, r.b));
    if (!(xmax - xmin < 4.0 * res) || !(ymax - ymin < 4.0 * res)) return;      // NaN / absurd UVs
    const double fx1 = floor(xmax), fy1 = floor(ymax);
    for (int i = (int)floor(xmin); i <= fx1; i++) {
        for (int j = (int)floor(ymin); j <= fy1; j++) {
            int x = i, y = j;
            if (x >= res) x = res - 1;
            if (y >= res) y = res - 1;
            double bc[3];
            V2 px;
            px.a = (double)x; px.b = (double)y;
            tx_tri_coords(p, q, r, px, bc);
            if (bc[0] >= 0 && bc[1] >= 0 && bc[2] >= 0) {
                const float fr = (float)(bc[0] * t0.r + bc[1] * t1.r + bc[2] * t2.r);
                const float fg = (float)(bc[0] * t0.g + bc[1] * t1.g + bc[2] * t2.g);
                const float fb = (float)(bc[0] * t0.b + bc[1] * t1.b + bc[2] * t2.b);
                const int row = res - j, col = i;
                if (row < 0 || row >= res || col < 0 || col >= res) continue;    // out of bounds in the reference
                const unsigned bgra = ((unsigned)(int)fb & 0xffu) | (((unsigned)(int)fg & 0xffu) << 8) |
                                      (((unsigned)(int)fr & 0xffu) << 16) | 0xff000000u;
                atomicMax(canvas + (size_t)row * res + col, (order << 32) | bgra);
            }
        }
    }
}

// where the position of cloud point `id` (original index) comes from
template <typename PT> struct PosSorted {      // an index: sorted records + inverse permutation
    const PT *pts;
    const uint32_t *inv;
    __device__ __forceinline__ void get(int id, double x[3]) const
    {
        const PT rec = pts[inv[id]];
        x[0] = (double)rec.x; x[1] = (double)rec.y; x[2] = (double)rec.z;
    }
};
struct PosPlain {                               // n x 3 doubles in original order
    const double *xyz;
    __device__ __forceinline__ void get(int id, double x[3]) const
    {
        x[0] = xyz[3 * (size_t)id]; x[1] = xyz[3 * (size_t)id + 1]; x[2] = xyz[3 * (size_t)id + 2];
    }
};

template <typename POS>
__global__ void __launch_bounds__(64)
tex_face_kernel(const POS pos, uint32_t n_points, const pt_attr *attrs, const MeshVertex *mv,
                const int32_t *idx, int k, const int32_t *faces, uint32_t n_faces, uint32_t n_vertices,
                int res, unsigned long long *canvas, unsigned long long *stats)
{
    const uint32_t f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= n_faces) return;
    int vi[3];
    MeshVertex tv[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        vi[c] = faces[3 * (size_t)f + c];
        if (vi[c] < 0 || (uint32_t)vi[c] >= n_vertices) return;      // malformed face: nothing to draw
        tv[c] = mv[vi[c]];
    }
    // union of the corners' neighbour lists (src/pointsTransfer.cpp:470-479), by point index
    int nb[TEX_MAX_NB], n_nb = 0;
    for (int c = 0; c < 3; ++c)
        for (int j = 0; j < k; ++j) {
            const int id = idx[(size_t)vi[c] * k + j];
            if (id < 0 || (uint32_t)id >= n_points) continue;
            bool seen = false;
            for (int e = 0; e < n_nb; ++e) seen |= nb[e] == id;
            if (!seen) nb[n_nb++] = id;
        }
    // Plane_3(r, p, q) and its 2-D frame (:490-494)
    const double R[3] = {tv[0].x, tv[0].y, tv[0].z};
    const double e1[3] = {tv[1].x - R[0], tv[1].y - R[1], tv[1].z - R[2]};
    const double e2[3] = {tv[2].x - R[0], tv[2].y - R[1], tv[2].z - R[2]};
    double n[3], b1[3], b2[3];
    n[0] = e1[1] * e2[2] - e1[2] * e2[1];
    n[1] = e1[2] * e2[0] - e1[0] * e2[2];
    n[2] = e1[0] * e2[1] - e1[1] * e2[0];
    {
        const double a = n[0], b = n[1], c = n[2];
        if (a == 0.0) { b1[0] = 1; b1[1] = 0; b1[2] = 0; }
        else if (b == 0.0) { b1[0] = 0; b1[1] = 1; b1[2] = 0; }
        else if (c == 0.0) { b1[0] = 0; b1[1] = 0; b1[2] = 1; }
        else if (fabs(a) <= fabs(b) && fabs(a) <= fabs(c)) { b1[0] = 0; b1[1] = -c; b1[2] = b; }
        else if (fabs(b) <= fabs(a) && fabs(b) <= fabs(c)) { b1[0] = -c; b1[1] = 0; b1[2] = a; }
        else { b1[0] = -b; b1[1] = a; b1[2] = 0; }
    }
    b2[0] = n[1] * b1[2] - n[2] * b1[1];
    b2[1] = n[2] * b1[0] - n[0] * b1[2];
    b2[2] = n[0] * b1[1] - n[1] * b1[0];

    V2 P[TEX_MAX_PTS];
    TexVertex V[TEX_MAX_PTS];
    int np = 3;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const double x[3] = {tv[c].x, tv[c].y, tv[c].z};
        P[c] = tx_to_2d(x, R, n, b1, b2);
        V[c].u = tv[c].u; V[c].v = tv[c].v;
        V[c].r = tv[c].r; V[c].g = tv[c].g; V[c].b = tv[c].b;
    }
    for (int e = 0; e < n_nb; ++e) {
        double x[3];
        pos.get(nb[e], x);
        const V2 xp = tx_to_2d(x, R, n, b1, b2);
        double bc[3];
        tx_tri_coords(P[0], P[1], P[2], xp, bc);
        if (bc[0] >= 0 && bc[1] >= 0 && bc[2] >= 0) {        // :530
            const pt_attr at = attrs[nb[e]];
            P[np] = xp;
            V[np].u = bc[0] * tv[0].u + bc[1] * tv[1].u + bc[2] * tv[2].u;      // :572
            V[np].v = bc[0] * tv[0].v + bc[1] * tv[1].v + bc[2] * tv[2].v;      // :573
            V[np].r = at.r; V[np].g = at.g; V[np].b = at.b;
            ++np;
        }
    }
    unsigned drawn = 0;
    const unsigned long long fkey = (unsigned long long)f << 8;
    if (np == 3) {                                           // :540-544
        tx_draw_triangle(V[0], V[1], V[2], res, canvas, fkey);
        drawn = 1;
    } else {                                                 // :545-581, Delaunay by its definition
        for (int a = 0; a < np; ++a)
            for (int b = a + 1; b < np; ++b)
                for (int c = b + 1; c < np; ++c) {
                    const double o = tx_area2(P[a], P[b], P[c]);
                    if (o == 0.0 || o != o) continue;
                    bool ok = true;
                    for (int d = 0; d < np && ok; ++d) {
                        if (d == a || d == b || d == c) continue;
                        // in-circle determinant of the index-sorted quadruple, signed by the
                        // permutation that sorts (a, b, c, d): see oracle/pt_texture_oracle.c
                        int q0 = a, q1 = b, q2 = c, q3 = d, sw = 0;
                        if (q3 < q2) { const int t = q3; q3 = q2; q2 = t; ++sw; }
                        if (q2 < q1) { const int t = q2; q2 = q1; q1 = t; ++sw; }
                        if (q1 < q0) { const int t = q1; q1 = q0; q0 = t; ++sw; }
                        double s = tx_incircle(P[q0], P[q1], P[q2], P[q3]);
                        if (sw & 1) s = -s;
                        if (o < 0) s = -s;
                        if (s > 0) ok = false;
                    }
                    if (!ok) continue;
                    tx_draw_triangle(V[a], V[b], V[c], res, canvas, fkey | (drawn < 255u ? drawn : 255u));
                    ++drawn;
                }
    }
    if (stats) {
        atomicAdd(&stats[0], (unsigned long long)drawn);
        atomicAdd(&stats[1], (unsigned long long)(np - 3));
    }
}

__global__ void __launch_bounds__(256)
tex_resolve_kernel(const unsigned long long *canvas, size_t n_pix, uint32_t *tex)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_pix) tex[i] = (uint32_t)(canvas[i] & 0xffffffffull);     // never written: 0 (alpha 0)
}

// The 25 x 25 padding window as two separable 25-tap maxima (OpenCV ignores the border), then the
// combine of each texel's own value with its window's maximum.  PAD gives both:
//   PadBgra    :593-611 on BGRA texels: byte-wise maxima, padded = texture + (dilated & ~alpha)
//   PadHeight  height words (E + 1, or 0 without a value): word maxima, since byte-wise ones would
//              mix the two bytes of a code; a texel without a value takes the window's largest code
struct PadBgra {
    using Out = uint32_t;
    __device__ __forceinline__ static uint32_t max(uint32_t a, uint32_t b) { return __vmaxu4(a, b); }
    __device__ __forceinline__ static Out combine(uint32_t t, uint32_t m)
    {
        const uint32_t alpha = t >> 24;
        const uint32_t not_alpha = (alpha ^ 0xffu) * 0x01010101u;  // ~alpha replicated to the 4 channels
        return __vaddus4(t, m & not_alpha);
    }
};
struct PadHeight {
    using Out = uint16_t;
    __device__ __forceinline__ static uint32_t max(uint32_t a, uint32_t b) { return ::max(a, b); }
    __device__ __forceinline__ static Out combine(uint32_t w, uint32_t m)
    {
        const uint32_t t = w ? w : m;
        return (uint16_t)(t ? t - 1u : 0u);
    }
};

template <typename PAD>
__global__ void __launch_bounds__(256) pad_window_h_kernel(const uint32_t *img, int res, uint32_t *tmp)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)res * res) return;
    const int y = (int)(i / res), x = (int)(i % res);
    uint32_t m = 0;
    for (int dx = -12; dx <= 12; ++dx) {
        const int xx = x + dx;
        if (xx >= 0 && xx < res) m = PAD::max(m, img[(size_t)y * res + xx]);
    }
    tmp[i] = m;
}
// reads only its own texel of img, so out may be img
template <typename PAD>
__global__ void __launch_bounds__(256)
pad_window_v_kernel(const uint32_t *img, const uint32_t *tmp, int res, typename PAD::Out *out)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)res * res) return;
    const int y = (int)(i / res), x = (int)(i % res);
    uint32_t m = 0;
    for (int dy = -12; dy <= 12; ++dy) {
        const int yy = y + dy;
        if (yy >= 0 && yy < res) m = PAD::max(m, tmp[(size_t)yy * res + x]);
    }
    out[i] = PAD::combine(img[i], m);
}

static inline unsigned tcdiv(size_t a, size_t b) { return (unsigned)((a + b - 1) / b); }

// tmp: res * res words of scratch
template <typename PAD>
static void launch_pad_window(const uint32_t *img, uint32_t *tmp, int res, typename PAD::Out *out, cudaStream_t s)
{
    const size_t n_pix = (size_t)res * res;
    pad_window_h_kernel<PAD><<<tcdiv(n_pix, 256), 256, 0, s>>>(img, res, tmp);
    pad_window_v_kernel<PAD><<<tcdiv(n_pix, 256), 256, 0, s>>>(img, tmp, res, out);
    count_launch(2);
}

// Pads the given 8-bit maps (null entries skipped) in place.
static int bake_pad(std::initializer_list<uint8_t *> imgs, int res, cudaStream_t s)
{
    bool any = false;
    for (uint8_t *img : imgs) any |= img != nullptr;
    if (!any) return PT_OK;
    uint32_t *d_tmp = nullptr;
    PT_TRY(pool_alloc((void **)&d_tmp, 4 * (size_t)res * res, s));
    for (uint8_t *img : imgs)
        if (img) launch_pad_window<PadBgra>((const uint32_t *)img, d_tmp, res, (uint32_t *)img, s);
    pool_free(d_tmp, s);
    return PT_OK;
}

// Mesh upload + (optionally) the neighbour search + face kernel + post-process.  `ix` gives the
// stream, the query kernels (when d_idx_given is null) and the attribute array.
template <typename POS>
static int texture_pipeline(pt_index *ix, POS pos, uint32_t n_points, const pt_attr *attrs, bool search,
                            const int32_t *idx_host, const void *vertices, size_t n_vertices,
                            const int32_t *faces, size_t n_faces, int k, double radius, int res, int pad,
                            uint8_t *bgra_out, pt_texture_stats *st)
{
    cudaStream_t s = ix->stream;
    const size_t n_pix = (size_t)res * res;
    Raw80t *d_raw = nullptr;
    MeshVertex *d_mv = nullptr;
    double *d_xyz = nullptr;
    int32_t *d_idx = nullptr, *d_faces = nullptr;
    unsigned long long *d_canvas = nullptr, *d_stats = nullptr;
    uint32_t *d_tex = nullptr;
    cudaEvent_t ev[4] = {};
    int rc = PT_OK;
    auto fail = [&](cudaError_t e) { if (e != cudaSuccess && rc == PT_OK) rc = map_cuda_error(e); return e != cudaSuccess; };
    do {
        for (auto &e : ev) if (fail(cudaEventCreate(&e))) break;
        if (rc != PT_OK) break;
        if (pool_alloc((void **)&d_raw, sizeof(Raw80t) * n_vertices, s) || pool_alloc((void **)&d_mv, sizeof(MeshVertex) * n_vertices, s) ||
            pool_alloc((void **)&d_xyz, sizeof(double) * 3 * n_vertices, s) || pool_alloc((void **)&d_idx, sizeof(int32_t) * n_vertices * k, s) ||
            pool_alloc((void **)&d_faces, sizeof(int32_t) * 3 * n_faces, s) || pool_alloc((void **)&d_canvas, sizeof(unsigned long long) * n_pix, s) ||
            pool_alloc((void **)&d_stats, 16, s) || pool_alloc((void **)&d_tex, 4 * n_pix, s)) {
            rc = PT_ERR_OUT_OF_MEMORY;
            break;
        }
        if (fail(cudaEventRecord(ev[0], s))) break;
        if (fail(cudaMemcpyAsync(d_raw, vertices, sizeof(Raw80t) * n_vertices, cudaMemcpyHostToDevice, s))) break;
        if (fail(cudaMemcpyAsync(d_faces, faces, sizeof(int32_t) * 3 * n_faces, cudaMemcpyHostToDevice, s))) break;
        if (fail(cudaMemsetAsync(d_canvas, 0, sizeof(unsigned long long) * n_pix, s))) break;
        if (fail(cudaMemsetAsync(d_stats, 0, 16, s))) break;
        if (n_vertices) {
            tex_unpack_vertices_kernel<<<tcdiv(n_vertices, 256), 256, 0, s>>>(d_raw, (uint32_t)n_vertices, d_mv, d_xyz);
            count_launch();
        }
        if (search) {
            // the neighbour search of every UNIQUE vertex (the reference searches 3 x per face, :474)
            QueryParams qp{};
            fill_params(ix, qp);
            qp.queries = d_xyz; qp.m = (uint32_t)n_vertices; qp.k = k;
            qp.r2 = radius_to_r2(radius);
            qp.idx_out = d_idx;
            if ((rc = launch_query(ix, qp, s)) != PT_OK) break;
        } else if (n_vertices) {
            if (fail(cudaMemcpyAsync(d_idx, idx_host, sizeof(int32_t) * n_vertices * k, cudaMemcpyHostToDevice, s))) break;
        }
        if (fail(cudaEventRecord(ev[1], s))) break;
        if (n_faces) {
            tex_face_kernel<POS><<<tcdiv(n_faces, 64), 64, 0, s>>>(pos, n_points, attrs, d_mv, d_idx, k, d_faces,
                                                                (uint32_t)n_faces, (uint32_t)n_vertices, res, d_canvas,
                                                                d_stats);
            count_launch();
        }
        tex_resolve_kernel<<<tcdiv(n_pix, 256), 256, 0, s>>>(d_canvas, n_pix, d_tex);
        count_launch();
        if (fail(cudaEventRecord(ev[2], s))) break;
        if (pad && (rc = bake_pad({(uint8_t *)d_tex}, res, s)) != PT_OK) break;
        if (fail(cudaEventRecord(ev[3], s))) break;
        if (fail(cudaGetLastError())) break;
        if (fail(cudaMemcpyAsync(bgra_out, d_tex, 4 * n_pix, cudaMemcpyDeviceToHost, s))) break;
        unsigned long long h_stats[2] = {0, 0};
        if (fail(cudaMemcpyAsync(h_stats, d_stats, 16, cudaMemcpyDeviceToHost, s))) break;
        if (fail(cudaStreamSynchronize(s))) break;
        if (st) {
            st->triangles = h_stats[0];
            st->inside_points = h_stats[1];
            cudaEventElapsedTime(&st->knn_ms, ev[0], ev[1]);
            cudaEventElapsedTime(&st->draw_ms, ev[1], ev[2]);
            cudaEventElapsedTime(&st->pad_ms, ev[2], ev[3]);
        }
    } while (0);
    cudaStreamSynchronize(s);
    void *frees[] = {d_raw, d_mv, d_xyz, d_idx, d_faces, d_canvas, d_stats, d_tex};
    for (void *p : frees) pool_free(p, s);
    for (auto &e : ev) if (e) cudaEventDestroy(e);
    cudaGetLastError();
    return rc;
}

// original index -> position in the sorted cloud, built once per index
template <typename PT>
static int index_inverse_perm(pt_index *ix)
{
    if (!ix->inv_perm && ix->n) {
        PT_TRY(dev_alloc((void **)&ix->inv_perm, sizeof(uint32_t) * (size_t)ix->n));
        tex_inverse_perm_kernel<PT><<<tcdiv(ix->n, 256), 256, 0, ix->stream>>>((const PT *)ix->pts, ix->n, ix->inv_perm);
        count_launch();
    }
    return PT_OK;
}

template <typename PT>
static int texture_render_index(pt_index *ix, const void *vertices, size_t n_vertices, const int32_t *faces,
                                size_t n_faces, int k, double radius, int res, int pad, uint8_t *bgra_out,
                                pt_texture_stats *st)
{
    PT_TRY(index_inverse_perm<PT>(ix));
    PosSorted<PT> pos{(const PT *)ix->pts, ix->inv_perm};
    return texture_pipeline(ix, pos, ix->n, ix->attrs, true, nullptr, vertices, n_vertices, faces, n_faces, k, radius,
                            res, pad, bgra_out, st);
}

// ---- per-texel bake (DESIGN.md section 8, "Per-texel bake") ---------------------------------------
// Texel (col, row) of a res x res image (row 0 on top) samples p = (col + 0.5, res - row - 0.5) in
// UV * res units.  Face f covers it when all barycentrics of p in (U * res, V * res) are >= 0
// (tx_tri_coords); where faces overlap the highest face index wins.  The sample position is the
// barycentric mix of the winning face's 3-D corners, fp64, never contracted.
//
// Vertices are read through a stride, so both the caller's n x 5 (x, y, z, u, v) rows and the
// n x 8 rows (x, y, z, u, v, nx, ny, nz) of bake_unpack_vertices_kernel can be rasterised.
constexpr int BAKE_TILE = 32;                  // one warp per (face, 32 x 32-texel tile of its box)

struct BakeMesh {
    const double  *v;          // n_vertices rows of `stride` doubles: x, y, z, u, v, ...
    int            stride;
    uint32_t       n_vertices;
    const int32_t *faces;
    uint32_t       n_faces;
    int            res;
};

// corners of face f; false for an out-of-range vertex index (the face covers nothing)
__device__ __forceinline__ bool bake_corners(const BakeMesh &M, uint32_t f, const double *c[3])
{
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        const int32_t vi = M.faces[3 * (size_t)f + j];
        if (vi < 0 || (uint32_t)vi >= M.n_vertices) return false;
        c[j] = M.v + (size_t)vi * M.stride;
    }
    return true;
}

// UV triangle in UV * res units (the multiplications of tx_draw_triangle)
__device__ __forceinline__ void bake_uv(const BakeMesh &M, const double *const c[3], V2 t[3])
{
#pragma unroll
    for (int j = 0; j < 3; ++j) { t[j].a = c[j][3] * M.res; t[j].b = c[j][4] * M.res; }
}

__device__ __forceinline__ V2 bake_texel_point(int res, int col, int row)
{
    V2 p;
    p.a = (double)col + 0.5;
    p.b = (double)(res - row) - 0.5;
    return p;
}

// barycentrics of texel tex's centre on the face with corners c, as the texel stage computes them
__device__ __forceinline__ void bake_texel_bary(const BakeMesh &M, const double *const c[3], uint32_t tex, double bc[3])
{
    V2 t[3];
    bake_uv(M, c, t);
    tx_tri_coords(t[0], t[1], t[2], bake_texel_point(M.res, (int)(tex % (uint32_t)M.res), (int)(tex / (uint32_t)M.res)), bc);
}

// Texels whose centre lies in the UV triangle's bounding box, widened by one texel so that rounding
// in the barycentrics can never reach a texel outside it, clipped to the image.  false: none
// (NaN UVs, or a box outside the image).
__device__ __forceinline__ bool bake_box(const V2 t[3], int res, int &c0, int &r0, int &nc, int &nr)
{
    const double xmin = fmin(t[0].a, fmin(t[1].a, t[2].a)), xmax = fmax(t[0].a, fmax(t[1].a, t[2].a));
    const double ymin = fmin(t[0].b, fmin(t[1].b, t[2].b)), ymax = fmax(t[0].b, fmax(t[1].b, t[2].b));
    if (!(xmin <= xmax) || !(ymin <= ymax) || t[0].a != t[0].a || t[1].a != t[1].a || t[2].a != t[2].a ||
        t[0].b != t[0].b || t[1].b != t[1].b || t[2].b != t[2].b)
        return false;
    const double lim = (double)(res - 1);
    const double cl = fmax(ceil(xmin - 0.5) - 1.0, 0.0), ch = fmin(floor(xmax - 0.5) + 1.0, lim);
    const double rl = fmax(ceil((double)res - 0.5 - ymax) - 1.0, 0.0), rh = fmin(floor((double)res - 0.5 - ymin) + 1.0, lim);
    if (!(cl <= ch) || !(rl <= rh)) return false;
    c0 = (int)cl; r0 = (int)rl;
    nc = (int)ch - c0 + 1; nr = (int)rh - r0 + 1;
    return true;
}

__global__ void __launch_bounds__(256) bake_tile_count_kernel(const BakeMesh M, unsigned long long *tiles)
{
    const uint32_t f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= M.n_faces) return;
    const double *c[3];
    V2 t[3];
    int c0, r0, nc, nr;
    unsigned long long n = 0;
    if (bake_corners(M, f, c)) {
        bake_uv(M, c, t);
        if (bake_box(t, M.res, c0, r0, nc, nr))
            n = (unsigned long long)((nc + BAKE_TILE - 1) / BAKE_TILE) * (unsigned long long)((nr + BAKE_TILE - 1) / BAKE_TILE);
    }
    tiles[f] = n;
}

// Work item w (< total = first[n_faces - 1] + tiles of the last face, exclusive scan `first`) is tile
// w - first[f] of face f.  A warp walks its tile column by column (lane = column, coalesced) and
// claims every covered texel with atomicMax(owner, f + 1): the highest covering face wins whatever
// the schedule.
__global__ void __launch_bounds__(256)
bake_raster_kernel(const BakeMesh M, const unsigned long long *first, const unsigned long long *last_tiles,
                   uint32_t *owner)
{
    const unsigned long long total = first[M.n_faces - 1] + *last_tiles;
    const unsigned lane = threadIdx.x & 31u;
    const unsigned long long warps = (unsigned long long)gridDim.x * (blockDim.x >> 5);
    for (unsigned long long w = ((unsigned long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; w < total; w += warps) {
        uint32_t lo = 0, hi = M.n_faces;          // last face with first[f] <= w
        while (hi - lo > 1) {
            const uint32_t mid = (lo + hi) >> 1;
            if (first[mid] <= w) lo = mid; else hi = mid;
        }
        const uint32_t f = lo;
        const double *c[3];
        bake_corners(M, f, c);                    // a face with tiles has valid corners
        V2 t[3];
        bake_uv(M, c, t);
        int c0, r0, nc, nr;
        bake_box(t, M.res, c0, r0, nc, nr);
        const unsigned long long tile = w - first[f];
        const int tiles_x = (nc + BAKE_TILE - 1) / BAKE_TILE;
        const int tx = (int)(tile % (unsigned long long)tiles_x), ty = (int)(tile / (unsigned long long)tiles_x);
        const int col = c0 + tx * BAKE_TILE + (int)lane;
        if (col >= c0 + nc) continue;
        const int row_end = min(r0 + (ty + 1) * BAKE_TILE, r0 + nr);
        for (int row = r0 + ty * BAKE_TILE; row < row_end; ++row) {
            double bc[3];
            tx_tri_coords(t[0], t[1], t[2], bake_texel_point(M.res, col, row), bc);
            if (bc[0] >= 0 && bc[1] >= 0 && bc[2] >= 0)
                atomicMax(owner + (size_t)row * M.res + col, f + 1u);
        }
    }
}

struct BakeCovered {
    const uint32_t *owner;
    __device__ __forceinline__ bool operator()(uint32_t t) const { return owner[t] != 0u; }
};

// position of sample i (texel texels[i]) on its owner face, and the face itself when face_out is set
__global__ void __launch_bounds__(256)
bake_position_kernel(const BakeMesh M, const uint32_t *owner, const uint32_t *texels, uint32_t count, double *xyz,
                     int32_t *face_out)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    const uint32_t tex = texels[i];
    const uint32_t f = owner[tex] - 1u;
    if (face_out) face_out[i] = (int32_t)f;
    const double *c[3];
    bake_corners(M, f, c);
    double bc[3];
    bake_texel_bary(M, c, tex, bc);
#pragma unroll
    for (int a = 0; a < 3; ++a)
        xyz[3 * (size_t)i + a] = __dadd_rn(__dadd_rn(__dmul_rn(bc[0], c[0][a]), __dmul_rn(bc[1], c[1][a])),
                                           __dmul_rn(bc[2], c[2][a]));
}

// Owner map -> samples in ascending texel order.  M.faces / M.v are device pointers on the current
// device.  texel_out / xyz_out: room for res * res samples, or both null (count only); face_out
// (owner face per sample, may be null) needs them.  Synchronises `s`; *count_out is the number of
// covered texels.
static int bake_texels(const BakeMesh &M, uint32_t *texel_out, double *xyz_out, int32_t *face_out, size_t *count_out,
                       cudaStream_t s)
{
    const size_t n_pix = (size_t)M.res * M.res;
    unsigned long long *d_tiles = nullptr, *d_first = nullptr;
    uint32_t *d_owner = nullptr, *d_sel = nullptr, *d_count = nullptr;
    void *d_tmp = nullptr;
    int rc = PT_OK;
    auto fail = [&](cudaError_t e) { if (e != cudaSuccess && rc == PT_OK) rc = map_cuda_error(e); return e != cudaSuccess; };
    *count_out = 0;
    do {
        const size_t nf = M.n_faces ? M.n_faces : 1;
        size_t scan_bytes = 0, select_bytes = 0;
        thrust::counting_iterator<uint32_t> ids(0);
        if (fail(cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, d_tiles, d_first, (int)nf, s))) break;
        if (fail(cub::DeviceSelect::If(nullptr, select_bytes, ids, d_sel, d_count, (int)n_pix, BakeCovered{d_owner}, s))) break;
        if (pool_alloc((void **)&d_tiles, sizeof(unsigned long long) * nf, s) ||
            pool_alloc((void **)&d_first, sizeof(unsigned long long) * nf, s) ||
            pool_alloc((void **)&d_owner, sizeof(uint32_t) * n_pix, s) || pool_alloc((void **)&d_count, sizeof(uint32_t), s) ||
            pool_alloc(&d_tmp, scan_bytes > select_bytes ? scan_bytes : select_bytes, s) ||
            (!texel_out && pool_alloc((void **)&d_sel, sizeof(uint32_t) * n_pix, s))) {
            rc = PT_ERR_OUT_OF_MEMORY;
            break;
        }
        uint32_t *sel = texel_out ? texel_out : d_sel;
        if (fail(cudaMemsetAsync(d_owner, 0, sizeof(uint32_t) * n_pix, s))) break;
        if (M.n_faces) {
            bake_tile_count_kernel<<<tcdiv(M.n_faces, 256), 256, 0, s>>>(M, d_tiles);
            count_launch();
            if (fail(cub::DeviceScan::ExclusiveSum(d_tmp, scan_bytes, d_tiles, d_first, (int)M.n_faces, s))) break;
            // enough warps to fill the device several times over; each strides over the work list
            bake_raster_kernel<<<148 * 16, 256, 0, s>>>(M, d_first, d_tiles + (M.n_faces - 1), d_owner);
            count_launch(2);
        }
        if (fail(cub::DeviceSelect::If(d_tmp, select_bytes, ids, sel, d_count, (int)n_pix, BakeCovered{d_owner}, s))) break;
        count_launch();
        uint32_t count = 0;
        if (fail(cudaMemcpyAsync(&count, d_count, sizeof count, cudaMemcpyDeviceToHost, s))) break;
        if (fail(cudaStreamSynchronize(s))) break;
        if (xyz_out && count) {
            bake_position_kernel<<<tcdiv(count, 256), 256, 0, s>>>(M, d_owner, sel, count, xyz_out, face_out);
            count_launch();
        }
        if (fail(cudaGetLastError())) break;
        *count_out = count;
    } while (0);
    void *frees[] = {d_tiles, d_first, d_owner, d_sel, d_count, d_tmp};
    for (void *p : frees) pool_free(p, s);
    if (fail(cudaStreamSynchronize(s))) *count_out = 0;
    return rc;
}

// e(n) = clamp(floor((n + 1) * 127.5 + 0.5), 0, 255), fp64 from the fp32 component
__device__ __forceinline__ uint32_t bake_encode(float n)
{
    const double v = floor(__dadd_rn(__dmul_rn(__dadd_rn((double)n, 1.0), 127.5), 0.5));
    return (uint32_t)fmin(fmax(v, 0.0), 255.0);
}

// sample i -> its texel in the three maps; an empty neighbour list (rgba alpha 0) leaves zeros
__global__ void __launch_bounds__(256)
bake_compose_kernel(const uint32_t *texels, uint32_t count, const uint8_t *rgba, const float *normal,
                    uint32_t *bgra, uint32_t *nbgra, float *nf, unsigned long long *empty)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    const uchar4 c = reinterpret_cast<const uchar4 *>(rgba)[i];
    if (c.w == 0) {
        if (empty) atomicAdd(empty, 1ull);
        return;
    }
    const size_t t = texels[i];
    const float x = normal[3 * (size_t)i], y = normal[3 * (size_t)i + 1], z = normal[3 * (size_t)i + 2];
    if (bgra) bgra[t] = (uint32_t)c.z | ((uint32_t)c.y << 8) | ((uint32_t)c.x << 16) | 0xff000000u;
    if (nbgra) nbgra[t] = bake_encode(z) | (bake_encode(y) << 8) | (bake_encode(x) << 16) | 0xff000000u;
    if (nf) { nf[3 * t] = x; nf[3 * t + 1] = y; nf[3 * t + 2] = z; }
}

// Zeroes the requested maps, scatters the samples into them and pads the 8-bit ones in place.
static int bake_compose(const uint32_t *texels, size_t count, const uint8_t *rgba, const float *normal, int res,
                        int pad, uint8_t *bgra_out, uint8_t *normal_bgra_out, float *normal_out,
                        unsigned long long *d_empty, cudaStream_t s)
{
    const size_t n_pix = (size_t)res * res;
    if (bgra_out) PT_CUDA(cudaMemsetAsync(bgra_out, 0, 4 * n_pix, s));
    if (normal_bgra_out) PT_CUDA(cudaMemsetAsync(normal_bgra_out, 0, 4 * n_pix, s));
    if (normal_out) PT_CUDA(cudaMemsetAsync(normal_out, 0, sizeof(float) * 3 * n_pix, s));
    if (count) {
        bake_compose_kernel<<<tcdiv(count, 256), 256, 0, s>>>(texels, (uint32_t)count, rgba, normal, (uint32_t *)bgra_out,
                                                              (uint32_t *)normal_bgra_out, normal_out, d_empty);
        count_launch();
    }
    if (pad) PT_TRY(bake_pad({bgra_out, normal_bgra_out}, res, s));
    PT_CUDA(cudaGetLastError());
    return PT_OK;
}

// ---- tangent-space bake (DESIGN.md section 8, "Tangent-space bake") -----------------------------
// Everything below is fp64 with every operation rounded on its own (no contraction, no rsqrt), in
// the order the definition states, so that oracle/pt_bake_oracle.c equals it bit for bit:
// a.b = (a.x b.x + a.y b.y) + a.z b.z; "usable" = all components finite and a.a > 0; normalising
// divides each component by sqrt(a.a).  Mesh rows are 8 doubles: x y z u v nx ny nz.  Frame rows
// are 8 doubles: N xyz, T xyz, w, 0 -- all zero for a vertex without a frame.
constexpr int BAKE_ROW = 8;

struct D3 { double x, y, z; };

__device__ __forceinline__ D3 d3_add(D3 a, D3 b) { return {__dadd_rn(a.x, b.x), __dadd_rn(a.y, b.y), __dadd_rn(a.z, b.z)}; }
__device__ __forceinline__ D3 d3_sub(D3 a, D3 b) { return {__dsub_rn(a.x, b.x), __dsub_rn(a.y, b.y), __dsub_rn(a.z, b.z)}; }
__device__ __forceinline__ D3 d3_scale(double s, D3 a) { return {__dmul_rn(s, a.x), __dmul_rn(s, a.y), __dmul_rn(s, a.z)}; }
__device__ __forceinline__ double d3_dot(D3 a, D3 b)
{
    return __dadd_rn(__dadd_rn(__dmul_rn(a.x, b.x), __dmul_rn(a.y, b.y)), __dmul_rn(a.z, b.z));
}
__device__ __forceinline__ D3 d3_cross(D3 a, D3 b)
{
    return {__dsub_rn(__dmul_rn(a.y, b.z), __dmul_rn(a.z, b.y)), __dsub_rn(__dmul_rn(a.z, b.x), __dmul_rn(a.x, b.z)),
            __dsub_rn(__dmul_rn(a.x, b.y), __dmul_rn(a.y, b.x))};
}
__device__ __forceinline__ bool d3_finite(D3 a) { return isfinite(a.x) && isfinite(a.y) && isfinite(a.z); }
__device__ __forceinline__ bool d3_usable(D3 a) { return d3_finite(a) && d3_dot(a, a) > 0.0; }
__device__ __forceinline__ D3 d3_normalise(D3 a)
{
    const double l = __dsqrt_rn(d3_dot(a, a));
    return {__ddiv_rn(a.x, l), __ddiv_rn(a.y, l), __ddiv_rn(a.z, l)};
}
__device__ __forceinline__ D3 d3_load(const double *p) { return {p[0], p[1], p[2]}; }
// (b0 a + b1 b) + b2 c, per component
__device__ __forceinline__ D3 d3_mix(const double bc[3], D3 a, D3 b, D3 c)
{
    return d3_add(d3_add(d3_scale(bc[0], a), d3_scale(bc[1], b)), d3_scale(bc[2], c));
}
// the unit tangent of unit normal n from t: t - (n.t) n normalised, or the fallback F(n) -- the axis
// e_i with the smallest |n_i| (lowest i on ties), e_i - n_i n normalised
__device__ __forceinline__ D3 bake_tangent_dir(D3 n, D3 t)
{
    const D3 r = d3_sub(t, d3_scale(d3_dot(n, t), n));
    if (d3_usable(r)) return d3_normalise(r);
    const double ax = fabs(n.x), ay = fabs(n.y), az = fabs(n.z);
    const int i = (ax <= ay && ax <= az) ? 0 : (ay <= az ? 1 : 2);
    const double ni = i == 0 ? n.x : (i == 1 ? n.y : n.z);
    const D3 e = {i == 0 ? 1.0 : 0.0, i == 1 ? 1.0 : 0.0, i == 2 ? 1.0 : 0.0};
    return d3_normalise(d3_sub(e, d3_scale(ni, n)));
}

struct FaceFrame { D3 t, b, g; };

// T_f, B_f (both 0 when det == 0 or a component is not finite) and G_f = e1 x e2 of a face with
// valid corners; UV differences in UV units, independent of the resolution
__device__ __forceinline__ FaceFrame bake_face_frame(const double *const c[3])
{
    const D3 xa = d3_load(c[0]);
    const D3 e1 = d3_sub(d3_load(c[1]), xa), e2 = d3_sub(d3_load(c[2]), xa);
    const double du1 = __dsub_rn(c[1][3], c[0][3]), dv1 = __dsub_rn(c[1][4], c[0][4]);
    const double du2 = __dsub_rn(c[2][3], c[0][3]), dv2 = __dsub_rn(c[2][4], c[0][4]);
    const double det = __dsub_rn(__dmul_rn(du1, dv2), __dmul_rn(du2, dv1));
    const double r = __ddiv_rn(1.0, det);
    FaceFrame F;
    F.t = d3_scale(r, d3_sub(d3_scale(dv2, e1), d3_scale(dv1, e2)));
    F.b = d3_scale(r, d3_sub(d3_scale(du1, e2), d3_scale(du2, e1)));
    if (det == 0.0 || !d3_finite(F.t) || !d3_finite(F.b)) F.t = F.b = D3{0.0, 0.0, 0.0};
    F.g = d3_cross(e1, e2);
    return F;
}

// per face: T_f B_f G_f (9 doubles) and its three corner entries (vertex id, corner id 3f + j); a
// face with an out-of-range index pushes the key n_vertices, which sorts behind every vertex
__global__ void __launch_bounds__(256)
bake_face_frame_kernel(const BakeMesh M, double *face_tbg, uint32_t *corner_vertex, uint32_t *corner_id)
{
    const uint32_t f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= M.n_faces) return;
    const double *c[3];
    const bool ok = bake_corners(M, f, c);
    FaceFrame F = {};
    if (ok) F = bake_face_frame(c);
    double *o = face_tbg + 9 * (size_t)f;
    o[0] = F.t.x; o[1] = F.t.y; o[2] = F.t.z;
    o[3] = F.b.x; o[4] = F.b.y; o[5] = F.b.z;
    o[6] = F.g.x; o[7] = F.g.y; o[8] = F.g.z;
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        corner_vertex[3 * (size_t)f + j] = ok ? (uint32_t)M.faces[3 * (size_t)f + j] : M.n_vertices;
        corner_id[3 * (size_t)f + j] = 3u * f + (uint32_t)j;
    }
}

__device__ __forceinline__ uint32_t bake_lower_bound(const uint32_t *a, uint32_t n, uint32_t key)
{
    uint32_t lo = 0, hi = n;
    while (lo < hi) {
        const uint32_t mid = lo + ((hi - lo) >> 1);
        if (a[mid] < key) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// One thread per vertex: the sums over its corners in ascending corner id (= face order, then
// a, b, c: the sort is stable), then N, T and w.  No atomics, so the sums are the oracle's.
__global__ void __launch_bounds__(256)
bake_vertex_frame_kernel(const BakeMesh M, const double *face_tbg, const uint32_t *sorted_vertex,
                         const uint32_t *sorted_corner, uint32_t n_corners, double *frames, float *tangents)
{
    const uint32_t v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= M.n_vertices) return;
    const uint32_t lo = bake_lower_bound(sorted_vertex, n_corners, v);
    const uint32_t hi = bake_lower_bound(sorted_vertex, n_corners, v + 1u);
    D3 T = {0.0, 0.0, 0.0}, B = T, G = T;
    for (uint32_t i = lo; i < hi; ++i) {
        const double *fr = face_tbg + 9 * (size_t)(sorted_corner[i] / 3u);
        T = d3_add(T, d3_load(fr));
        B = d3_add(B, d3_load(fr + 3));
        G = d3_add(G, d3_load(fr + 6));
    }
    const D3 nv = d3_load(M.v + (size_t)v * M.stride + 5);
    double out[BAKE_ROW] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    if (d3_usable(nv) || d3_usable(G)) {
        const D3 N = d3_normalise(d3_usable(nv) ? nv : G);
        const D3 Th = bake_tangent_dir(N, T);
        const double w = d3_dot(d3_cross(N, Th), B) < 0.0 ? -1.0 : 1.0;
        out[0] = N.x; out[1] = N.y; out[2] = N.z;
        out[3] = Th.x; out[4] = Th.y; out[5] = Th.z;
        out[6] = w;
    }
#pragma unroll
    for (int j = 0; j < BAKE_ROW; ++j) frames[(size_t)v * BAKE_ROW + j] = out[j];
    if (tangents)
#pragma unroll
        for (int j = 0; j < 4; ++j) tangents[4 * (size_t)v + j] = (float)out[3 + j];
}

// Vertex frames of a mesh of rows of 8 doubles into frames (n_vertices x 8) and, when set,
// tangents (n_vertices x float4).  Needs 3 * n_faces <= INT_MAX (the sort's item count).
// Asynchronous on s.
static int bake_frames(const BakeMesh &M, double *frames, float *tangents, cudaStream_t s)
{
    if (!M.n_vertices) return PT_OK;
    const size_t n_corners = 3 * (size_t)M.n_faces;
    const size_t nc = n_corners ? n_corners : 1;
    double *d_tbg = nullptr;
    uint32_t *d_key = nullptr, *d_val = nullptr, *d_key_s = nullptr, *d_val_s = nullptr;
    void *d_tmp = nullptr;
    int rc = PT_OK;
    auto fail = [&](cudaError_t e) { if (e != cudaSuccess && rc == PT_OK) rc = map_cuda_error(e); return e != cudaSuccess; };
    do {
        // keys are vertex ids <= n_vertices (the sentinel): sort only the bits they use
        const int end_bit = 32 - __builtin_clz(M.n_vertices);
        size_t sort_bytes = 0;
        if (fail(cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, d_key, d_key_s, d_val, d_val_s, (int)nc, 0, end_bit, s)))
            break;
        if (pool_alloc((void **)&d_tbg, sizeof(double) * 9 * (M.n_faces ? M.n_faces : 1), s) ||
            pool_alloc((void **)&d_key, sizeof(uint32_t) * nc, s) || pool_alloc((void **)&d_val, sizeof(uint32_t) * nc, s) ||
            pool_alloc((void **)&d_key_s, sizeof(uint32_t) * nc, s) || pool_alloc((void **)&d_val_s, sizeof(uint32_t) * nc, s) ||
            pool_alloc(&d_tmp, sort_bytes ? sort_bytes : 1, s)) {
            rc = PT_ERR_OUT_OF_MEMORY;
            break;
        }
        if (M.n_faces) {
            bake_face_frame_kernel<<<tcdiv(M.n_faces, 256), 256, 0, s>>>(M, d_tbg, d_key, d_val);
            count_launch();
            if (fail(cub::DeviceRadixSort::SortPairs(d_tmp, sort_bytes, d_key, d_key_s, d_val, d_val_s, (int)n_corners, 0,
                                                     end_bit, s)))
                break;
            count_launch();
        }
        bake_vertex_frame_kernel<<<tcdiv(M.n_vertices, 256), 256, 0, s>>>(M, d_tbg, d_key_s, d_val_s, (uint32_t)n_corners,
                                                                        frames, tangents);
        count_launch();
        fail(cudaGetLastError());
    } while (0);
    void *frees[] = {d_tbg, d_key, d_val, d_key_s, d_val_s, d_tmp};
    for (void *p : frees) pool_free(p, s);
    return rc;
}

// What a sample of the tangent and height bakes needs of its texel: the owner face's corners, the
// barycentrics of the texel centre, the corners' vertex frame rows and the unit mesh normal N (the
// mixed N rows, normalised).  false when the sample is malformed or the mixed normal is not usable.
struct TexelFrame {
    const double *c[3];
    double        bc[3];
    const double *fr[3];
    D3            N;
};

__device__ __forceinline__ bool bake_texel_frame(const BakeMesh &M, const double *frames, uint32_t tex, int32_t f,
                                                 TexelFrame &X)
{
    if (f < 0 || (uint32_t)f >= M.n_faces || tex >= (uint32_t)M.res * (uint32_t)M.res || !bake_corners(M, (uint32_t)f, X.c))
        return false;
    bake_texel_bary(M, X.c, tex, X.bc);
#pragma unroll
    for (int j = 0; j < 3; ++j) X.fr[j] = frames + (size_t)M.faces[3 * (size_t)f + j] * BAKE_ROW;
    const D3 n = d3_mix(X.bc, d3_load(X.fr[0]), d3_load(X.fr[1]), d3_load(X.fr[2]));
    if (!d3_usable(n)) return false;
    X.N = d3_normalise(n);
    return true;
}

// One thread per sample: the texel's frame, its mixed tangent made orthonormal to N, the handedness
// of the owner face's B_f, and the blended cloud normal in that basis.  An empty neighbour list
// (alpha 0) or an unusable mixed normal leaves the texel 0.
__global__ void __launch_bounds__(256)
bake_tangent_compose_kernel(const BakeMesh M, const double *frames, const uint32_t *texels, const int32_t *sample_faces,
                            uint32_t count, const uint8_t *rgba, const float *normal, uint32_t *tbgra, float *tnf,
                            unsigned long long *empty)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    if (rgba[4 * (size_t)i + 3] == 0) {
        if (empty) atomicAdd(empty, 1ull);
        return;
    }
    const uint32_t tex = texels[i];
    TexelFrame X;
    if (!bake_texel_frame(M, frames, tex, sample_faces[i], X)) return;
    const D3 tm = d3_mix(X.bc, d3_load(X.fr[0] + 3), d3_load(X.fr[1] + 3), d3_load(X.fr[2] + 3));
    const D3 N = X.N;
    const D3 T = bake_tangent_dir(N, tm);
    const D3 x = d3_cross(N, T);
    const double w = d3_dot(x, bake_face_frame(X.c).b) < 0.0 ? -1.0 : 1.0;
    const D3 B = d3_scale(w, x);
    const D3 m = {(double)normal[3 * (size_t)i], (double)normal[3 * (size_t)i + 1], (double)normal[3 * (size_t)i + 2]};
    const float sx = (float)d3_dot(m, T), sy = (float)d3_dot(m, B), sz = (float)d3_dot(m, N);
    if (tbgra) tbgra[tex] = bake_encode(sz) | (bake_encode(sy) << 8) | (bake_encode(sx) << 16) | 0xff000000u;
    if (tnf) { tnf[3 * (size_t)tex] = sx; tnf[3 * (size_t)tex + 1] = sy; tnf[3 * (size_t)tex + 2] = sz; }
}

// Zeroes the requested tangent maps, composes the samples into them and pads the 8-bit one.
static int bake_compose_tangent(const BakeMesh &M, const double *frames, const uint32_t *texels,
                                const int32_t *sample_faces, size_t count, const uint8_t *rgba, const float *normal,
                                int pad, uint8_t *tbgra_out, float *tnormal_out, unsigned long long *d_empty,
                                cudaStream_t s)
{
    const size_t n_pix = (size_t)M.res * M.res;
    if (tbgra_out) PT_CUDA(cudaMemsetAsync(tbgra_out, 0, 4 * n_pix, s));
    if (tnormal_out) PT_CUDA(cudaMemsetAsync(tnormal_out, 0, sizeof(float) * 3 * n_pix, s));
    if (count) {
        bake_tangent_compose_kernel<<<tcdiv(count, 256), 256, 0, s>>>(M, frames, texels, sample_faces, (uint32_t)count, rgba,
                                                                     normal, (uint32_t *)tbgra_out, tnormal_out, d_empty);
        count_launch();
    }
    if (pad) PT_TRY(bake_pad({tbgra_out}, M.res, s));
    PT_CUDA(cudaGetLastError());
    return PT_OK;
}

// 80-byte Point records -> rows of 8 doubles (x y z u v nx ny nz), what the raster and the frames read
__global__ void __launch_bounds__(256) bake_unpack_vertices_kernel(const Raw80t *raw, uint32_t n, double *rows)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const Raw80t r = raw[i];
    double *o = rows + (size_t)i * BAKE_ROW;
    o[0] = r.ver[0]; o[1] = r.ver[1]; o[2] = r.ver[2];
    o[3] = r.U; o[4] = r.V;
    o[5] = r.normal[0]; o[6] = r.normal[1]; o[7] = r.normal[2];
}

// ---- height bake (DESIGN.md section 8, "Height bake") ---------------------------------------------
// h = (sum_j w_j ((p_j - x) . N)) / W over the sample's neighbour list: the blend's weights, the
// texel's unit mesh normal N of the tangent bake, sums sequential in neighbour order from +0.0.
// NaN (always the quiet NaN 0x7fc00000) is "no value".  Samples per launch of the query + height
// kernel in the bake: the neighbour lists of one chunk are 4 k bytes per sample.
constexpr uint32_t HEIGHT_CHUNK = 1u << 22;
constexpr uint32_t HEIGHT_NAN = 0x7fc00000u;

__device__ __forceinline__ double shfl_d(double v, int src) { return __shfl_sync(0xffffffffu, v, src); }

// A warp takes 32 consecutive samples.  First each lane computes the normal of one of them; then
// the warp walks them in `width` rounds, a group of `width` (the power of two >= k) lanes per
// sample: lane j of a group gathers neighbour j through the position source (independent random
// reads, in parallel), computes d2 in the metric's operation order and w_j (p_j - x).N, and the
// group adds the terms in neighbour order through shuffles.  Every lane runs the same loops, so
// the shuffles see the full warp.
template <typename POS>
__global__ void __launch_bounds__(256)
bake_height_kernel(const BakeMesh M, const double *frames, const uint32_t *texels, const int32_t *sample_faces,
                   const double *xyz, uint32_t count, const int32_t *idx, int k, int width, const POS pos,
                   uint32_t n_points, float *height)
{
    const unsigned lane = threadIdx.x & 31u;
    const uint32_t base = (uint32_t)(((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5) * 32u;
    if (base >= count) return;                                    // warp-uniform
    D3 myN = {0.0, 0.0, 0.0}, myX = myN;
    bool myOk = false;
    if (base + lane < count) {
        const uint32_t i = base + lane;
        TexelFrame X;
        myOk = bake_texel_frame(M, frames, texels[i], sample_faces[i], X);
        if (myOk) myN = X.N;
        myX = d3_load(xyz + 3 * (size_t)i);
    }
    const unsigned per_round = 32u / (unsigned)width;
    const unsigned g = lane / (unsigned)width, j = lane % (unsigned)width, g0 = g * (unsigned)width;
    for (unsigned r = 0; r < (unsigned)width; ++r) {
        const unsigned src = r * per_round + g;                    // < 32
        const D3 N = {shfl_d(myN.x, src), shfl_d(myN.y, src), shfl_d(myN.z, src)};
        const D3 x = {shfl_d(myX.x, src), shfl_d(myX.y, src), shfl_d(myX.z, src)};
        const bool ok = __shfl_sync(0xffffffffu, (int)myOk, src) != 0;
        const uint32_t s = base + src;
        bool has = false;
        double d2 = 0.0, o = 0.0;
        if (ok && s < count && (int)j < k) {
            const int id = idx[(size_t)s * k + j];
            if (id >= 0 && (uint32_t)id < n_points) {
                double p[3];
                pos.get(id, p);
                const D3 pj = {p[0], p[1], p[2]};
                d2 = dist2_exact(x.x, x.y, x.z, pj.x, pj.y, pj.z);
                o = d3_dot(d3_sub(pj, x), N);
                has = true;
            }
        }
        // the list is its leading run of valid entries
        const unsigned seg = (__ballot_sync(0xffffffffu, has) >> g0) & (width == 32 ? 0xffffffffu : ((1u << width) - 1u));
        const int cnt = __ffsll(~(unsigned long long)seg) - 1;
        int mode = shfl_d(d2, g0) == 0.0 ? 1 : 0;
        double W = 0.0, S = 0.0;
        bool done = cnt == 0;
        for (int pass = 0; pass < 2; ++pass) {
            if (!__any_sync(0xffffffffu, !done)) break;
            const double w = blend_weight(mode, d2, (int)j);
            const double wo = __dmul_rn(w, o);
            double w_sum = 0.0, s_sum = 0.0;
            for (int jj = 0; jj < k; ++jj) {
                const double wj = shfl_d(w, (int)g0 + jj), woj = shfl_d(wo, (int)g0 + jj);
                if (jj < cnt) {
                    w_sum = __dadd_rn(w_sum, wj);
                    s_sum = __dadd_rn(s_sum, woj);
                }
            }
            if (!done) {
                W = w_sum;
                S = s_sum;
                done = W > 0.0 && W < INFINITY;
            }
            mode = 2;
        }
        if (j == 0 && cnt > 0 && s < count) {
            const float h = __double2float_rn(__ddiv_rn(S, W));
            height[texels[s]] = h != h ? __uint_as_float(HEIGHT_NAN) : h;
        }
    }
}

__global__ void __launch_bounds__(256) bake_height_fill_kernel(float *h, size_t n)
{
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        h[i] = __uint_as_float(HEIGHT_NAN);
}

// float -> uint32 with the same order (-0 below +0)
__device__ __forceinline__ uint32_t height_key(float h)
{
    const uint32_t u = __float_as_uint(h);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float height_unkey(uint32_t k)
{
    return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

// mm[0] = min key, mm[1] = max key of the non-NaN heights (start 0xffffffff / 0), *valued (may be null)
// += their count
__global__ void __launch_bounds__(256)
bake_height_minmax_kernel(const float *h, size_t n, uint32_t *mm, unsigned long long *valued)
{
    uint32_t lo = 0xffffffffu, hi = 0u;
    unsigned long long c = 0;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const float v = h[i];
        if (v != v) continue;
        const uint32_t key = height_key(v);
        lo = min(lo, key);
        hi = max(hi, key);
        ++c;
    }
    for (int off = 16; off; off >>= 1) {
        lo = min(lo, __shfl_xor_sync(0xffffffffu, lo, off));
        hi = max(hi, __shfl_xor_sync(0xffffffffu, hi, off));
        c += __shfl_xor_sync(0xffffffffu, c, off);
    }
    if ((threadIdx.x & 31u) == 0 && c) {
        atomicMin(mm, lo);
        atomicMax(mm + 1, hi);
        if (valued) atomicAdd(valued, c);
    }
}

// the code range: the caller's when `fixed`, else the heights' min and max, (0, 0) without any
__global__ void bake_height_range_kernel(const uint32_t *mm, int fixed, double lo, double hi, double *range)
{
    if (!fixed) {
        const bool any = mm[0] <= mm[1];
        lo = any ? (double)height_unkey(mm[0]) : 0.0;
        hi = any ? (double)height_unkey(mm[1]) : 0.0;
    }
    range[0] = lo;
    range[1] = hi;
}

// E(h) = clamp(floor((h - lo) * s + 0.5), 0, 65535), s = 65535 / (hi - lo); 0 for every h when hi == lo
__device__ __forceinline__ uint32_t height_encode(float h, double lo, double hi)
{
    if (hi == lo) return 0u;
    const double s = __ddiv_rn(65535.0, __dsub_rn(hi, lo));
    const double e = floor(__dadd_rn(__dmul_rn(__dsub_rn((double)h, lo), s), 0.5));
    return (uint32_t)fmin(fmax(e, 0.0), 65535.0);
}

// Per texel: code16 = E(h), 0 without a value; or, for the padding, word = E(h) + 1, 0 without a value.
__global__ void __launch_bounds__(256)
bake_height_encode_kernel(const float *h, size_t n, const double *range, uint16_t *code16, uint32_t *word)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float v = h[i];
    const uint32_t e = v != v ? 0u : height_encode(v, range[0], range[1]) + 1u;
    if (code16) code16[i] = (uint16_t)(e ? e - 1u : 0u);
    if (word) word[i] = e;
}

static int bake_height_width(int k)
{
    int w = 1;
    while (w < k) w <<= 1;
    return w;
}

template <typename POS>
static int launch_height(const BakeMesh &M, const double *frames, const uint32_t *texels, const int32_t *sample_faces,
                         const double *xyz, size_t count, const int32_t *idx, int k, const POS &pos,
                         uint32_t n_points, float *height, cudaStream_t s)
{
    if (!count) return PT_OK;
    bake_height_kernel<POS><<<tcdiv(count, 256), 256, 0, s>>>(M, frames, texels, sample_faces, xyz, (uint32_t)count, idx, k,
                                                              bake_height_width(k), pos, n_points, height);
    count_launch();
    PT_CUDA(cudaGetLastError());
    return PT_OK;
}

static bool height_range_fixed(const double *r)
{
    return r && std::isfinite(r[0]) && std::isfinite(r[1]) && r[0] < r[1];
}

// From the float map: the code range into range_out (device, 2 doubles), the number of valued texels
// into *d_valued (device, added to; may be null) and, when code16 is set, the 16-bit map, padded when pad != 0.
static int bake_height_finish(const float *height, int res, int pad, const double *range_in, double *range_out,
                              uint16_t *code16, unsigned long long *d_valued, cudaStream_t s)
{
    const size_t n_pix = (size_t)res * res;
    uint32_t *d_mm = nullptr, *d_word = nullptr, *d_tmp = nullptr;
    int rc = PT_OK;
    auto fail = [&](cudaError_t e) { if (e != cudaSuccess && rc == PT_OK) rc = map_cuda_error(e); return e != cudaSuccess; };
    do {
        const bool padded = code16 && pad;
        if (pool_alloc((void **)&d_mm, 2 * sizeof(uint32_t), s) ||
            (padded && (pool_alloc((void **)&d_word, 4 * n_pix, s) || pool_alloc((void **)&d_tmp, 4 * n_pix, s)))) {
            rc = PT_ERR_OUT_OF_MEMORY;
            break;
        }
        if (fail(cudaMemsetAsync(d_mm, 0xff, sizeof(uint32_t), s)) || fail(cudaMemsetAsync(d_mm + 1, 0, sizeof(uint32_t), s)))
            break;
        bake_height_minmax_kernel<<<148 * 8, 256, 0, s>>>(height, n_pix, d_mm, d_valued);
        const bool fixed = height_range_fixed(range_in);
        bake_height_range_kernel<<<1, 1, 0, s>>>(d_mm, fixed ? 1 : 0, fixed ? range_in[0] : 0.0, fixed ? range_in[1] : 0.0,
                                                 range_out);
        count_launch(2);
        if (code16) {
            bake_height_encode_kernel<<<tcdiv(n_pix, 256), 256, 0, s>>>(height, n_pix, range_out, padded ? nullptr : code16,
                                                                        d_word);
            count_launch();
            if (padded) launch_pad_window<PadHeight>(d_word, d_tmp, res, code16, s);
        }
        fail(cudaGetLastError());
    } while (0);
    void *frees[] = {d_mm, d_word, d_tmp};
    for (void *p : frees) pool_free(p, s);
    return rc;
}

static bool bake_wants_tangent_maps(const pt_bake_outputs &o) { return o.tangent_bgra || o.tangent_normal; }
static bool bake_wants_frames(const pt_bake_outputs &o) { return bake_wants_tangent_maps(o) || o.vertex_tangents; }
static bool bake_wants_object_maps(const pt_bake_outputs &o) { return o.bgra || o.normal_bgra || o.normal; }
static bool bake_wants_height(const pt_bake_height *h) { return h && (h->height || h->height_u16); }

template <typename PT>
static int launch_height_index(pt_index *ix, const BakeMesh &M, const double *frames, const uint32_t *texels,
                               const int32_t *sample_faces, const double *xyz, size_t count, const int32_t *idx, int k,
                               float *height, cudaStream_t s)
{
    PT_TRY(index_inverse_perm<PT>(ix));
    const PosSorted<PT> pos{(const PT *)ix->pts, ix->inv_perm};
    return launch_height(M, frames, texels, sample_faces, xyz, count, idx, k, pos, ix->n, height, s);
}

static int texture_bake(pt_index *ix, const void *vertices, size_t n_vertices, const int32_t *faces, size_t n_faces,
                        int k, double radius, int res, int pad, const pt_bake_outputs &o, pt_bake_height *hb,
                        pt_bake_stats *st)
{
    cudaStream_t s = ix->stream;
    const size_t n_pix = (size_t)res * res;
    const bool heights = bake_wants_height(hb);
    const bool maps = bake_wants_object_maps(o) || bake_wants_tangent_maps(o) || heights;
    const bool tmaps = bake_wants_tangent_maps(o), frames = bake_wants_frames(o) || heights;
    Raw80t *d_raw = nullptr;
    double *d_rows = nullptr, *d_q = nullptr, *d_frames = nullptr, *d_range = nullptr;
    int32_t *d_faces = nullptr, *d_sface = nullptr, *d_idx = nullptr;
    uint32_t *d_texels = nullptr;
    uint8_t *d_rgba = nullptr, *d_bgra = nullptr, *d_nbgra = nullptr, *d_tbgra = nullptr;
    float *d_normal = nullptr, *d_nf = nullptr, *d_tnf = nullptr, *d_vt = nullptr, *d_height = nullptr;
    uint16_t *d_h16 = nullptr;
    unsigned long long *d_empty = nullptr;
    cudaEvent_t ev[4] = {};
    std::vector<cudaEvent_t> marks;                // around each query chunk when heights are baked
    size_t count = 0;
    int rc = PT_OK;
    auto fail = [&](cudaError_t e) { if (e != cudaSuccess && rc == PT_OK) rc = map_cuda_error(e); return e != cudaSuccess; };
    do {
        for (auto &e : ev) if (fail(cudaEventCreate(&e))) break;
        if (rc != PT_OK) break;
        if (pool_alloc((void **)&d_raw, sizeof(Raw80t) * n_vertices, s) ||
            pool_alloc((void **)&d_rows, sizeof(double) * BAKE_ROW * n_vertices, s) ||
            pool_alloc((void **)&d_faces, sizeof(int32_t) * 3 * n_faces, s) ||
            pool_alloc((void **)&d_empty, sizeof(unsigned long long) * (heights ? 2 : 1), s) ||
            (maps && (pool_alloc((void **)&d_texels, sizeof(uint32_t) * n_pix, s) ||
                      pool_alloc((void **)&d_q, sizeof(double) * 3 * n_pix, s))) ||
            ((tmaps || heights) && pool_alloc((void **)&d_sface, sizeof(int32_t) * n_pix, s)) ||
            (heights && (pool_alloc((void **)&d_height, sizeof(float) * n_pix, s) ||
                         pool_alloc((void **)&d_range, 2 * sizeof(double), s))) ||
            (heights && hb->height_u16 && pool_alloc((void **)&d_h16, sizeof(uint16_t) * n_pix, s)) ||
            (frames && pool_alloc((void **)&d_frames, sizeof(double) * BAKE_ROW * n_vertices, s)) ||
            (o.bgra && pool_alloc((void **)&d_bgra, 4 * n_pix, s)) ||
            (o.normal_bgra && pool_alloc((void **)&d_nbgra, 4 * n_pix, s)) ||
            (o.normal && pool_alloc((void **)&d_nf, sizeof(float) * 3 * n_pix, s)) ||
            (o.tangent_bgra && pool_alloc((void **)&d_tbgra, 4 * n_pix, s)) ||
            (o.tangent_normal && pool_alloc((void **)&d_tnf, sizeof(float) * 3 * n_pix, s)) ||
            (o.vertex_tangents && pool_alloc((void **)&d_vt, sizeof(float) * 4 * n_vertices, s))) {
            rc = PT_ERR_OUT_OF_MEMORY;
            break;
        }
        if (fail(cudaEventRecord(ev[0], s))) break;
        if (fail(cudaMemcpyAsync(d_raw, vertices, sizeof(Raw80t) * n_vertices, cudaMemcpyHostToDevice, s))) break;
        if (fail(cudaMemcpyAsync(d_faces, faces, sizeof(int32_t) * 3 * n_faces, cudaMemcpyHostToDevice, s))) break;
        if (fail(cudaMemsetAsync(d_empty, 0, sizeof(unsigned long long), s))) break;
        if (n_vertices) {
            bake_unpack_vertices_kernel<<<tcdiv(n_vertices, 256), 256, 0, s>>>(d_raw, (uint32_t)n_vertices, d_rows);
            count_launch();
        }
        const BakeMesh M{d_rows, BAKE_ROW, (uint32_t)n_vertices, d_faces, (uint32_t)n_faces, res};
        if (maps && (rc = bake_texels(M, d_texels, d_q, d_sface, &count, s)) != PT_OK) break;
        if (frames && (rc = bake_frames(M, d_frames, d_vt, s)) != PT_OK) break;
        if (fail(cudaEventRecord(ev[1], s))) break;
        // heights need the neighbour lists: the query and the height kernel then run in chunks, so
        // the lists take at most HEIGHT_CHUNK * k * 4 bytes
        const size_t chunk = heights ? HEIGHT_CHUNK : (count ? count : 1);
        if (pool_alloc((void **)&d_rgba, 4 * (count ? count : 1), s) || pool_alloc((void **)&d_normal, sizeof(float) * 3 * (count ? count : 1), s) ||
            (heights && pool_alloc((void **)&d_idx, sizeof(int32_t) * k * std::min(chunk, count ? count : 1), s))) {
            rc = PT_ERR_OUT_OF_MEMORY;
            break;
        }
        if (heights) {
            bake_height_fill_kernel<<<148 * 8, 256, 0, s>>>(d_height, n_pix);
            count_launch();
        }
        QueryParams qp{};
        fill_params(ix, qp);
        qp.k = k;
        qp.r2 = radius_to_r2(radius);
        for (size_t c0 = 0; c0 < count; c0 += chunk) {
            const size_t cm = std::min(chunk, count - c0);
            if (heights) {
                marks.emplace_back();
                if (fail(cudaEventCreate(&marks.back())) || fail(cudaEventRecord(marks.back(), s))) break;
            }
            qp.queries = d_q + 3 * c0; qp.m = (uint32_t)cm;
            qp.rgba_out = d_rgba + 4 * c0; qp.normal_out = d_normal + 3 * c0;
            qp.idx_out = d_idx;
            if ((rc = launch_query(ix, qp, s)) != PT_OK) break;
            if (!heights) continue;
            marks.emplace_back();
            if (fail(cudaEventCreate(&marks.back())) || fail(cudaEventRecord(marks.back(), s))) break;
            rc = ix->coord_f64 ? launch_height_index<PointD>(ix, M, d_frames, d_texels + c0, d_sface + c0, d_q + 3 * c0, cm,
                                                             d_idx, k, d_height, s)
                               : launch_height_index<PointF>(ix, M, d_frames, d_texels + c0, d_sface + c0, d_q + 3 * c0, cm,
                                                             d_idx, k, d_height, s);
            if (rc != PT_OK) break;
        }
        if (rc != PT_OK) break;
        if (fail(cudaEventRecord(ev[2], s))) break;
        if (bake_wants_object_maps(o) &&
            (rc = bake_compose(d_texels, count, d_rgba, d_normal, res, pad, d_bgra, d_nbgra, d_nf, d_empty, s)) != PT_OK)
            break;
        // the empty lists are counted by whichever composition runs
        if (tmaps && (rc = bake_compose_tangent(M, d_frames, d_texels, d_sface, count, d_rgba, d_normal, pad, d_tbgra,
                                                d_tnf, bake_wants_object_maps(o) ? nullptr : d_empty, s)) != PT_OK)
            break;
        if (heights) {
            if (fail(cudaMemsetAsync(d_empty + 1, 0, sizeof(unsigned long long), s))) break;
            if ((rc = bake_height_finish(d_height, res, pad, hb->range, d_range, d_h16, d_empty + 1, s)) != PT_OK) break;
        }
        if (fail(cudaEventRecord(ev[3], s))) break;
        if (o.bgra && fail(cudaMemcpyAsync(o.bgra, d_bgra, 4 * n_pix, cudaMemcpyDeviceToHost, s))) break;
        if (o.normal_bgra && fail(cudaMemcpyAsync(o.normal_bgra, d_nbgra, 4 * n_pix, cudaMemcpyDeviceToHost, s))) break;
        if (o.normal && fail(cudaMemcpyAsync(o.normal, d_nf, sizeof(float) * 3 * n_pix, cudaMemcpyDeviceToHost, s))) break;
        if (o.tangent_bgra && fail(cudaMemcpyAsync(o.tangent_bgra, d_tbgra, 4 * n_pix, cudaMemcpyDeviceToHost, s))) break;
        if (o.tangent_normal &&
            fail(cudaMemcpyAsync(o.tangent_normal, d_tnf, sizeof(float) * 3 * n_pix, cudaMemcpyDeviceToHost, s)))
            break;
        if (o.vertex_tangents && n_vertices &&
            fail(cudaMemcpyAsync(o.vertex_tangents, d_vt, sizeof(float) * 4 * n_vertices, cudaMemcpyDeviceToHost, s)))
            break;
        if (heights) {
            if (hb->height && fail(cudaMemcpyAsync(hb->height, d_height, sizeof(float) * n_pix, cudaMemcpyDeviceToHost, s)))
                break;
            if (hb->height_u16 &&
                fail(cudaMemcpyAsync(hb->height_u16, d_h16, sizeof(uint16_t) * n_pix, cudaMemcpyDeviceToHost, s)))
                break;
            if (fail(cudaMemcpyAsync(hb->range_used, d_range, 2 * sizeof(double), cudaMemcpyDeviceToHost, s))) break;
        }
        unsigned long long empty[2] = {0, 0};
        if (fail(cudaMemcpyAsync(empty, d_empty, sizeof(unsigned long long) * (heights ? 2 : 1), cudaMemcpyDeviceToHost, s)))
            break;
        if (fail(cudaStreamSynchronize(s))) break;
        if (heights) hb->texels = empty[1];
        if (st) {
            st->texels = count;
            st->empty = empty[0];
            cudaEventElapsedTime(&st->raster_ms, ev[0], ev[1]);
            cudaEventElapsedTime(&st->knn_ms, ev[1], ev[2]);
            cudaEventElapsedTime(&st->pad_ms, ev[2], ev[3]);
            if (heights) {                         // the height kernels between the query chunks count as pad_ms
                float knn = 0.0f, t = 0.0f;
                for (size_t c = 0; c + 1 < marks.size(); c += 2)
                    if (cudaEventElapsedTime(&t, marks[c], marks[c + 1]) == cudaSuccess) knn += t;
                st->pad_ms += st->knn_ms - knn;
                st->knn_ms = knn;
            }
        }
    } while (0);
    cudaStreamSynchronize(s);
    void *frees[] = {d_raw, d_rows, d_faces, d_texels, d_q, d_sface, d_frames, d_rgba, d_normal, d_bgra, d_nbgra, d_nf,
                     d_tbgra, d_tnf, d_vt, d_empty, d_idx, d_height, d_range, d_h16};
    for (void *p : frees) pool_free(p, s);
    for (auto &e : ev) if (e) cudaEventDestroy(e);
    for (auto &e : marks) if (e) cudaEventDestroy(e);
    cudaStreamSynchronize(s);
    cudaGetLastError();
    return rc;
}

}  // namespace pt

using namespace pt;

extern "C" int pt_texture_render(pt_index *ix, const void *vertices, size_t n_vertices, const int32_t *faces,
                                 size_t n_faces, int k, double radius, int resolution, int pad,
                                 uint8_t *bgra_out, pt_texture_stats *stats)
{
    if (!ix || (!vertices && n_vertices) || (!faces && n_faces) || !bgra_out || resolution < 1 || resolution > 32768 ||
        n_vertices > 0x7ffffff0ull || n_faces >= (1ull << 24))
        return PT_ERR_INVALID_ARG;
    if (k < 1 || k > PT_MAX_K) return PT_ERR_UNSUPPORTED;
    if (ix->ids) return PT_ERR_UNSUPPORTED;           // slab indexes answer with global ids
    if (!ix->attrs && ix->n) return PT_ERR_INVALID_ARG;
    PT_CUDA(cudaSetDevice(ix->device));
    return ix->coord_f64 ? texture_render_index<PointD>(ix, vertices, n_vertices, faces, n_faces, k, radius, resolution, pad, bgra_out, stats)
                         : texture_render_index<PointF>(ix, vertices, n_vertices, faces, n_faces, k, radius, resolution, pad, bgra_out, stats);
}

extern "C" int pt_texture_render_lists(const void *points, size_t n, const void *vertices, size_t n_vertices,
                                       const int32_t *faces, size_t n_faces, const int32_t *idx, int k,
                                       int resolution, int pad, int device, uint8_t *bgra_out,
                                       pt_texture_stats *stats)
{
    if ((!points && n) || (!vertices && n_vertices) || (!faces && n_faces) || (!idx && n_vertices) || !bgra_out ||
        resolution < 1 || resolution > 32768 || n >= 0x7fffffffull || n_vertices > 0x7ffffff0ull || n_faces >= (1ull << 24))
        return PT_ERR_INVALID_ARG;
    if (k < 1 || k > PT_MAX_K) return PT_ERR_UNSUPPORTED;
    if (pt_device_count() == 0) return PT_ERR_NO_DEVICE;
    if (device < 0) PT_CUDA(cudaGetDevice(&device));
    PT_CUDA(cudaSetDevice(device));
    // a bare handle: a stream plus the cloud's positions and attributes in original order
    pt_index tmp;
    tmp.device = device;
    double *xyz = nullptr;
    bool representable = true;
    int rc = map_cuda_error(cudaStreamCreateWithFlags(&tmp.stream, cudaStreamNonBlocking));
    if (rc == PT_OK) rc = ingest_points_aos(&tmp, points, n, PT_COORD_AUTO, &xyz, &representable);
    if (rc == PT_OK) {
        PosPlain pos{xyz};
        rc = texture_pipeline(&tmp, pos, (uint32_t)n, tmp.attrs, false, idx, vertices, n_vertices, faces, n_faces, k,
                              -1.0, resolution, pad, bgra_out, stats);
    }
    if (tmp.stream) cudaStreamSynchronize(tmp.stream);
    dev_free(xyz);
    pool_free(tmp.attrs, tmp.stream);
    if (tmp.stream) cudaStreamSynchronize(tmp.stream);
    if (tmp.stream) cudaStreamDestroy(tmp.stream);
    cudaGetLastError();
    return rc;
}

extern "C" int pt_bake_samples_device(const double *vertices_xyzuv, size_t n_vertices, const int32_t *faces,
                                      size_t n_faces, int resolution, uint32_t *texel_out, double *xyz_out,
                                      int32_t *face_out, size_t *count_out, int device, void *stream)
{
    if ((!vertices_xyzuv && n_vertices) || (!faces && n_faces) || !count_out || resolution < 1 || resolution > 16384 ||
        n_vertices > 0x7ffffff0ull || n_faces >= (1ull << 31) || (!texel_out != !xyz_out) || (face_out && !texel_out))
        return PT_ERR_INVALID_ARG;
    *count_out = 0;
    if (pt_device_count() == 0) return PT_ERR_NO_DEVICE;
    if (device >= 0) PT_CUDA(cudaSetDevice(device));
    const BakeMesh M{vertices_xyzuv, 5, (uint32_t)n_vertices, faces, (uint32_t)n_faces, resolution};
    return bake_texels(M, texel_out, xyz_out, face_out, count_out, (cudaStream_t)stream);
}

extern "C" int pt_bake_texels_device(const double *vertices_xyzuv, size_t n_vertices, const int32_t *faces,
                                     size_t n_faces, int resolution, uint32_t *texel_out, double *xyz_out,
                                     size_t *count_out, int device, void *stream)
{
    return pt_bake_samples_device(vertices_xyzuv, n_vertices, faces, n_faces, resolution, texel_out, xyz_out, nullptr,
                                  count_out, device, stream);
}

// the corner list of the frames is sorted with an int item count
static bool bake_corners_fit(size_t n_faces) { return n_faces <= (size_t)INT32_MAX / 3; }

extern "C" int pt_bake_frames_device(const double *vertices_xyzuvn, size_t n_vertices, const int32_t *faces,
                                     size_t n_faces, double *frames_out, float *tangents_out, int device, void *stream)
{
    if ((!vertices_xyzuvn && n_vertices) || (!faces && n_faces) || (!frames_out && n_vertices) ||
        n_vertices > 0x7ffffff0ull)
        return PT_ERR_INVALID_ARG;
    if (!bake_corners_fit(n_faces)) return PT_ERR_UNSUPPORTED;
    if (pt_device_count() == 0) return PT_ERR_NO_DEVICE;
    if (device >= 0) PT_CUDA(cudaSetDevice(device));
    const BakeMesh M{vertices_xyzuvn, BAKE_ROW, (uint32_t)n_vertices, faces, (uint32_t)n_faces, 1};
    return bake_frames(M, frames_out, tangents_out, (cudaStream_t)stream);
}

extern "C" int pt_bake_compose_tangent_device(const double *vertices_xyzuvn, const double *frames, size_t n_vertices,
                                              const int32_t *faces, size_t n_faces, const uint32_t *texels,
                                              const int32_t *sample_faces, size_t count, const uint8_t *rgba,
                                              const float *normal, int resolution, int pad, uint8_t *tangent_bgra_out,
                                              float *tangent_normal_out, int device, void *stream)
{
    if ((n_vertices && (!vertices_xyzuvn || !frames)) || (!faces && n_faces) ||
        (count && (!texels || !sample_faces || !rgba || !normal)) || resolution < 1 || resolution > 16384 ||
        count > (size_t)resolution * resolution || n_vertices > 0x7ffffff0ull || n_faces >= (1ull << 31) ||
        (!tangent_bgra_out && !tangent_normal_out))
        return PT_ERR_INVALID_ARG;
    if (pt_device_count() == 0) return PT_ERR_NO_DEVICE;
    if (device >= 0) PT_CUDA(cudaSetDevice(device));
    const BakeMesh M{vertices_xyzuvn, BAKE_ROW, (uint32_t)n_vertices, faces, (uint32_t)n_faces, resolution};
    return bake_compose_tangent(M, frames, texels, sample_faces, count, rgba, normal, pad, tangent_bgra_out,
                                tangent_normal_out, nullptr, (cudaStream_t)stream);
}

extern "C" int pt_bake_compose_device(const uint32_t *texels, size_t count, const uint8_t *rgba, const float *normal,
                                      int resolution, int pad, uint8_t *bgra_out, uint8_t *normal_bgra_out,
                                      float *normal_out, int device, void *stream)
{
    if ((count && (!texels || !rgba || !normal)) || resolution < 1 || resolution > 16384 ||
        count > (size_t)resolution * resolution || (!bgra_out && !normal_bgra_out && !normal_out))
        return PT_ERR_INVALID_ARG;
    if (pt_device_count() == 0) return PT_ERR_NO_DEVICE;
    if (device >= 0) PT_CUDA(cudaSetDevice(device));
    return bake_compose(texels, count, rgba, normal, resolution, pad, bgra_out, normal_bgra_out, normal_out, nullptr,
                        (cudaStream_t)stream);
}

extern "C" int pt_texture_bake_height(pt_index *ix, const void *vertices, size_t n_vertices, const int32_t *faces,
                                      size_t n_faces, int k, double radius, int resolution, int pad,
                                      const pt_bake_outputs *out, pt_bake_height *height, pt_bake_stats *stats)
{
    const pt_bake_outputs none = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    const pt_bake_outputs &o = out ? *out : none;
    const bool heights = bake_wants_height(height);
    if (!ix || (!vertices && n_vertices) || (!faces && n_faces) || (height && !heights) ||
        (!bake_wants_object_maps(o) && !bake_wants_frames(o) && !heights) || resolution < 1 || resolution > 16384 ||
        n_vertices > 0x7ffffff0ull || n_faces >= (1ull << 31))
        return PT_ERR_INVALID_ARG;
    if (k < 1 || k > PT_MAX_K) return PT_ERR_UNSUPPORTED;
    if ((bake_wants_frames(o) || heights) && !bake_corners_fit(n_faces)) return PT_ERR_UNSUPPORTED;
    if (ix->ids) return PT_ERR_UNSUPPORTED;           // slab indexes answer with global ids
    if (!ix->attrs && ix->n) return PT_ERR_INVALID_ARG;
    if (pt_device_count() == 0) return PT_ERR_NO_DEVICE;
    PT_CUDA(cudaSetDevice(ix->device));
    return texture_bake(ix, vertices, n_vertices, faces, n_faces, k, radius, resolution, pad, o, height, stats);
}

extern "C" int pt_texture_bake_ex(pt_index *ix, const void *vertices, size_t n_vertices, const int32_t *faces,
                                  size_t n_faces, int k, double radius, int resolution, int pad,
                                  const pt_bake_outputs *out, pt_bake_stats *stats)
{
    if (!out) return PT_ERR_INVALID_ARG;
    return pt_texture_bake_height(ix, vertices, n_vertices, faces, n_faces, k, radius, resolution, pad, out, nullptr,
                                  stats);
}

extern "C" int pt_bake_compose_height_device(const double *vertices_xyzuvn, const double *frames, size_t n_vertices,
                                             const int32_t *faces, size_t n_faces, const uint32_t *texels,
                                             const int32_t *sample_faces, const double *sample_xyz, size_t count,
                                             const int32_t *idx, int k, const double *cloud_xyz, size_t n_points,
                                             int resolution, int pad, const double *range_in, float *height_out,
                                             uint16_t *height_u16_out, double *range_out, int device, void *stream)
{
    if ((n_vertices && (!vertices_xyzuvn || !frames)) || (!faces && n_faces) ||
        (count && (!texels || !sample_faces || !sample_xyz || !idx)) || (!cloud_xyz && n_points) || resolution < 1 ||
        resolution > 16384 || count > (size_t)resolution * resolution || n_vertices > 0x7ffffff0ull ||
        n_faces >= (1ull << 31) || n_points > (size_t)INT32_MAX || (!height_out && !height_u16_out))
        return PT_ERR_INVALID_ARG;
    if (k < 1 || k > PT_MAX_K || !bake_corners_fit(n_faces)) return PT_ERR_UNSUPPORTED;
    if (pt_device_count() == 0) return PT_ERR_NO_DEVICE;
    if (device >= 0) PT_CUDA(cudaSetDevice(device));
    cudaStream_t s = (cudaStream_t)stream;
    const size_t n_pix = (size_t)resolution * resolution;
    const BakeMesh M{vertices_xyzuvn, BAKE_ROW, (uint32_t)n_vertices, faces, (uint32_t)n_faces, resolution};
    float *h = height_out;
    double *range = range_out;
    int rc = PT_OK;
    do {
        if ((!h && (rc = pool_alloc((void **)&h, sizeof(float) * n_pix, s)) != PT_OK) ||
            (!range && (rc = pool_alloc((void **)&range, 2 * sizeof(double), s)) != PT_OK))
            break;
        bake_height_fill_kernel<<<148 * 8, 256, 0, s>>>(h, n_pix);
        count_launch();
        if ((rc = launch_height(M, frames, texels, sample_faces, sample_xyz, count, idx, k, PosPlain{cloud_xyz},
                                (uint32_t)n_points, h, s)) != PT_OK)
            break;
        rc = bake_height_finish(h, resolution, pad, range_in, range, height_u16_out, nullptr, s);
    } while (0);
    if (h != height_out) pool_free(h, s);
    if (range != range_out) pool_free(range, s);
    return rc;
}

extern "C" int pt_texture_bake(pt_index *ix, const void *vertices, size_t n_vertices, const int32_t *faces,
                               size_t n_faces, int k, double radius, int resolution, int pad, uint8_t *bgra_out,
                               uint8_t *normal_bgra_out, float *normal_out, pt_bake_stats *stats)
{
    const pt_bake_outputs out = {bgra_out, normal_bgra_out, normal_out, nullptr, nullptr, nullptr};
    return pt_texture_bake_ex(ix, vertices, n_vertices, faces, n_faces, k, radius, resolution, pad, &out, stats);
}

/*
 * points_transfer.h -- C ABI of the B200-native pointsTransfer hot path.
 *
 * This is the drop-in boundary.  Each entry point replaces one call site of
 * the reference (horizon-research/3D-Reconstruction-From-Point-Cloud, paths
 * relative to its root):
 *
 *   pt_index_build   <- `Tree tree(points.begin(), points.end());`
 *                       src/pointsTransfer.cpp:259 (typedefs :37-40); the lazy
 *                       CGAL kd-tree build hidden in the first query as well.
 *   pt_knn           <- `K_neighbor_search search(tree, q, K);` + the result
 *                       iteration, src/pointsTransfer.cpp:474-478, metric
 *                       src/Distance.h:6-11, radius transform src/Distance.h:97.
 *   pt_transfer      <- the per-sample transfer loop src/pointsTransfer.cpp:
 *                       465-479 + the colour blend semantics of :95-103.
 *   pt_texture_render<- the face loop body after the searches and the texture
 *                       post-process, src/pointsTransfer.cpp:484-611 + draw_triangle :66-107.
 *   pt_texture_bake  <- no reference counterpart: per-texel colour and normal maps on
 *                       the mesh's UV atlas (the "texel" samples of the transfer);
 *                       pt_texture_bake_ex adds tangent-space normal maps and the
 *                       per-vertex tangents they are expressed in, pt_texture_bake_height
 *                       height (displacement) maps.
 *   pt_index_free    <- `tree` going out of scope at src/pointsTransfer.cpp:626.
 *
 * Records are the reference's own 80-byte AoS `struct Point`
 * (src/Point.h:1-6): double ver[3] @0, double normal[3] @24, int color[3] @48,
 * double U @64, double V @72.  They are passed as `const void*` so a caller can
 * hand over `points.data()` of its `std::vector<Point>` unchanged.
 *
 * Contract (SURVEY.md section 8 row B4): plain pointers and sizes only; int
 * status returned (0 = ok), nothing thrown across the ABI; blocking -- every
 * call is stream-synchronised on return; one handle <-> one caller thread at a
 * time (thread-compatible); results in query order; neighbours in ascending
 * (d2, index) order, ties broken by lowest point index; short lists padded with
 * index -1 / d2 +inf.  There is NO CPU fallback: without a CUDA device every
 * compute entry point returns PT_ERR_NO_DEVICE.
 */
#ifndef POINTS_TRANSFER_H
#define POINTS_TRANSFER_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PT_OK                 0
#define PT_ERR_INVALID_ARG    1
#define PT_ERR_CUDA           2
#define PT_ERR_NO_DEVICE      3
#define PT_ERR_OUT_OF_MEMORY  4
#define PT_ERR_UNSUPPORTED    5  /* e.g. k > PT_MAX_K */
#define PT_ERR_NOT_REPRESENTABLE 6 /* coord_mode = PT_COORD_F32 but input is not fp32-exact */
#define PT_ERR_NON_FINITE     7  /* NaN/inf coordinate in the cloud */

#define PT_MAX_K 32
#define PT_POINT_STRIDE 80 /* sizeof(struct Point), src/Point.h */

/* Coordinate storage of the index.  The metric is always evaluated in fp64 in
 * the reference's operation order (src/Distance.h:6-11).  F32 storage (16-byte
 * float4 records) is lossless only when every cloud coordinate is exactly
 * representable in fp32; AUTO checks that on the device and falls back to the
 * 32-byte fp64 records otherwise, so neighbour indices stay bit-exact. */
#define PT_COORD_AUTO 0
#define PT_COORD_F32  1
#define PT_COORD_F64  2

typedef struct pt_index pt_index; /* opaque; owns device memory + one stream */

typedef struct pt_build_opts {
    int device;            /* CUDA ordinal; -1 = current device */
    int coord_mode;        /* PT_COORD_* */
    const int32_t *ids;    /* optional n global point ids, strictly increasing
                              (slab of a sharded cloud); NULL => 0..n-1 */
    int reserved[8];       /* must be zero */
} pt_build_opts;

typedef struct pt_index_info {
    uint64_t n_points;
    uint64_t n_leaves;       /* 32-point buckets of the curve-sorted cloud */
    int      n_levels;       /* box-pyramid levels */
    int      coord_mode;     /* PT_COORD_F32 or PT_COORD_F64 actually used */
    int      device;
    int      last_fallback_samples; /* samples the last query launch handed to the exact warp
                                       kernel (queue proof obligation not met); -1 unknown */
    double   bbox_lo[3], bbox_hi[3];
    uint64_t device_bytes;   /* resident after the build */
    float    build_ms;       /* device time of the last build (CUDA events) */
    float    last_query_ms;  /* device time of the last pt_knn/pt_transfer call: the chunked
                                H2D copy, kernels and D2H copy are pipelined over 3 streams */
    float    last_h2d_ms, last_d2h_ms; /* 0: overlapped, not separately measurable */
} pt_index_info;

/* Library / device probing (no compute). */
const char *pt_version(void);
const char *pt_status_string(int status);
int         pt_device_count(void); /* 0 when no CUDA device/driver */

/* Host-buffer API: the reference-facing plugin surface. ------------------- */

int pt_index_build(const void *points, size_t n, const pt_build_opts *opts,
                   pt_index **out);
int pt_index_free(pt_index *index);
int pt_index_get_info(const pt_index *index, pt_index_info *info);

/* Diagnostics of the last query launch on this index (synchronises the device):
 * out2[0] = samples re-run by the exact warp kernel (= last_fallback_samples),
 * out2[1] = samples the grid kernel handed to the box-pyramid kernels. */
int pt_index_fallback_counts(const pt_index *index, uint32_t out2[2]);

/* radius < 0 or +inf: unbounded k-NN (the reference's mode).  Otherwise only
 * points with d2 <= Distance::transformed_distance(radius) (src/Distance.h:97).
 * idx_out[m*k] (int32), d2_out[m*k] (double, may be NULL). */
int pt_knn(pt_index *index, const void *queries, size_t m, int k, double radius,
           int32_t *idx_out, double *d2_out);

/* k-NN + fused distance-weighted colour/normal blend (DESIGN.md "blend").
 * idx_out / d2_out may be NULL; rgba_out[m*4] (r,g,b,255), normal_out[m*3]. */
int pt_transfer(pt_index *index, const void *queries, size_t m, int k,
                double radius, int32_t *idx_out, double *d2_out,
                uint8_t *rgba_out, float *normal_out);

/* Everything the reference does after the neighbour search, for a whole mesh
 * (src/pointsTransfer.cpp:462-611): per face the union of the K nearest cloud points of its
 * corners, projection onto the face plane + in-triangle filter (:484-537), Delaunay
 * sub-triangulation with barycentric UVs (:539-581), rasterisation of every sub-triangle with
 * interpolated colours (draw_triangle, :66-107) and, with pad != 0, the 25x25 dilate + gutter
 * (:593-611).  vertices: n_vertices Point records (position, U, V, colour are read); faces:
 * 3 int32 vertex indices per face (n_faces < 2^24); bgra_out: resolution * resolution * 4 bytes
 * in HOST memory, row 0 first, byte order B G R A as cv::Mat CV_8UC4 -- what the reference hands
 * to cv::imwrite("texture.png").  Pixels nobody draws are 0 (the reference leaves them
 * uninitialised); the reference's out-of-bounds row / column writes are skipped. */
typedef struct pt_texture_stats {
    uint64_t triangles;      /* sub-triangles drawn */
    uint64_t inside_points;  /* neighbours kept by the in-triangle filter, all faces */
    float    knn_ms, draw_ms, pad_ms;   /* device time of the three stages */
} pt_texture_stats;
int pt_texture_render(pt_index *index, const void *vertices, size_t n_vertices,
                      const int32_t *faces, size_t n_faces, int k, double radius,
                      int resolution, int pad, uint8_t *bgra_out, pt_texture_stats *stats);

/* Per-texel bake (DESIGN.md section 8, "Per-texel bake"): every texel of the mesh's UV atlas that
 * a face covers becomes one sample, answered by the k-NN + fused blend of pt_transfer, and the
 * results are written back as images.  Texel (col, row) of a resolution x resolution image (row 0
 * on top) samples the UV point ((col + 0.5) / res, (res - row - 0.5) / res): the texel-centre
 * convention of standard texture sampling, half a texel away from pt_texture_render's lattice.
 * A face covers a texel when the barycentrics of that point in its UV triangle are all >= 0;
 * where faces overlap the highest face index wins; degenerate UV triangles and faces with an
 * out-of-range vertex index cover nothing.  The sample position is the fp64 barycentric mix of
 * the winning face's 3-D corners.
 *   bgra_out         blended colour as B G R 255 (cv::Mat CV_8UC4 layout)
 *   normal_bgra_out  object-space normal map: B G R A = e(z) e(y) e(x) 255 with
 *                    e(n) = clamp(floor((n + 1) * 127.5 + 0.5), 0, 255), so RGB shows xyz
 *   normal_out       the blended unit normal, 3 floats per texel
 * Uncovered texels, and covered texels whose neighbour list is empty (radius-bounded search),
 * are 0 in all three maps.  pad != 0 runs the two 8-bit maps through the texture's 25 x 25
 * dilate + gutter; normal_out is never padded.  Host buffers, blocking.  vertices: Point records
 * (position, U, V are read); faces: 3 int32 per face (n_faces < 2^31).  Any of the three outputs
 * may be NULL, but not all.  resolution 1..16384. */
typedef struct pt_bake_stats {
    uint64_t texels;   /* covered texels = samples answered */
    uint64_t empty;    /* covered texels whose neighbour list came back empty */
    float    raster_ms, knn_ms, pad_ms;   /* device time of the stages: upload + raster + compaction,
                                             k-NN + blend, scatter into the maps + padding */
} pt_bake_stats;
int pt_texture_bake(pt_index *index, const void *vertices, size_t n_vertices,
                    const int32_t *faces, size_t n_faces, int k, double radius,
                    int resolution, int pad, uint8_t *bgra_out /* res*res*4 */,
                    uint8_t *normal_bgra_out /* res*res*4 */, float *normal_out /* res*res*3 */,
                    pt_bake_stats *stats);

/* Tangent-space bake (DESIGN.md section 8, "Tangent-space bake").  pt_texture_bake_ex runs one
 * texel raster and one k-NN pass for every requested output:
 *   bgra, normal_bgra, normal  as pt_texture_bake (res*res*4, res*res*4, res*res*3)
 *   tangent_bgra     tangent-space normal map, B G R A = e(z) e(y) e(x) 255 (res*res*4 bytes),
 *                    padded like the other 8-bit maps when pad != 0
 *   tangent_normal   the blended normal in the texel's tangent frame, 3 floats per texel (res*res*3),
 *                    never padded
 *   vertex_tangents  per vertex (T.x, T.y, T.z, w) in fp32, the glTF TANGENT layout: the unit
 *                    tangent and the handedness w = +-1 with bitangent = w * (N x T); (0, 0, 0, 0)
 *                    for a vertex without a frame (n_vertices*4 floats)
 * Any output may be NULL, but not all; all are host buffers.  The convention is glTF's / OpenGL's:
 * +X along +U, +Y along +V (up in the image: row 0 is the top row), +Z out of the surface.  Frames
 * come from the mesh's per-vertex normals (Point.normal; the summed face normals where a normal is
 * zero or not finite) and its UVs; a UV seam is a duplicated vertex, so frames split there.
 * Faces with an out-of-range vertex index are skipped.  The tangent outputs need
 * 3 * n_faces <= INT32_MAX, otherwise PT_ERR_UNSUPPORTED before any input is read.  With only
 * vertex_tangents requested nothing is rasterised or searched (stats texels = empty = 0).  The
 * frames are part of raster_ms, the tangent composition part of pad_ms. */
typedef struct pt_bake_outputs {
    uint8_t *bgra;             /* res*res*4 */
    uint8_t *normal_bgra;      /* res*res*4 */
    float   *normal;           /* res*res*3 */
    uint8_t *tangent_bgra;     /* res*res*4 */
    float   *tangent_normal;   /* res*res*3 */
    float   *vertex_tangents;  /* n_vertices*4 */
} pt_bake_outputs;
int pt_texture_bake_ex(pt_index *index, const void *vertices, size_t n_vertices,
                       const int32_t *faces, size_t n_faces, int k, double radius,
                       int resolution, int pad, const pt_bake_outputs *out,
                       pt_bake_stats *stats);

/* Height bake (DESIGN.md section 8, "Height bake"): the cloud's signed height above the mesh along
 * the interpolated mesh normal N (the +Z of the tangent maps, the direction renderers displace
 * along).  Per covered texel with sample position x and neighbours p_j (the k-NN list, blend
 * weights w_j, W = sum w_j): h = (float)((sum_j w_j (p_j - x).N) / W), positive where the cloud
 * lies outside the mesh.
 *   height      h per texel (res*res floats), NaN where there is no value (uncovered texel,
 *               empty neighbour list, unusable mesh normal); never padded
 *   height_u16  E(h) = clamp(floor((h - lo) * 65535 / (hi - lo) + 0.5), 0, 65535), 0 without a
 *               value and for every texel when hi == lo (res*res uint16); padded like the 8-bit
 *               maps when pad != 0, a texel without a value taking the largest code in its
 *               25 x 25 window.  Decode with h = lo + E * (hi - lo) / 65535.
 *   range       in: a finite lo < hi fixes the code range; otherwise it is the min and max of the
 *               valued heights ((0, 0) without any)
 *   range_used  out: the (lo, hi) the codes use
 *   texels      out: texels with a value
 * Either map may be NULL, but not both. */
typedef struct pt_bake_height {
    float    *height;        /* res*res, NaN = no value, never padded (may be NULL) */
    uint16_t *height_u16;    /* res*res, padded when pad != 0 (may be NULL) */
    double    range[2];      /* in: lo < hi, finite => fixed code range; else automatic */
    double    range_used[2]; /* out */
    uint64_t  texels;        /* out: texels with a value */
} pt_bake_height;
/* One texel raster and one k-NN pass for the outputs of `out` and `height`; either may be NULL, but
 * not both.  pt_texture_bake_ex(..., out, stats) is this call with height = NULL.  With heights the
 * neighbour lists are kept, so the search runs in chunks of at most 2^22 samples (4 k bytes of
 * lists each); the outputs do not depend on it.  The height stage needs 3 * n_faces <= INT32_MAX,
 * otherwise PT_ERR_UNSUPPORTED before any input is read; its time is part of pad_ms. */
int pt_texture_bake_height(pt_index *index, const void *vertices, size_t n_vertices,
                           const int32_t *faces, size_t n_faces, int k, double radius,
                           int resolution, int pad, const pt_bake_outputs *out /* may be NULL */,
                           pt_bake_height *height /* may be NULL, not both */, pt_bake_stats *stats);

/* Normal estimation (DESIGN.md section 8, "Normal estimation"): the cloud's own normals by PCA over
 * each point's k nearest neighbours, for clouds whose normals are missing (zero) or noisy.  Per
 * point i: its k-NN list on this index (k, radius as pt_knn; the list normally holds i itself), no
 * estimate with fewer than 3 entries; the centroid and the 3 x 3 scatter of the neighbours, no
 * estimate when its trace is 0 (all neighbours at one position); cyclic Jacobi, and the unit
 * eigenvector of the smallest eigenvalue is the normal.  Orientation, first rule that applies:
 * (a) the point's input normal m is usable (finite, m.m > 0): n.m >= 0; (b) a viewpoint v is given:
 * n.(v - p_i) >= 0; (c) the component of largest magnitude is >= 0 (lowest axis on ties).
 * Everything is fp64 with every operation rounded on its own, so the results are deterministic.
 *   normal_out     n x 3 floats, original point order, (0, 0, 0) without an estimate (may be NULL)
 *   variation_out  n floats, surface variation lambda0 / (lambda0 + lambda1 + lambda2) (PCL's
 *                  "curvature"), the quiet NaN 0x7fc00000 without an estimate (may be NULL)
 *   store          != 0: every estimated normal replaces the point's normal in the index's
 *                  attributes, so later pt_transfer / bake calls blend it; points without an
 *                  estimate keep their input normal.  An index without attributes
 *                  (pt_index_build_device with attrs = NULL) cannot store: PT_ERR_INVALID_ARG.
 *   viewpoint      NULL or 3 finite doubles in host memory (rule (b)), else PT_ERR_INVALID_ARG
 * Both outputs may be NULL only with store set.  k < 3: PT_ERR_INVALID_ARG; k > PT_MAX_K:
 * PT_ERR_UNSUPPORTED.  The lists are kept, so the points are processed in chunks of at most 2^22
 * (4 k bytes of lists each).  On a slab index (pt_build_opts.ids) the neighbours are that index's
 * own points, ghost points included, and the outputs are in the index's own point order.  Host
 * buffers, blocking; stats (may be NULL): points estimated and the device time of the k-NN and the
 * PCA stages. */
typedef struct pt_normals_stats {
    uint64_t estimated;      /* points with an estimate */
    float    knn_ms, pca_ms; /* device time of the k-NN self-queries and of the PCA kernel */
} pt_normals_stats;
int pt_index_estimate_normals(pt_index *index, int k, double radius, const double *viewpoint /* 3 or NULL */,
                              int store, float *normal_out, float *variation_out, pt_normals_stats *stats);

/* Normal orientation (DESIGN.md section 8, "Normal orientation"): flips the signs of the normals
 * the index holds so that they agree along the cloud's surface, by propagation along the minimum
 * spanning forest of the k-NN graph (Hoppe et al.; CGAL's mst_orient_normals).  It orients, it does
 * not estimate: run pt_index_estimate_normals with store first for a cloud without normals.  Point i
 * takes part when its stored normal m_i is usable (finite, m.m > 0), with the unit normal n_i.  The
 * edges join the points that take part and are in one another's k-NN list (k, radius as pt_knn, the
 * union of both directions); edge {i, j} weighs w = 1 - |n_i.n_j| and edges are ordered by
 * (w, min id, max id), so the forest is unique.  Each connected component is oriented from its own
 * root, its point of largest z (lowest id on ties): with a viewpoint v the root's normal faces v
 * (n.(v - p) >= 0), otherwise its z is made positive (its largest component where z is 0).  Along
 * every forest edge the child keeps the parent's sign where n_p.n_c >= 0, else takes the opposite.
 * Components are not oriented relative to one another: a radius that splits the graph, or a cloud of
 * separate parts, gives several (stats components; root_out shows which root each point followed).
 * Everything is fp64 with every operation rounded on its own, so the results are deterministic.
 *   normal_out   n x 3 floats, original point order: the stored normal, each component negated
 *                where its sign is flipped (exact); unchanged for points that do not take part
 *                (may be NULL)
 *   root_out     n int32: the id of the point's component root, -1 where it does not take part
 *                (may be NULL)
 *   store        != 0: the oriented normals replace the stored ones, so later pt_transfer / bake
 *                calls blend them
 *   viewpoint    NULL or 3 finite doubles in host memory, else PT_ERR_INVALID_ARG
 * Both outputs may be NULL only with store set.  k < 2 or an index without attributes:
 * PT_ERR_INVALID_ARG; k > PT_MAX_K: PT_ERR_UNSUPPORTED.  The edges are counted in 32 bits, so
 * n * k must be <= INT32_MAX, otherwise PT_ERR_UNSUPPORTED before any work.  All lists are kept
 * (4 n k bytes) and the graph takes about 24 bytes per edge.  On a slab index (pt_build_opts.ids)
 * the graph is that index's own points.  Host buffers, blocking; stats (may be NULL). */
typedef struct pt_orient_stats {
    uint64_t oriented;    /* points that take part */
    uint64_t flipped;     /* of those, points whose normal was negated */
    uint64_t components;  /* connected components of the graph (trees of the forest) */
    uint64_t edges;       /* undirected edges of the graph */
    float    knn_ms, mst_ms;   /* device time of the k-NN self-queries and of the rest (edges,
                                  spanning forest, signs) */
} pt_orient_stats;
int pt_index_orient_normals(pt_index *index, int k, double radius, const double *viewpoint /* 3 or NULL */,
                            int store, float *normal_out /* n*3 */, int32_t *root_out /* n */,
                            pt_orient_stats *stats);

/* Device-buffer API: same operations with inputs/outputs already resident in
 * HBM on the index's device (bench `value`, multi-GPU slabs).  `stream` is a
 * cudaStream_t passed as void* (NULL = the CUDA default stream); these calls
 * are asynchronous with respect to the host unless stated. -------------- */

/* 16-byte point attribute record kept in original point order. */
typedef struct pt_attr {
    float   nx, ny, nz;
    uint8_t r, g, b, a;
} pt_attr;

/* 32-byte candidate record exchanged between slabs (NCCL payload). */
typedef struct pt_cand {
    double  d2;      /* +inf when empty */
    int32_t id;      /* global point id, -1 when empty */
    uint8_t r, g, b, a;
    float   nx, ny, nz;
    int32_t pad_;
} pt_cand;

/* pos: n records of 4 floats (x,y,z,unused) when coord_f64 == 0, or 4 doubles
 * (x,y,z,unused) when coord_f64 != 0.  attrs may be NULL (no blend possible).
 * ids as in pt_build_opts (device pointer).  Synchronises before returning. */
int pt_index_build_device(const void *pos, int coord_f64, const pt_attr *attrs,
                          const int32_t *ids, size_t n, int device,
                          pt_index **out);

/* queries_xyz: m*3 doubles.  Any output pointer may be NULL.  cand_out[m*k]
 * receives the per-slab candidate lists for the multi-GPU merge.
 * radius2_per_query (may be NULL): per-query squared search bound that
 * overrides `radius` (used for halo searches bounded by the owner's k-th d2;
 * a candidate must have d2 <= bound). */
int pt_query_device(pt_index *index, const double *queries_xyz, size_t m, int k,
                    double radius, const double *radius2_per_query,
                    int32_t *idx_out, double *d2_out, uint8_t *rgba_out,
                    float *normal_out, pt_cand *cand_out, void *stream);

/* pt_index_estimate_normals on device buffers (normal_out n*3 floats, variation_out n floats, either
 * may be NULL), asynchronous on `stream`; same arguments, rules and results.  viewpoint is in host
 * memory.  With store the index's attributes change in `stream` order: synchronise `stream` before
 * other calls on the index. */
int pt_estimate_normals_device(pt_index *index, int k, double radius, const double *viewpoint, int store,
                               float *normal_out, float *variation_out, void *stream);

/* K5: merge n_lists candidate lists per query (lists[l*m*k + q*k + j], each
 * ascending, padded) into the global top-k and blend.  Runs on `device`. */
int pt_merge_device(const pt_cand *lists, int n_lists, size_t m, int k,
                    int32_t *idx_out, double *d2_out, uint8_t *rgba_out,
                    float *normal_out, pt_cand *cand_out, int device, void *stream);

/* The two device-buffer pieces pt_texture_bake is built from, so the texel samples can go through
 * pt_query_device or a sharded path.  Run on `device` (-1: the current one).
 * pt_bake_texels_device: vertices_xyzuv n_vertices x 5 doubles (x, y, z, u, v), faces 3 int32 per
 * face; the covered texels in ascending texel order (texel id = row * resolution + col) and their
 * sample positions.  texel_out / xyz_out need room for resolution^2 samples (texel_out uint32,
 * xyz_out 3 doubles each), or are both NULL to only count.  Synchronises `stream` and returns the
 * count in *count_out (host). */
int pt_bake_texels_device(const double *vertices_xyzuv, size_t n_vertices,
                          const int32_t *faces, size_t n_faces, int resolution,
                          uint32_t *texel_out, double *xyz_out, size_t *count_out,
                          int device, void *stream);
/* pt_bake_samples_device: pt_bake_texels_device plus the owner face of every sample in face_out
 * (room for resolution^2 int32, may be NULL; needs texel_out). */
int pt_bake_samples_device(const double *vertices_xyzuv, size_t n_vertices,
                           const int32_t *faces, size_t n_faces, int resolution,
                           uint32_t *texel_out, double *xyz_out, int32_t *face_out,
                           size_t *count_out, int device, void *stream);
/* pt_bake_compose_device: the maps of pt_texture_bake from count samples (texels as above, rgba
 * count x 4 and normal count x 3 as pt_query_device returns them).  Outputs as pt_texture_bake's,
 * in device memory; any may be NULL, but not all.  Asynchronous on `stream`. */
int pt_bake_compose_device(const uint32_t *texels, size_t count, const uint8_t *rgba,
                           const float *normal, int resolution, int pad, uint8_t *bgra_out,
                           uint8_t *normal_bgra_out, float *normal_out, int device, void *stream);
/* The device pieces of the tangent bake.  vertices_xyzuvn: n_vertices x 8 doubles
 * (x, y, z, u, v, nx, ny, nz); the texel calls above read rows of 5 (the first five columns).
 * pt_bake_frames_device: the vertex frames into frames_out (n_vertices x 8 doubles:
 * N xyz, T xyz, w, 0; all zero for a vertex without a frame) and, when tangents_out is not NULL,
 * the exported fp32 tangents (n_vertices x 4).  3 * n_faces <= INT32_MAX, otherwise
 * PT_ERR_UNSUPPORTED.  Asynchronous on `stream`. */
int pt_bake_frames_device(const double *vertices_xyzuvn, size_t n_vertices,
                          const int32_t *faces, size_t n_faces, double *frames_out,
                          float *tangents_out, int device, void *stream);
/* pt_bake_compose_tangent_device: the two tangent maps of pt_texture_bake_ex from count samples
 * (texels and sample_faces of pt_bake_samples_device, rgba / normal of pt_query_device on their
 * positions, frames of pt_bake_frames_device).  Outputs in device memory, either may be NULL but
 * not both; tangent_bgra_out is padded when pad != 0.  Asynchronous on `stream`. */
int pt_bake_compose_tangent_device(const double *vertices_xyzuvn, const double *frames,
                                   size_t n_vertices, const int32_t *faces, size_t n_faces,
                                   const uint32_t *texels, const int32_t *sample_faces,
                                   size_t count, const uint8_t *rgba, const float *normal,
                                   int resolution, int pad, uint8_t *tangent_bgra_out,
                                   float *tangent_normal_out, int device, void *stream);
/* pt_bake_compose_height_device: the height maps of pt_texture_bake_height from count samples
 * (texels, sample_faces and sample_xyz of pt_bake_samples_device, frames of pt_bake_frames_device)
 * and their neighbour lists idx (count x k, original point ids ascending by (d2, id), -1 or any id
 * outside 0..n_points-1 ends a list, as pt_query_device returns them).  cloud_xyz: n_points x 3
 * doubles in original order.  range_in (host, 2 doubles, may be NULL: automatic) as
 * pt_bake_height.range; range_out (device, 2 doubles, may be NULL) receives the range used.
 * height_out (res*res floats) and height_u16_out (res*res uint16, padded when pad != 0) are device
 * buffers, either may be NULL but not both.  3 * n_faces <= INT32_MAX, otherwise
 * PT_ERR_UNSUPPORTED.  Asynchronous on `stream`. */
int pt_bake_compose_height_device(const double *vertices_xyzuvn, const double *frames,
                                  size_t n_vertices, const int32_t *faces, size_t n_faces,
                                  const uint32_t *texels, const int32_t *sample_faces,
                                  const double *sample_xyz, size_t count, const int32_t *idx, int k,
                                  const double *cloud_xyz, size_t n_points, int resolution, int pad,
                                  const double *range_in, float *height_out,
                                  uint16_t *height_u16_out, double *range_out, int device,
                                  void *stream);

/* Halo exchange helpers for slab-sharded clouds (DESIGN.md section 6).  Fixed-capacity routing,
 * so the exchange needs no host synchronisation: per peer a send block of (cap + 1) rows of 4
 * doubles -- row 0 = (count, overflow, 0, 0), rows 1.. = (x, y, z, squared bound) of the samples
 * whose k-th-neighbour ball reaches that peer's box -- and the sample index of every row.
 * boxes: n_ranks x 6 doubles (lo xyz, hi xyz).  counts: n_ranks words (reset by the call);
 * overflow_flag is OR-ed with 1 when a block did not fit (the caller then takes its exact
 * variable-size path). */
int pt_halo_route_device(const double *queries_xyz, const pt_cand *own_cand, size_t m, int k,
                         double radius, const double *boxes, int n_ranks, int self,
                         uint32_t cap, double *send, int32_t *sel, uint32_t *counts,
                         uint32_t *overflow_flag, void *stream);
/* received blocks (n_ranks x (cap+1) x 4) -> query rows + per-row squared bounds (-1 = unused) */
int pt_halo_prepare_device(const double *recv, int n_ranks, uint32_t cap, double *queries_out,
                           double *radius2_out, void *stream);
/* merge one peer's returned lists (cap x k records) into the owner's lists in place + re-blend */
int pt_halo_merge_device(pt_cand *own_cand, const pt_cand *back, const int32_t *sel,
                         const uint32_t *count, uint32_t cap, int k, int32_t *idx_out,
                         double *d2_out, uint8_t *rgba_out, float *normal_out, void *stream);

/* Sample routing of a slab-sharded cloud: samples arrive in arbitrary order; slab r owns the
 * samples with cuts[r] <= x < cuts[r + 1] (cuts: n_ranks + 1 doubles in DEVICE memory, cuts[0]
 * = -inf, cuts[n_ranks] = +inf).  Per destination a block of `cap` rows of 4 doubles (x, y, z,
 * +inf = per-query squared bound of pt_query_device); unused rows are NaN (answered with empty
 * lists), sel[r * cap + j] = index of the sample in that row or -1, counts[r] = rows used,
 * *overflow_flag = 1 when a block did not fit (nothing is dropped silently: enlarge cap). */
int pt_route_samples_device(const double *queries_xyz, size_t m, const double *cuts, int n_ranks,
                            uint32_t cap, double *send, int32_t *sel, uint32_t *counts,
                            uint32_t *overflow_flag, void *stream);
/* The way back: dst[sel[t]] = src[t] for every row t with sel[t] >= 0 (rows of row_bytes
 * bytes, a multiple of 4). */
int pt_scatter_rows_device(const void *src, const int32_t *sel, size_t rows, uint32_t row_bytes,
                           void *dst, void *stream);

/* Ghost-zone check for slab indexes that also hold the other slabs' points within `halo` of
 * this slab's box: ORs 1 into *flag if some sample's k-th-neighbour ball (d2[m*k], bounded by
 * radius) reaches another slab's box and may leave the ghost zone, i.e. the step needs the
 * exchange after all.  boxes as in pt_halo_route_device (the slabs' OWN boxes). */
int pt_ghost_check_device(const double *queries_xyz, const double *d2, size_t m, int k,
                          double radius, const double *boxes, int n_ranks, int self,
                          double halo, uint32_t *flag, void *stream);

/* Host-buffer step of ONE slab of a sharded cloud whose index also holds the other slabs' points
 * within `halo` of its box (ghost zone): pt_transfer on the samples this slab owns plus the
 * pt_ghost_check_device test, fused per pipeline chunk.  queries: m Point records (80 B), or
 * m x 3 doubles when queries_are_xyz != 0.  boxes: n_ranks x 6 doubles in HOST memory.
 * *needs_exchange = 1 when some sample's k-th-neighbour ball may leave the ghost zone towards
 * another slab: the results of such a call are not final and the caller runs the exchange
 * (DESIGN.md section 6).  Ids are the index's global ids. */
int pt_transfer_slab(pt_index *index, const void *queries, int queries_are_xyz, size_t m, int k,
                     double radius, const double *boxes, int n_ranks, int self, double halo,
                     int32_t *idx_out, double *d2_out, uint8_t *rgba_out, float *normal_out,
                     int *needs_exchange);

/* A cloud sharded over several GPUs of one box, host side in C++ (csrc/pt_sharded.cu): x-slabs
 * at point-count quantiles, one pt_index per slab holding the slab plus a ghost zone of width
 * `halo`, samples routed to the slab whose x-range holds them, one host thread per slab.  Same
 * contract as pt_knn / pt_transfer (blocking, query order, ascending (d2, index), ids are indices
 * into the caller's `points`); results are exact for any geometry: a call that finds a ghost
 * zone too narrow widens `halo`, rebuilds the slabs and answers again (counted in `rebuilds`),
 * at most 7 times per call and never past the diagonal of the cloud's bounding box.
 * `points` must stay valid until pt_sharded_free.  n < 2^31 points in total. */
typedef struct pt_sharded pt_sharded;
typedef struct pt_sharded_opts {
    int        n_devices;  /* number of slabs, 1..64 */
    const int *devices;    /* CUDA ordinal of every slab (may repeat); NULL => slab r on r mod device count */
    double     halo;       /* ghost-zone width; <= 0: 4x the expected k_hint-th neighbour distance,
                              at most the bounding-box diagonal */
    int        k_hint;     /* k the halo estimate is made for (default 20) */
    int        coord_mode; /* PT_COORD_* */
    int        reserved[8];
} pt_sharded_opts;
typedef struct pt_sharded_info {
    int      n_slabs, rebuilds;
    double   halo;
    uint64_t n_points;
    uint64_t slab_points[64], slab_ghosts[64];
    int      slab_device[64];
} pt_sharded_info;
int pt_sharded_build(const void *points, size_t n, const pt_sharded_opts *opts, pt_sharded **out);
int pt_sharded_free(pt_sharded *sharded);
int pt_sharded_get_info(const pt_sharded *sharded, pt_sharded_info *info);
int pt_sharded_knn(pt_sharded *sharded, const void *queries, size_t m, int k, double radius,
                   int32_t *idx_out, double *d2_out);
int pt_sharded_transfer(pt_sharded *sharded, const void *queries, size_t m, int k, double radius,
                        int32_t *idx_out, double *d2_out, uint8_t *rgba_out, float *normal_out);
/* pt_texture_bake_height on the sharded cloud (DESIGN.md section 8, "Sharded bake"): same arguments,
 * argument rules, error codes and output layouts, and every output -- maps, vertex_tangents, height
 * (NaN bits included), height_u16, range_used, height->texels, stats->texels, stats->empty -- is
 * byte-identical to pt_texture_bake_height on one pt_index built from the same cloud, for any slab
 * count and device list.  Slab 0's device (the home device) rasterises the texels, builds the frames
 * and composes, encodes and pads the maps; every slab answers the samples in its x-range on its own
 * device, heights included, from its own records.  A ghost zone found too narrow widens the halo and
 * rebuilds the slabs as pt_sharded_transfer does (counted in `rebuilds`).  Stats:
 *   raster_ms  device time on the home device: upload, raster, compaction, frames
 *   knn_ms     host wall time of routing the samples, the copies between devices, the slabs'
 *              queries, ghost checks and heights, and the scatter back into sample order, ending
 *              in a synchronise
 *   pad_ms     device time on the home device: composition, tangent maps, height range and
 *              encoding, padding */
int pt_sharded_bake(pt_sharded *sharded, const void *vertices, size_t n_vertices,
                    const int32_t *faces, size_t n_faces, int k, double radius,
                    int resolution, int pad, const pt_bake_outputs *out /* may be NULL */,
                    pt_bake_height *height /* may be NULL, not both */, pt_bake_stats *stats);
/* pt_index_estimate_normals on the sharded cloud (DESIGN.md section 8, "Sharded normal estimation"):
 * same arguments, argument rules and error codes (a NULL handle: PT_ERR_INVALID_ARG), and
 * normal_out (n x 3) and variation_out (n), in the order of the caller's `points`, are
 * byte-identical to pt_index_estimate_normals on one pt_index built from the same cloud (NaN bits
 * included), as is stats->estimated, for any slab count, device list, halo and coordinate mode.
 * Every slab estimates the points it owns on its own device, from its own records, with the
 * ghost-zone check on those rows; a ghost zone found too narrow widens the halo and rebuilds the
 * slabs as pt_sharded_transfer does (counted in `rebuilds`).  store != 0: every estimated normal
 * replaces the point's normal in every slab that holds the point (its owner and the ghost zones),
 * so later pt_sharded_transfer / pt_sharded_bake calls blend it, and the handle keeps the stored
 * normals (12 bytes per point, from the first store on) so that rebuilt slabs hold them too; points
 * without an estimate keep their input normal.  Nothing is written or stored before every slab has
 * passed its check.  Stats:
 *   estimated  points with an estimate
 *   knn_ms     host wall time of the slab stage: the slabs' self-queries, ghost checks and PCA
 *              kernels, rebuilds included, the copies to the host, the scatter into point order
 *              and the store, ending in a synchronise
 *   pca_ms     device time of the PCA kernels, summed over the slabs, in the final attempt */
int pt_sharded_estimate_normals(pt_sharded *sharded, int k, double radius,
                                const double *viewpoint /* 3 or NULL */, int store, float *normal_out,
                                float *variation_out, pt_normals_stats *stats);
/* pt_index_orient_normals on the sharded cloud (DESIGN.md section 8, "Sharded normal orientation"):
 * same arguments, argument rules and error codes (a NULL handle: PT_ERR_INVALID_ARG), and
 * normal_out (n x 3) and root_out (n, global ids), in the order of the caller's `points`, are
 * byte-identical to pt_index_orient_normals on one pt_index built from the same cloud, as are
 * stats->oriented, flipped, components and edges, for any slab count, device list, halo and
 * coordinate mode.  A point takes part when the normal its records hold (the stored one, else its
 * input normal) is usable.  Every slab builds the edges of the points it owns and the minimum
 * spanning forest of the edges between them on its own device, with the ghost-zone check on its
 * own rows; a ghost zone found too narrow widens the halo and rebuilds the slabs as
 * pt_sharded_transfer does (counted in `rebuilds`).  Slab 0's device (the home device) joins those
 * forests and the edges between slabs into the cloud's forest and orients every component from
 * its root.  One difference from the single index: the n * k <= INT32_MAX limit applies to each
 * slab's records (own and ghost) times k, not to the whole cloud, so a cloud too large for one
 * index can be oriented; a slab over it is PT_ERR_UNSUPPORTED.  A cloud within the single index's
 * limit is within every slab's.  store != 0 as in pt_sharded_estimate_normals: the oriented normal
 * of every point that takes part replaces its normal in every slab that holds it, and the handle
 * keeps it for rebuilt slabs.  Nothing is written or stored before every slab has passed its check.
 * Stats:
 *   knn_ms     host wall time of the slab stage: self-queries, ghost checks, edges and the slabs'
 *              forests, rebuilds included, ending in a synchronise
 *   mst_ms     host wall time of the rest: the copies to the home device, the cloud's forest,
 *              roots, signs, the outputs and the store */
int pt_sharded_orient_normals(pt_sharded *sharded, int k, double radius,
                              const double *viewpoint /* 3 or NULL */, int store,
                              float *normal_out /* n*3 */, int32_t *root_out /* n */,
                              pt_orient_stats *stats);

/* pt_texture_render for neighbour lists that were computed elsewhere (e.g. pt_sharded_knn): the
 * cloud's positions and colours are uploaded to `device` in original order, idx[n_vertices * k]
 * (host) indexes `points`. */
int pt_texture_render_lists(const void *points, size_t n, const void *vertices, size_t n_vertices,
                            const int32_t *faces, size_t n_faces, const int32_t *idx, int k,
                            int resolution, int pad, int device, uint8_t *bgra_out,
                            pt_texture_stats *stats);

/* Tuning / introspection. */
/* Options: "knn_variant" (-1 auto [default]: grid kernel first, then scan / thread / warp for
 * the samples it hands over; 6 grid, 5 scan kernel, 2 thread kernel, 0 warp kernel),
 * "order" (0 Morton, 1 Hilbert [default], 2 Hilbert + kd refinement: no cell tables),
 * "grid" (1 build the uniform-grid cell tables [default]), "grid_tma" (1 stage candidate runs
 * with cp.async.bulk [default], 0 per-lane cp.async), "grid_pair" (1 [default]: two samples per
 * warp when k <= 16 and the first attempt's candidates are expected to fit a half-warp; 2: whenever
 * k <= 16; 0: never; the read-only "grid_pair_used" tells what the last launch did), "grid_span"
 * (1 [default]: the two-samples-per-warp launch looks up each parent cell once and copies whole
 * spans of the sorted cloud, reading attributes in sorted order; 0: one look-up and one copy per
 * cell; the read-only "grid_span_used" tells whether the last grid launch did so), "chain_pdl"
 * (1 [default]: the kernels that answer the samples a grid launch hands over are launched as
 * programmatic dependents, so their launch overlaps the kernel before them; 0: plain stream order),
 * "grid_claim" (1 [default]: the span kernel's warps claim their next pair with an atomic when a
 * launch has more than two pairs per resident warp; 0: every warp takes a fixed stride of pairs),
 * "grid_min_occ10" / "grid_admit100" / "grid_lookup_cost" (search-schedule tuning, see grid_plan:
 * finest table = finest level with >= 4.0 points per occupied cell; a block is tried first when
 * it reaches 1.00 expected k-th-neighbour distances; one bucket look-up costs 8 candidates), "sort_bits" (ordered key bits from the top, 8 per
 * radix pass; default 0 = auto: 40 up to 2^27 points, else 48),
 * "pool_keep_mb" (memory the library's private pool keeps mapped after a build or a free; default
 * -1 = up to a quarter of the device: a rebuild then reuses it -- 8.8 ms instead of 12-60 ms for
 * 50 M points -- and 0 hands everything back),
 * "sort" (1 hand-written radix sort [default], 0 cub), "host_chunks" (pipeline chunks of the
 * host-buffer API, default 8), "queue_cap" (tests: per-sample traversal queue entries, at most
 * the compiled 12), "verbose", "smem_pad" (diagnosis), "pool_guard" (debug: 256 guard bytes
 * around every device allocation of the library, compared when it is released; the read-only
 * "pool_guard_hits" counts the allocations found damaged). */
int pt_set_option(const char *name, int value);
int pt_get_option(const char *name, int *value);
/* Work counters of the query kernel since the last reset (16 words; all zero unless the library
 * was built with -DPT_STATS, a diagnosis build).  Synchronises the device. */
int pt_debug_stats(uint64_t *out16, int reset);
/* The same counters, n words of them (up to 32 hold counters, any further words are zero): the
 * span kernel's look-ups, copies and warp finish times follow the first 16 (see
 * pt_knn_traverse.cuh).  Synchronises the device. */
int pt_debug_stats_n(uint64_t *out, int n, int reset);
/* Number of kernels this library launched since process start (gpu_launches). */
uint64_t pt_kernel_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* POINTS_TRANSFER_H */

// pt_index.cuh -- the opaque handle behind the C ABI and internal entry points.
#pragma once

#include <functional>
#include <vector>

#include "pt_common.cuh"

struct pt_index {
    int          device = 0;
    int          coord_f64 = 0;
    uint32_t     n = 0;
    uint32_t     n_leaves = 0;
    int          w_levels = 0;
    int          t_levels = 0;
    void        *pts = nullptr;      // PointF/PointD [n_leaves*LEAF], Morton order
    pt_attr     *attrs = nullptr;    // [n] original order (may be null)
    pt_attr     *attrs_curve = nullptr; // [n] attrs in sorted order (float4 records with cell tables only)
    int32_t     *ids = nullptr;      // [n] original order (may be null)
    pt::Box     *boxes = nullptr;    // all pyramid levels, level 0 first
    pt::Pyramid  pyr{};
    double       bb_lo[3]{}, bb_hi[3]{};
    pt::GridBucket *grid_mem = nullptr;   // all cell tables (pt_grid.cu), pooled allocation
    size_t       grid_bytes = 0;
    void        *blk_mem = nullptr;       // block-run table and runs (build_blocks), pooled allocation
    size_t       blk_bytes = 0;
    pt::GridParams grid{};                // tables of this index (n_tables == 0: none)
    uint64_t     level_cells[22]{};       // occupied cells per lattice level (0: not counted)
    uint32_t    *fallback_word = nullptr; // device: samples the last launch handed to the warp kernel
    uint32_t    *inv_perm = nullptr;      // original index -> position in pts (index_inverse_perm, built on demand)
    uint64_t     device_bytes = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t  ev[4]{};
    float        build_ms = 0, last_query_ms = 0, last_h2d_ms = 0, last_d2h_ms = 0;

    int          sm_count = 148;
    // grow-only workspaces for the host-buffer API
    void  *ws_raw = nullptr;   size_t ws_raw_bytes = 0;    // uploaded 80-byte query records
    void  *ws_q = nullptr;     size_t ws_q_bytes = 0;      // m*3 doubles
    void  *ws_out = nullptr;   size_t ws_out_bytes = 0;    // idx | d2 | rgba | normal
    cudaStream_t cs[16]{};                                  // chunk streams of the host-buffer API
    cudaEvent_t  cev[16]{};
};

namespace pt {

// Input accessors for the build: where the unsorted coordinates come from.
struct InF4 {   // n x float4 (x,y,z,unused)
    const float4 *p;
    __device__ __forceinline__ void load(uint32_t i, double &x, double &y, double &z) const
    {
        float4 v = p[i];
        x = v.x; y = v.y; z = v.z;
    }
};
struct InD4 {   // n x double4-like (x,y,z,unused), 32-byte records
    const double *p;
    __device__ __forceinline__ void load(uint32_t i, double &x, double &y, double &z) const
    {
        const double2 *q = reinterpret_cast<const double2 *>(p + 4 * (size_t)i);
        double2 a = q[0], b = q[1];
        x = a.x; y = a.y; z = b.x;
    }
};
struct InD3 {   // n x 3 packed doubles
    const double *p;
    __device__ __forceinline__ void load(uint32_t i, double &x, double &y, double &z) const
    {
        x = p[3 * (size_t)i]; y = p[3 * (size_t)i + 1]; z = p[3 * (size_t)i + 2];
    }
};

// Builds the sorted leaves + box pyramid into `ix` (which already holds device/stream/attrs/
// ids).  out_f64 selects PointD storage.  Synchronises ix->stream before returning.
int build_index_f4(pt_index *ix, const float4 *pos, uint32_t n, bool out_f64);
int build_index_d4(pt_index *ix, const double *pos, uint32_t n, bool out_f64);
int build_index_d3(pt_index *ix, const double *pos, uint32_t n, bool out_f64);

// Upload + unpack the reference's 80-byte AoS records.
int ingest_points_aos(pt_index *ix, const void *points, size_t n, int coord_mode,
                      double **xyz_out /* n*3 doubles, device, caller frees */,
                      bool *representable);
int unpack_queries_aos(const void *raw80_dev, size_t m, double *xyz_dev, cudaStream_t s);

int launch_query(pt_index *ix, const QueryParams &qp, cudaStream_t s);
// the index's part of the query parameters (pt_api.cu); the caller adds the samples, k, r2, outputs
void fill_params(const pt_index *ix, QueryParams &qp);
// squared radius bound: +inf for a negative, NaN or infinite radius
double radius_to_r2(double radius);
// ix->inv_perm (original index -> position in pts), built on ix->stream on first use (pt_texture.cu)
int index_inverse_perm(pt_index *ix);
// The k-NN self-query of every point of ix (pt_normals.cu), asynchronous on s, in chunks of at most
// HEIGHT_CHUNK sorted records: row r (sorted record r) gets the list of the point it holds, in the
// index's own ids.  keep: lists holds n x k and row r's list is at lists + r k; else lists holds one
// chunk's rows and is reused.  then(c0, cm, lists of rows c0 .. c0 + cm) follows each chunk's query
// and returns a status.  marks (may be null): an event before the first chunk and after each query.
// rows (device, may be null): only the n_rows sorted records rows[0 .. n_rows - 1] are queried, and
// row r is sorted record rows[r].  ghost (may be null): launch_ghost_check on each chunk's rows.
struct BakeGhost;
using ChunkThen = std::function<int(uint32_t c0, uint32_t cm, const int32_t *lists)>;
int self_query_chunks(pt_index *ix, int k, double radius, int32_t *lists, bool keep, const ChunkThen &then,
                      std::vector<cudaEvent_t> *marks, cudaStream_t s, const uint32_t *rows = nullptr,
                      uint32_t n_rows = 0, const BakeGhost *ghost = nullptr);
// The argument rules of pt_index_estimate_normals that do not concern the index: PT_OK or its error.
int normals_check_args(int k, const double *viewpoint, bool store, bool any_output);
// One slab of pt_sharded_estimate_normals (pt_normals.cu), on ix's device and stream: the normals of
// the records the slab owns -- those whose x the host's cut rule (the number of the n_slabs - 1
// ascending interior `cuts` c with !(x < c)) gives to slab `self`, n_own of them as build_slabs
// counted (PT_ERR_UNSUPPORTED otherwise) -- into normal_out (n_own x 3) / variation_out (n_own),
// host buffers, in ascending local id.  check: the ghost-zone check runs on the own rows against
// the slabs' own boxes (host, n_slabs x 6) and `halo`, and *needs = 1 when it flags the step.  Adds
// the points estimated to *estimated and sets *pca_ms to the PCA kernels' device time.
// Synchronises.
struct NormalsSlab {
    const double *cuts;
    int n_slabs, self;
    size_t n_own;
    const double *boxes;
    double halo;
    bool check;
};
int normals_slab(pt_index *ix, int k, double radius, const double *viewpoint, const NormalsSlab &sl,
                 float *normal_out, float *variation_out, unsigned long long *estimated, float *pca_ms,
                 int *needs);
// The rows a slab owns and their self-query, shared by normals_slab and orient_slab (pt_normals.cu).
// slab_rows_select, on ix's device and stream: boxes, cuts and a zeroed flag to the device, and
// rows[0 .. n_rows - 1] = the sorted positions of the records the cut rule gives to slab `self`, in
// ascending order; n_rows != sl.n_own is PT_ERR_UNSUPPORTED.  Synchronises.  tmp holds tmp_bytes,
// enough for a cub select over ix->n records.  slab_rows_query: self_query_chunks over those rows,
// with the ghost-zone check when sl.check; *flag turns non-zero when it flags the step.
struct SlabRows {
    double *boxes = nullptr;          // device: n_slabs x 6 own boxes, then the n_slabs - 1 cuts
    uint32_t *rows = nullptr, *count = nullptr, *flag = nullptr;
    void *tmp = nullptr;
    size_t tmp_bytes = 0;
    uint32_t n_rows = 0;
};
int slab_rows_select(pt_index *ix, const NormalsSlab &sl, SlabRows &w);
int slab_rows_query(pt_index *ix, int k, double radius, const NormalsSlab &sl, const SlabRows &w, int32_t *lists,
                    bool keep, const ChunkThen &then, std::vector<cudaEvent_t> *marks);
void slab_rows_free(SlabRows &w, cudaStream_t s);
// The argument rules of pt_index_orient_normals that do not concern the index: PT_OK or its error.
int orient_check_args(int k, const double *viewpoint, bool store, bool any_output);
// An edge of the orientation graph (pt_orient.cu)
struct OrientEdge {
    unsigned long long w;     // bits of w = 1 - |d| >= +0
    unsigned long long key;   // lo << 32 | hi (point ids)
    uint32_t u, v;            // rows; v's LAB_BIT: d < 0
};
// One slab of pt_sharded_orient_normals (pt_orient.cu), on ix's device and stream: the self-query of
// the own rows as normals_slab runs it (*needs = 1 when the ghost check flags the step), the edges of
// the own points' lists, and the minimum spanning forest of the intra-slab edges.  Replaces `forest`
// and `cross` with that forest's edges and the slab's cross edges (one end owned elsewhere), their
// u, v and key in global ids (ix->ids), and sets *intra to the intra-slab edge count.  Synchronises.
int orient_slab(pt_index *ix, int k, double radius, const NormalsSlab &sl, std::vector<OrientEdge> &forest,
                std::vector<OrientEdge> &cross, uint64_t *intra, int *needs);
// The rest of pt_sharded_orient_normals, on the current device and stream s: the minimum spanning
// forest of the slabs' forests and cross edges (sorted by key and deduplicated first; *unique_cross
// counts what is left) over the cloud's n points, then roots, signs and outputs in point order.
// Host arrays: normal (n x 3, the doubles the slabs' records were built from: the stored normal
// widened, else the input normal), pos (with a viewpoint the n x 3 positions, else the n z values,
// as the caller gave them), normal_out (n x 3) and root_out (n).
// counts: oriented, flipped, components.  Synchronises.
struct OrientHome {
    size_t n;
    const double *normal;
    const double *pos;
    const double *viewpoint;
    float *normal_out;
    int32_t *root_out;
};
int orient_home(const OrientHome &h, const std::vector<std::vector<OrientEdge>> &forest,
                const std::vector<std::vector<OrientEdge>> &cross, uint64_t *unique_cross,
                unsigned long long counts[3], cudaStream_t s);
// Writes values (host, n x 3 floats in ix's local order, x NaN: leave that point as it is) into the
// normals of ix's attrs and attrs_curve, on ix's stream; synchronises.
int normals_store(pt_index *ix, const float *values);
// marks != null: appends an event recorded on s
cudaError_t record_mark(std::vector<cudaEvent_t> *marks, cudaStream_t s);
// Stream-ordered allocation from the library's PRIVATE memory pool of the current device (the
// application's default pool is never touched); release with pool_free.  dev_alloc / dev_free:
// cudaMalloc / cudaFree for the long-lived buffers.  Both carry guard words under "pool_guard".
int pool_alloc(void **p, size_t bytes, cudaStream_t s);
void pool_free(void *p, cudaStream_t s);
int dev_alloc(void **p, size_t bytes);
void dev_free(void *p);
int guard_hits();
void pool_trim(int device, size_t keep_bytes);
int build_grid(pt_index *ix, const unsigned long long *keys, int low_shift, const double lo[3],
               double inv_cell21, double extent);
int grid_plan(const pt_index *ix, int k, double r2, GridParams &gp);
// The block runs of ix's cell tables (pt_knn.cu), when they fit the memory budget; synchronises.
int build_blocks(pt_index *ix);
int launch_merge(const pt_cand *lists, int n_lists, uint32_t m, int k, int32_t *idx_out,
                 double *d2_out, uint8_t *rgba_out, float *normal_out, pt_cand *cand_out,
                 cudaStream_t s);

int launch_ghost_check(const double *q, const double *d2, uint32_t m, int k, double r2,
                       const double *boxes, int n_ranks, int self, double halo, uint32_t *flag,
                       cudaStream_t s);
int launch_halo_route(const double *q, const pt_cand *own, uint32_t m, int k, double r2,
                      const double *boxes, int n_ranks, int self, uint32_t cap, double *send,
                      int32_t *sel, uint32_t *counts, uint32_t *overflow_flag, cudaStream_t s);
int launch_halo_prepare(const double *recv, int n_ranks, uint32_t cap, double *q_out, double *r2_out,
                        cudaStream_t s);
int launch_halo_merge(pt_cand *own, const pt_cand *back, const int32_t *sel, const uint32_t *count_ptr,
                      uint32_t cap, int k, int32_t *idx_out, double *d2_out, uint8_t *rgba_out,
                      float *normal_out, cudaStream_t s);

int launch_route_samples(const double *q, uint32_t m, const double *cuts, int n_ranks, uint32_t cap,
                         double *send, int32_t *sel, uint32_t *counts, uint32_t *overflow_flag,
                         cudaStream_t s);
int launch_scatter_rows(const void *src, const int32_t *sel, uint32_t rows, uint32_t row_bytes, void *dst,
                        cudaStream_t s);

size_t radix_sort_workspace_bytes(uint32_t n);
int radix_sort_pairs(unsigned long long *keys, unsigned long long *keys_alt, uint32_t *vals,
                     uint32_t *vals_alt, uint32_t n, int first_bit, int end_bit, void *workspace,
                     cudaStream_t s, unsigned long long **keys_out, uint32_t **vals_out);

int  get_option(const char *name, int *value);
int  set_option(const char *name, int value);
int  opt_knn_variant();
int  opt_order();
int  opt_sort();
int  opt_smem_pad();
int  opt_queue_cap();
int  opt_grid();
int  opt_grid_tma();
int  opt_grid_pair();
int  opt_grid_span();
int  opt_chain_pdl();
int  opt_sharded_copy();
int  opt_grid_claim();
int  opt_grid_block();
int  opt_grid_min_occ10();
int  opt_grid_admit100();
int  opt_grid_lookup_cost();
void note_grid_pair_used(int used);
void note_grid_span_used(int used);
void note_grid_block_used(int used);
int  opt_sort_bits();
size_t opt_pool_keep_bytes();
int  opt_pool_guard();
int  debug_stats(unsigned long long *out16, int reset);
int  debug_stats_n(unsigned long long *out, int n, int reset);

}  // namespace pt

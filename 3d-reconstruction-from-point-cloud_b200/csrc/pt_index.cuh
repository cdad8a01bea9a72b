// pt_index.cuh -- the opaque handle behind the C ABI and internal entry points.
#pragma once

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
    pt::GridParams grid{};                // tables of this index (n_tables == 0: none)
    uint64_t     level_cells[22]{};       // occupied cells per lattice level (0: not counted)
    uint32_t    *fallback_word = nullptr; // device: samples the last launch handed to the warp kernel
    uint32_t    *inv_perm = nullptr;      // original index -> position in pts (pt_texture.cu, built on demand)
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
int  opt_grid_claim();
int  opt_grid_min_occ10();
int  opt_grid_admit100();
int  opt_grid_lookup_cost();
void note_grid_pair_used(int used);
void note_grid_span_used(int used);
int  opt_sort_bits();
size_t opt_pool_keep_bytes();
int  opt_pool_guard();
int  debug_stats(unsigned long long *out16, int reset);
int  debug_stats_n(unsigned long long *out, int n, int reset);

}  // namespace pt

// pt_api.cu -- the C ABI (include/points_transfer.h).  Thin: argument checks, device memory
// and stream plumbing, then the kernels in pt_build.cu / pt_knn.cu.  No CPU fallback exists:
// without a CUDA device every compute entry point returns PT_ERR_NO_DEVICE.
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <new>

#include "pt_index.cuh"

namespace pt {

std::atomic<uint64_t> g_launches{0};
static std::atomic<int> g_verbose{-1};
static std::atomic<int> g_knn_variant{-1};  // -1 auto (default): grid kernel first; 6 grid, 5 scan, 2 thread, 0 warp
static std::atomic<int> g_sort{1};    // 1 hand-written radix sort (default), 0 cub::DeviceRadixSort
static std::atomic<int> g_order{1};   // 0 Morton, 1 Hilbert (default), 2 Hilbert + kd refinement (no cell tables)
static std::atomic<int> g_grid{1};        // build the uniform-grid cell tables (pt_grid.cu)
static std::atomic<int> g_grid_tma{1};    // stage candidate runs with cp.async.bulk (0: per-lane cp.async)
static std::atomic<int> g_pool_keep_mb{-1};   // memory kept cached in the library's pool after a build / free; < 0: a quarter of the device
static std::atomic<int> g_sort_bits{0};   // ordered key bits, from the top; 0 = auto (40 or 48: cells contiguous down to level 13 / 16)

bool verbose()
{
    int v = g_verbose.load();
    if (v < 0) {
        const char *e = getenv("PT_VERBOSE");
        v = (e && *e && *e != '0') ? 1 : 0;
        g_verbose.store(v);
    }
    return v != 0;
}

int map_cuda_error(cudaError_t e)
{
    switch (e) {
        case cudaSuccess: return PT_OK;
        case cudaErrorMemoryAllocation: return PT_ERR_OUT_OF_MEMORY;
        case cudaErrorNoDevice:
        case cudaErrorInsufficientDriver:
        case cudaErrorInvalidDevice: return PT_ERR_NO_DEVICE;
        default: return PT_ERR_CUDA;
    }
}

int opt_knn_variant() { return g_knn_variant.load(); }
int opt_order() { return g_order.load(); }
int opt_sort() { return g_sort.load(); }
int opt_grid() { return g_grid.load(); }
int opt_grid_tma() { return g_grid_tma.load(); }
static std::atomic<int> g_grid_pair{1};   // grid kernel: two samples per warp when k <= 16
int opt_grid_pair() { return g_grid_pair.load(); }
static std::atomic<int> g_grid_span{1};   // two samples per warp: one look-up per parent cell, one copy per span (0: per cell)
int opt_grid_span() { return g_grid_span.load(); }
static std::atomic<int> g_chain_pdl{1};   // hand-over kernels launched as programmatic dependents (0: plain stream order)
int opt_chain_pdl() { return g_chain_pdl.load(); }
static std::atomic<int> g_grid_claim{1};   // span kernel: warps claim their next pair with an atomic when each has > 2 pairs (0: static stride)
int opt_grid_claim() { return g_grid_claim.load(); }
static std::atomic<int> g_grid_block{1};   // span kernel: stage the block run of the sample's cell where the index has them (0: never)
int opt_grid_block() { return g_grid_block.load(); }
static std::atomic<int> g_grid_min_occ10{40};    // finest table: finest level with >= this / 10 points per occupied cell
static std::atomic<int> g_grid_lookup_cost{8};   // grid_plan: cost of one bucket look-up, in candidates
static std::atomic<int> g_grid_admit100{100};    // grid_plan: a block is tried first when rc cells >= this / 100 expected k-th distances
int opt_grid_admit100() { return g_grid_admit100.load(); }
int opt_grid_min_occ10() { return g_grid_min_occ10.load(); }
int opt_grid_lookup_cost() { return g_grid_lookup_cost.load(); }
static std::atomic<int> g_grid_pair_used{0};   // introspection: did the last grid launch run two samples per warp
void note_grid_pair_used(int used) { g_grid_pair_used.store(used); }
static std::atomic<int> g_grid_span_used{0};   // introspection: did the last grid launch run knn_grid_span_kernel
void note_grid_span_used(int used) { g_grid_span_used.store(used); }
static std::atomic<int> g_grid_block_used{0};   // introspection: did the last grid launch run knn_grid_block_kernel
void note_grid_block_used(int used) { g_grid_block_used.store(used); }
int opt_sort_bits() { return g_sort_bits.load(); }
size_t opt_pool_keep_bytes()
{
    const int mb = g_pool_keep_mb.load();
    if (mb >= 0) return (size_t)mb << 20;
    // auto: whatever the builds needed, up to 1/4 of the (current) device; asked once per device
    static std::atomic<unsigned long long> quarter[64];
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) { cudaGetLastError(); return (size_t)2048 << 20; }
    unsigned long long q = quarter[dev].load();
    if (q == 0) {
        size_t free_b = 0, total_b = 0;
        if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) { cudaGetLastError(); return (size_t)2048 << 20; }
        q = total_b / 4;
        quarter[dev].store(q);
    }
    return (size_t)q;
}
static std::atomic<int> g_pool_guard{0};   // debug: guard words around every device allocation (pt_build.cu)
int opt_pool_guard() { return g_pool_guard.load(); }
static std::atomic<int> g_host_chunks{8};   // host-buffer API: pipeline chunks per call (one stream each, up to 16)
int opt_host_chunks() { return g_host_chunks.load(); }
static std::atomic<int> g_queue_cap{1 << 20};   // tests: shrink the per-sample queue (exactness under spilling)
int opt_queue_cap() { return g_queue_cap.load(); }
static std::atomic<int> g_smem_pad{0};   // diagnosis: extra dynamic smem per query block (occupancy probe)
int opt_smem_pad() { return g_smem_pad.load(); }
static std::atomic<int> g_sharded_copy{0};   // tests: the sharded bake copies the rows of slabs on its home device too
int opt_sharded_copy() { return g_sharded_copy.load(); }

int set_option(const char *name, int value)
{
    if (!name) return PT_ERR_INVALID_ARG;
    if (!strcmp(name, "knn_variant")) {
        if (value != -1 && value != 0 && value != 2 && value != 5 && value != 6) return PT_ERR_INVALID_ARG;
        g_knn_variant.store(value);
        return PT_OK;
    }
    if (!strcmp(name, "order")) { g_order.store(value); return PT_OK; }
    if (!strcmp(name, "sort")) { g_sort.store(value); return PT_OK; }
    if (!strcmp(name, "grid")) { g_grid.store(value ? 1 : 0); return PT_OK; }
    if (!strcmp(name, "grid_tma")) { g_grid_tma.store(value ? 1 : 0); return PT_OK; }
    if (!strcmp(name, "grid_min_occ10")) { g_grid_min_occ10.store(value < 5 ? 5 : value); return PT_OK; }
    if (!strcmp(name, "grid_lookup_cost")) { g_grid_lookup_cost.store(value < 0 ? 0 : value); return PT_OK; }
    if (!strcmp(name, "grid_admit100")) { g_grid_admit100.store(value < 10 ? 10 : value); return PT_OK; }
    if (!strcmp(name, "grid_pair")) { g_grid_pair.store(value < 0 ? 0 : (value > 2 ? 2 : value)); return PT_OK; }
    if (!strcmp(name, "grid_span")) { g_grid_span.store(value ? 1 : 0); return PT_OK; }
    if (!strcmp(name, "chain_pdl")) { g_chain_pdl.store(value ? 1 : 0); return PT_OK; }
    if (!strcmp(name, "grid_claim")) { g_grid_claim.store(value ? 1 : 0); return PT_OK; }
    if (!strcmp(name, "grid_block")) { g_grid_block.store(value ? 1 : 0); return PT_OK; }
    if (!strcmp(name, "sort_bits")) { g_sort_bits.store(value); return PT_OK; }
    if (!strcmp(name, "pool_keep_mb")) { g_pool_keep_mb.store(value < 0 ? -1 : value); return PT_OK; }
    if (!strcmp(name, "pool_guard")) { g_pool_guard.store(value ? 1 : 0); return PT_OK; }
    if (!strcmp(name, "smem_pad")) { g_smem_pad.store(value < 0 ? 0 : value); return PT_OK; }
    if (!strcmp(name, "queue_cap")) { g_queue_cap.store(value < 2 ? 2 : value); return PT_OK; }
    if (!strcmp(name, "host_chunks")) { g_host_chunks.store(value < 1 ? 1 : (value > 64 ? 64 : value)); return PT_OK; }
    if (!strcmp(name, "sharded_copy")) { g_sharded_copy.store(value ? 1 : 0); return PT_OK; }
    if (!strcmp(name, "verbose")) { g_verbose.store(value ? 1 : 0); return PT_OK; }
    return PT_ERR_INVALID_ARG;
}
int get_option(const char *name, int *value)
{
    if (!name || !value) return PT_ERR_INVALID_ARG;
    if (!strcmp(name, "knn_variant")) { *value = g_knn_variant.load(); return PT_OK; }
    if (!strcmp(name, "order")) { *value = g_order.load(); return PT_OK; }
    if (!strcmp(name, "sort")) { *value = g_sort.load(); return PT_OK; }
    if (!strcmp(name, "grid")) { *value = g_grid.load(); return PT_OK; }
    if (!strcmp(name, "grid_tma")) { *value = g_grid_tma.load(); return PT_OK; }
    if (!strcmp(name, "grid_min_occ10")) { *value = g_grid_min_occ10.load(); return PT_OK; }
    if (!strcmp(name, "grid_lookup_cost")) { *value = g_grid_lookup_cost.load(); return PT_OK; }
    if (!strcmp(name, "grid_admit100")) { *value = g_grid_admit100.load(); return PT_OK; }
    if (!strcmp(name, "grid_pair")) { *value = g_grid_pair.load(); return PT_OK; }
    if (!strcmp(name, "grid_pair_used")) { *value = g_grid_pair_used.load(); return PT_OK; }
    if (!strcmp(name, "grid_span")) { *value = g_grid_span.load(); return PT_OK; }
    if (!strcmp(name, "grid_span_used")) { *value = g_grid_span_used.load(); return PT_OK; }
    if (!strcmp(name, "chain_pdl")) { *value = g_chain_pdl.load(); return PT_OK; }
    if (!strcmp(name, "grid_claim")) { *value = g_grid_claim.load(); return PT_OK; }
    if (!strcmp(name, "grid_block")) { *value = g_grid_block.load(); return PT_OK; }
    if (!strcmp(name, "grid_block_used")) { *value = g_grid_block_used.load(); return PT_OK; }
    if (!strcmp(name, "sort_bits")) { *value = g_sort_bits.load(); return PT_OK; }
    if (!strcmp(name, "pool_keep_mb")) { *value = g_pool_keep_mb.load(); return PT_OK; }
    if (!strcmp(name, "pool_guard")) { *value = g_pool_guard.load(); return PT_OK; }
    if (!strcmp(name, "pool_guard_hits")) { *value = guard_hits(); return PT_OK; }
    if (!strcmp(name, "smem_pad")) { *value = g_smem_pad.load(); return PT_OK; }
    if (!strcmp(name, "queue_cap")) { *value = g_queue_cap.load(); return PT_OK; }
    if (!strcmp(name, "host_chunks")) { *value = g_host_chunks.load(); return PT_OK; }
    if (!strcmp(name, "sharded_copy")) { *value = g_sharded_copy.load(); return PT_OK; }
    if (!strcmp(name, "verbose")) { *value = verbose() ? 1 : 0; return PT_OK; }
    return PT_ERR_INVALID_ARG;
}

static int grow(void **p, size_t *cap, size_t need)
{
    if (need <= *cap) return PT_OK;
    dev_free(*p);
    *p = nullptr;
    *cap = 0;
    size_t want = opt_pool_guard() ? need : need + need / 4;   // guard words sit right behind the bytes in use
    PT_TRY(dev_alloc(p, want));
    *cap = want;
    return PT_OK;
}

static void destroy_index(pt_index *ix);

static int new_index(int device, pt_index **out)
{
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) { cudaGetLastError(); return PT_ERR_NO_DEVICE; }
    if (device < 0) PT_CUDA(cudaGetDevice(&device));
    if (device >= count) return PT_ERR_INVALID_ARG;
    PT_CUDA(cudaSetDevice(device));
    pt_index *ix = new (std::nothrow) pt_index();
    if (!ix) return PT_ERR_OUT_OF_MEMORY;
    ix->device = device;
    e = cudaStreamCreateWithFlags(&ix->stream, cudaStreamNonBlocking);
    for (auto &ev : ix->ev)
        if (e == cudaSuccess) e = cudaEventCreate(&ev);
    if (e == cudaSuccess && dev_alloc((void **)&ix->fallback_word, 16) != PT_OK) e = cudaErrorMemoryAllocation;
    if (e == cudaSuccess) e = cudaMemset(ix->fallback_word, 0, 16);
    int sms = 0;
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    if (e != cudaSuccess) {          // nothing leaks on a half-constructed handle
        if (verbose()) fprintf(stderr, "[points_transfer] new_index: %s\n", cudaGetErrorString(e));
        destroy_index(ix);
        return map_cuda_error(e);
    }
    ix->sm_count = sms > 0 ? sms : 148;
    *out = ix;
    return PT_OK;
}

static void destroy_index(pt_index *ix)
{
    if (!ix) return;
    cudaSetDevice(ix->device);
    if (ix->stream) cudaStreamSynchronize(ix->stream);
    for (auto &c : ix->cs) if (c) cudaStreamSynchronize(c);
    // sorted points, boxes and cell tables come from the library's stream-ordered pool: back to it
    pool_free(ix->pts, ix->stream);
    pool_free(ix->boxes, ix->stream);
    pool_free(ix->grid_mem, ix->stream);
    pool_free(ix->blk_mem, ix->stream);
    pool_free(ix->attrs_curve, ix->stream);
    pool_free(ix->attrs, ix->stream);         // (attributes and ids too: cudaMalloc / cudaFree of 0.8 GB cost milliseconds)
    pool_free(ix->ids, ix->stream);
    if (ix->stream) cudaStreamSynchronize(ix->stream);
    pool_trim(ix->device, opt_pool_keep_bytes());   // "pool_keep_mb" of it stays mapped for the next build
    dev_free(ix->fallback_word); dev_free(ix->inv_perm);
    dev_free(ix->ws_raw); dev_free(ix->ws_q); dev_free(ix->ws_out);
    for (auto &c : ix->cs) if (c) cudaStreamDestroy(c);
    for (auto &e : ix->cev) if (e) cudaEventDestroy(e);
    for (auto &ev : ix->ev) if (ev) cudaEventDestroy(ev);
    if (ix->stream) cudaStreamDestroy(ix->stream);
    cudaGetLastError();
    delete ix;
}

double radius_to_r2(double radius)
{
    if (!(radius >= 0.0) || std::isinf(radius)) return INFINITY;
    return radius * radius;  // Distance::transformed_distance(d), src/Distance.h:97
}

void fill_params(const pt_index *ix, QueryParams &qp)
{
    qp.pts = ix->pts;
    qp.attrs = ix->attrs;
    qp.attrs_curve = ix->attrs_curve;
    qp.ids = ix->ids;
    qp.pyr = ix->pyr;
    qp.n = ix->n;
    qp.n_leaves = ix->n_leaves;
    qp.w_levels = ix->w_levels;
    qp.t_levels = ix->t_levels;
    qp.pq_cap = opt_queue_cap();
    qp.grid.n_tables = 0;      // launch_query plans the grid search
    qp.grid.n_attempts = 0;
}

}  // namespace pt

using namespace pt;

extern "C" {

const char *pt_version(void) { return "points_transfer_b200 0.1 (sm_100a)"; }

const char *pt_status_string(int status)
{
    switch (status) {
        case PT_OK: return "ok";
        case PT_ERR_INVALID_ARG: return "invalid argument";
        case PT_ERR_CUDA: return "CUDA error";
        case PT_ERR_NO_DEVICE: return "no CUDA device (there is no CPU fallback)";
        case PT_ERR_OUT_OF_MEMORY: return "out of device memory";
        case PT_ERR_UNSUPPORTED: return "unsupported parameter (k must be 1..32)";
        case PT_ERR_NOT_REPRESENTABLE: return "cloud coordinates are not fp32-representable";
        case PT_ERR_NON_FINITE: return "non-finite coordinate in the cloud";
        default: return "unknown status";
    }
}

int pt_device_count(void)
{
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess) { cudaGetLastError(); return 0; }
    return count;
}

uint64_t pt_kernel_launch_count(void) { return g_launches.load(); }
int pt_set_option(const char *name, int value) { return set_option(name, value); }
int pt_get_option(const char *name, int *value) { return get_option(name, value); }
int pt_debug_stats(uint64_t *out16, int reset)
{
    if (!out16) return PT_ERR_INVALID_ARG;
    return debug_stats(reinterpret_cast<unsigned long long *>(out16), reset);
}
int pt_debug_stats_n(uint64_t *out, int n, int reset)
{
    if (!out && n > 0) return PT_ERR_INVALID_ARG;
    return debug_stats_n(reinterpret_cast<unsigned long long *>(out), n, reset);
}

int pt_index_build(const void *points, size_t n, const pt_build_opts *opts, pt_index **out)
{
    if (!out || (!points && n) || n >= 0x7fffffffull) return PT_ERR_INVALID_ARG;
    *out = nullptr;
    int device = opts ? opts->device : -1;
    int mode = opts ? opts->coord_mode : PT_COORD_AUTO;
    if (mode < PT_COORD_AUTO || mode > PT_COORD_F64) return PT_ERR_INVALID_ARG;
    pt_index *ix = nullptr;
    PT_TRY(new_index(device, &ix));
    double *xyz = nullptr;
    bool representable = true;
    int rc = ingest_points_aos(ix, points, n, mode, &xyz, &representable);
    if (rc == PT_OK && mode == PT_COORD_F32 && !representable) rc = PT_ERR_NOT_REPRESENTABLE;
    if (rc == PT_OK && opts && opts->ids && n) {
        cudaError_t e = pool_alloc((void **)&ix->ids, sizeof(int32_t) * n, ix->stream) == PT_OK ? cudaSuccess : cudaErrorMemoryAllocation;
        if (e == cudaSuccess)
            e = cudaMemcpyAsync(ix->ids, opts->ids, sizeof(int32_t) * n, cudaMemcpyHostToDevice,
                                ix->stream);
        rc = map_cuda_error(e);
    }
    if (rc == PT_OK) {
        bool f64 = mode == PT_COORD_F64 || (mode == PT_COORD_AUTO && !representable);
        rc = build_index_d3(ix, xyz, (uint32_t)n, f64);
    }
    dev_free(xyz);
    if (rc != PT_OK) { destroy_index(ix); return rc; }
    *out = ix;
    return PT_OK;
}

int pt_index_build_device(const void *pos, int coord_f64, const pt_attr *attrs,
                          const int32_t *ids, size_t n, int device, pt_index **out)
{
    if (!out || (!pos && n) || n >= 0x7fffffffull) return PT_ERR_INVALID_ARG;
    *out = nullptr;
    pt_index *ix = nullptr;
    PT_TRY(new_index(device, &ix));
    int rc = PT_OK;
    if (n && attrs) {
        cudaError_t e = pool_alloc((void **)&ix->attrs, sizeof(pt_attr) * n, ix->stream) == PT_OK ? cudaSuccess : cudaErrorMemoryAllocation;
        if (e == cudaSuccess)
            e = cudaMemcpyAsync(ix->attrs, attrs, sizeof(pt_attr) * n, cudaMemcpyDeviceToDevice,
                                ix->stream);
        rc = map_cuda_error(e);
    }
    if (rc == PT_OK && n && ids) {
        cudaError_t e = pool_alloc((void **)&ix->ids, sizeof(int32_t) * n, ix->stream) == PT_OK ? cudaSuccess : cudaErrorMemoryAllocation;
        if (e == cudaSuccess)
            e = cudaMemcpyAsync(ix->ids, ids, sizeof(int32_t) * n, cudaMemcpyDeviceToDevice,
                                ix->stream);
        rc = map_cuda_error(e);
    }
    if (rc == PT_OK)
        rc = coord_f64 ? build_index_d4(ix, (const double *)pos, (uint32_t)n, true)
                       : build_index_f4(ix, (const float4 *)pos, (uint32_t)n, false);
    if (rc != PT_OK) { destroy_index(ix); return rc; }
    *out = ix;
    return PT_OK;
}

int pt_index_free(pt_index *index)
{
    destroy_index(index);
    return PT_OK;
}

int pt_index_get_info(const pt_index *ix, pt_index_info *info)
{
    if (!ix || !info) return PT_ERR_INVALID_ARG;
    memset(info, 0, sizeof *info);
    info->n_points = ix->n;
    info->n_leaves = ix->n_leaves;
    info->n_levels = ix->pyr.n_levels;
    info->coord_mode = ix->coord_f64 ? PT_COORD_F64 : PT_COORD_F32;
    info->device = ix->device;
    info->last_fallback_samples = -1;
    if (ix->fallback_word) {   // written by the last warp-kernel stage (device word; this call synchronises)
        uint32_t c = 0;
        if (cudaSetDevice(ix->device) == cudaSuccess &&
            cudaMemcpy(&c, ix->fallback_word, sizeof c, cudaMemcpyDeviceToHost) == cudaSuccess)
            info->last_fallback_samples = (int)c;
        cudaGetLastError();
    }
    for (int a = 0; a < 3; ++a) { info->bbox_lo[a] = ix->bb_lo[a]; info->bbox_hi[a] = ix->bb_hi[a]; }
    info->device_bytes = ix->device_bytes;
    info->build_ms = ix->build_ms;
    info->last_query_ms = ix->last_query_ms;
    info->last_h2d_ms = ix->last_h2d_ms;
    info->last_d2h_ms = ix->last_d2h_ms;
    return PT_OK;
}

int pt_index_fallback_counts(const pt_index *ix, uint32_t out2[2])
{
    if (!ix || !out2) return PT_ERR_INVALID_ARG;
    out2[0] = out2[1] = 0;
    if (!ix->fallback_word) return PT_OK;
    PT_CUDA(cudaSetDevice(ix->device));
    PT_CUDA(cudaMemcpy(out2, ix->fallback_word, 2 * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    return PT_OK;
}

static int query_device_on(pt_index *ix, const double *queries_xyz, size_t m, int k, double radius,
                           const double *radius2_per_query, int32_t *idx_out, double *d2_out,
                           uint8_t *rgba_out, float *normal_out, pt_cand *cand_out,
                           cudaStream_t stream)
{
    QueryParams qp{};
    fill_params(ix, qp);
    qp.queries = queries_xyz;
    qp.r2_per_query = radius2_per_query;
    qp.m = (uint32_t)m;
    qp.k = k;
    qp.r2 = radius_to_r2(radius);
    qp.idx_out = idx_out; qp.d2_out = d2_out; qp.rgba_out = rgba_out;
    qp.normal_out = normal_out; qp.cand_out = cand_out;
    return launch_query(ix, qp, stream);
}

int pt_query_device(pt_index *ix, const double *queries_xyz, size_t m, int k, double radius,
                    const double *radius2_per_query, int32_t *idx_out, double *d2_out,
                    uint8_t *rgba_out, float *normal_out, pt_cand *cand_out, void *stream)
{
    if (!ix || (!queries_xyz && m) || m > 0xfffffff0ull) return PT_ERR_INVALID_ARG;
    if (k < 1 || k > PT_MAX_K) return PT_ERR_UNSUPPORTED;
    if ((rgba_out || normal_out) && !ix->attrs && ix->n) return PT_ERR_INVALID_ARG;
    PT_CUDA(cudaSetDevice(ix->device));
    return query_device_on(ix, queries_xyz, m, k, radius, radius2_per_query, idx_out, d2_out,
                           rgba_out, normal_out, cand_out, (cudaStream_t)stream);
}

int pt_merge_device(const pt_cand *lists, int n_lists, size_t m, int k, int32_t *idx_out,
                    double *d2_out, uint8_t *rgba_out, float *normal_out, pt_cand *cand_out,
                    int device, void *stream)
{
    if ((!lists && m) || m > 0xfffffff0ull) return PT_ERR_INVALID_ARG;
    if (pt_device_count() == 0) return PT_ERR_NO_DEVICE;
    if (device >= 0) PT_CUDA(cudaSetDevice(device));
    return launch_merge(lists, n_lists, (uint32_t)m, k, idx_out, d2_out, rgba_out, normal_out,
                        cand_out, (cudaStream_t)stream);
}

int pt_halo_route_device(const double *queries_xyz, const pt_cand *own_cand, size_t m, int k,
                         double radius, const double *boxes, int n_ranks, int self, uint32_t cap,
                         double *send, int32_t *sel, uint32_t *counts, uint32_t *overflow_flag,
                         void *stream)
{
    if ((m && (!queries_xyz || !own_cand)) || !boxes || !send || !sel || !counts || !overflow_flag ||
        m > 0xfffffff0ull || self < 0 || self >= n_ranks)
        return PT_ERR_INVALID_ARG;
    return launch_halo_route(queries_xyz, own_cand, (uint32_t)m, k, radius_to_r2(radius), boxes,
                             n_ranks, self, cap, send, sel, counts, overflow_flag,
                             (cudaStream_t)stream);
}

int pt_route_samples_device(const double *queries_xyz, size_t m, const double *cuts, int n_ranks,
                            uint32_t cap, double *send, int32_t *sel, uint32_t *counts,
                            uint32_t *overflow_flag, void *stream)
{
    if ((m && !queries_xyz) || !cuts || !send || !sel || !counts || !overflow_flag || m > 0xfffffff0ull)
        return PT_ERR_INVALID_ARG;
    if (pt_device_count() == 0) return PT_ERR_NO_DEVICE;
    return launch_route_samples(queries_xyz, (uint32_t)m, cuts, n_ranks, cap, send, sel, counts,
                                overflow_flag, (cudaStream_t)stream);
}

int pt_scatter_rows_device(const void *src, const int32_t *sel, size_t rows, uint32_t row_bytes,
                           void *dst, void *stream)
{
    if ((rows && (!src || !sel || !dst)) || rows > 0xfffffff0ull) return PT_ERR_INVALID_ARG;
    if (pt_device_count() == 0) return PT_ERR_NO_DEVICE;
    return launch_scatter_rows(src, sel, (uint32_t)rows, row_bytes, dst, (cudaStream_t)stream);
}

int pt_ghost_check_device(const double *queries_xyz, const double *d2, size_t m, int k,
                          double radius, const double *boxes, int n_ranks, int self, double halo,
                          uint32_t *flag, void *stream)
{
    if ((m && (!queries_xyz || !d2)) || !boxes || !flag || m > 0xfffffff0ull) return PT_ERR_INVALID_ARG;
    return launch_ghost_check(queries_xyz, d2, (uint32_t)m, k, radius_to_r2(radius), boxes, n_ranks,
                              self, halo, flag, (cudaStream_t)stream);
}

int pt_halo_prepare_device(const double *recv, int n_ranks, uint32_t cap, double *queries_out,
                           double *radius2_out, void *stream)
{
    if (!recv || !queries_out || !radius2_out || n_ranks < 1) return PT_ERR_INVALID_ARG;
    return launch_halo_prepare(recv, n_ranks, cap, queries_out, radius2_out, (cudaStream_t)stream);
}

int pt_halo_merge_device(pt_cand *own_cand, const pt_cand *back, const int32_t *sel,
                         const uint32_t *count, uint32_t cap, int k, int32_t *idx_out,
                         double *d2_out, uint8_t *rgba_out, float *normal_out, void *stream)
{
    if (!own_cand || !back || !sel || !count) return PT_ERR_INVALID_ARG;
    return launch_halo_merge(own_cand, back, sel, count, cap, k, idx_out, d2_out, rgba_out,
                             normal_out, (cudaStream_t)stream);
}

// Host-buffer query.  Large batches are cut into chunks, each on its own stream (up to 16), so
// the H2D copy of the 80-byte records, the kernels and the D2H copy of the results overlap
// (pinned caller buffers make the copies truly asynchronous; pageable ones still work).
// Ghost-zone check of a slab index (pt_transfer_slab): host copies of the slabs' boxes.
struct GhostCheck {
    const double *boxes;   // n_ranks x 6, host
    int n_ranks, self;
    double halo;
    int *needs_exchange;   // out
};

static int host_query(pt_index *ix, const void *queries, size_t m, int k, double radius,
                      int32_t *idx_out, double *d2_out, uint8_t *rgba_out, float *normal_out,
                      bool queries_are_xyz = false, const GhostCheck *ghost = nullptr)
{
    if (!ix || (!queries && m) || m > 0xfffffff0ull) return PT_ERR_INVALID_ARG;
    if (k < 1 || k > PT_MAX_K) return PT_ERR_UNSUPPORTED;
    if ((rgba_out || normal_out) && !ix->attrs && ix->n) return PT_ERR_INVALID_ARG;
    if (ghost && ghost->needs_exchange) *ghost->needs_exchange = 0;
    if (m == 0) return PT_OK;
    PT_CUDA(cudaSetDevice(ix->device));
    cudaStream_t s = ix->stream;
    const size_t mk = m * (size_t)k;
    const bool need_d2 = d2_out || ghost;      // the ghost check reads the k-th d2 on the device
    // output workspace layout: d2 | idx | normal | rgba (descending alignment)
    size_t off_d2 = 0, off_idx = off_d2 + (need_d2 ? mk * 8 : 0);
    size_t off_nrm = off_idx + (idx_out ? mk * 4 : 0);
    size_t off_rgba = off_nrm + (normal_out ? m * 12 : 0);
    size_t total = off_rgba + (rgba_out ? m * 4 : 0);
    if (!queries_are_xyz) PT_TRY(grow(&ix->ws_raw, &ix->ws_raw_bytes, m * PT_POINT_STRIDE));
    PT_TRY(grow(&ix->ws_q, &ix->ws_q_bytes, m * 24));
    // tail of the output workspace: the slabs' boxes and the check flag of the ghost zone
    const size_t off_boxes = (total + 15) & ~(size_t)15;
    const size_t off_flag = off_boxes + (ghost ? sizeof(double) * 6 * (size_t)ghost->n_ranks : 0);
    PT_TRY(grow(&ix->ws_out, &ix->ws_out_bytes, off_flag + 16));
    char *o = (char *)ix->ws_out;
    if (ghost) {
        PT_CUDA(cudaMemcpyAsync(o + off_boxes, ghost->boxes, sizeof(double) * 6 * (size_t)ghost->n_ranks,
                                cudaMemcpyHostToDevice, s));
        PT_CUDA(cudaMemsetAsync(o + off_flag, 0, sizeof(uint32_t), s));
    }

    constexpr int NCS = 16;  // chunk streams (a chunk kernel has a ~0.27 ms latency floor, so chunks must overlap)
    size_t chunk = m;
    const size_t want = (size_t)opt_host_chunks();
    if (m >= 32768 && want > 1) chunk = (((m + want - 1) / want) + 31) & ~(size_t)31;
    const int n_chunks = (int)((m + chunk - 1) / chunk);
    const int n_streams = n_chunks < NCS ? n_chunks : NCS;
    for (int i = 0; i < n_streams; ++i) {
        if (!ix->cs[i]) PT_CUDA(cudaStreamCreateWithFlags(&ix->cs[i], cudaStreamNonBlocking));
        if (!ix->cev[i]) PT_CUDA(cudaEventCreateWithFlags(&ix->cev[i], cudaEventDisableTiming));
    }
    // Everything below may leave work in flight on the chunk streams: on any failure the
    // streams are drained before the status is returned, so no copy is still writing into the
    // caller's buffers after the call has reported an error (ABI: blocking on return).
    auto issue = [&]() -> int {
        PT_CUDA(cudaEventRecord(ix->ev[0], s));
        for (int i = 0; i < n_streams; ++i) PT_CUDA(cudaStreamWaitEvent(ix->cs[i], ix->ev[0], 0));
        for (int c = 0; c < n_chunks; ++c) {
            const int si = c % NCS;
            cudaStream_t st = ix->cs[si];
            const size_t c0 = (size_t)c * chunk;
            const size_t cm = m - c0 < chunk ? m - c0 : chunk;
            double *qd = (double *)ix->ws_q + 3 * c0;
            if (queries_are_xyz) {
                PT_CUDA(cudaMemcpyAsync(qd, (const double *)queries + 3 * c0, cm * 24,
                                        cudaMemcpyHostToDevice, st));
            } else {
                char *raw = (char *)ix->ws_raw + c0 * PT_POINT_STRIDE;
                PT_CUDA(cudaMemcpyAsync(raw, (const char *)queries + c0 * PT_POINT_STRIDE,
                                        cm * PT_POINT_STRIDE, cudaMemcpyHostToDevice, st));
                PT_TRY(unpack_queries_aos(raw, cm, qd, st));
            }
            PT_TRY(query_device_on(ix, qd, cm, k, radius, nullptr,
                                   idx_out ? (int32_t *)(o + off_idx) + c0 * k : nullptr,
                                   need_d2 ? (double *)(o + off_d2) + c0 * k : nullptr,
                                   rgba_out ? (uint8_t *)(o + off_rgba) + c0 * 4 : nullptr,
                                   normal_out ? (float *)(o + off_nrm) + c0 * 3 : nullptr, nullptr, st));
            if (ghost)
                PT_TRY(launch_ghost_check(qd, (double *)(o + off_d2) + c0 * k, (uint32_t)cm, k,
                                          radius_to_r2(radius), (const double *)(o + off_boxes),
                                          ghost->n_ranks, ghost->self, ghost->halo,
                                          (uint32_t *)(o + off_flag), st));
            if (d2_out) PT_CUDA(cudaMemcpyAsync(d2_out + c0 * k, (double *)(o + off_d2) + c0 * k, cm * k * 8, cudaMemcpyDeviceToHost, st));
            if (idx_out) PT_CUDA(cudaMemcpyAsync(idx_out + c0 * k, (int32_t *)(o + off_idx) + c0 * k, cm * k * 4, cudaMemcpyDeviceToHost, st));
            if (normal_out) PT_CUDA(cudaMemcpyAsync(normal_out + c0 * 3, (float *)(o + off_nrm) + c0 * 3, cm * 12, cudaMemcpyDeviceToHost, st));
            if (rgba_out) PT_CUDA(cudaMemcpyAsync(rgba_out + c0 * 4, (uint8_t *)(o + off_rgba) + c0 * 4, cm * 4, cudaMemcpyDeviceToHost, st));
        }
        for (int i = 0; i < n_streams; ++i) {
            PT_CUDA(cudaEventRecord(ix->cev[i], ix->cs[i]));
            PT_CUDA(cudaStreamWaitEvent(s, ix->cev[i], 0));
        }
        return PT_OK;
    };
    uint32_t flag = 0;
    int rc = issue();
    if (rc == PT_OK && ghost) rc = map_cuda_error(cudaMemcpyAsync(&flag, o + off_flag, sizeof flag, cudaMemcpyDeviceToHost, s));
    if (rc == PT_OK) rc = map_cuda_error(cudaEventRecord(ix->ev[3], s));
    if (rc != PT_OK) {
        for (int i = 0; i < n_streams; ++i) cudaStreamSynchronize(ix->cs[i]);
        cudaStreamSynchronize(s);
        cudaGetLastError();
        return rc;
    }
    PT_CUDA(cudaStreamSynchronize(s));
    if (ghost && ghost->needs_exchange) *ghost->needs_exchange = flag ? 1 : 0;
    ix->last_h2d_ms = 0.f;          // overlapped with the kernels: only the total is meaningful
    ix->last_d2h_ms = 0.f;
    cudaEventElapsedTime(&ix->last_query_ms, ix->ev[0], ix->ev[3]);
    return PT_OK;
}

int pt_knn(pt_index *index, const void *queries, size_t m, int k, double radius,
           int32_t *idx_out, double *d2_out)
{
    if (!idx_out && m) return PT_ERR_INVALID_ARG;
    return host_query(index, queries, m, k, radius, idx_out, d2_out, nullptr, nullptr);
}

int pt_transfer(pt_index *index, const void *queries, size_t m, int k, double radius,
                int32_t *idx_out, double *d2_out, uint8_t *rgba_out, float *normal_out)
{
    if ((!rgba_out && !normal_out) && m) return PT_ERR_INVALID_ARG;
    return host_query(index, queries, m, k, radius, idx_out, d2_out, rgba_out, normal_out);
}

int pt_transfer_slab(pt_index *index, const void *queries, int queries_are_xyz, size_t m, int k,
                     double radius, const double *boxes, int n_ranks, int self, double halo,
                     int32_t *idx_out, double *d2_out, uint8_t *rgba_out, float *normal_out,
                     int *needs_exchange)
{
    if (!boxes || !needs_exchange || n_ranks < 1 || n_ranks > 4096 || self < 0 || self >= n_ranks)
        return PT_ERR_INVALID_ARG;
    GhostCheck g{boxes, n_ranks, self, halo, needs_exchange};
    return host_query(index, queries, m, k, radius, idx_out, d2_out, rgba_out, normal_out,
                      queries_are_xyz != 0, &g);
}

}  // extern "C"

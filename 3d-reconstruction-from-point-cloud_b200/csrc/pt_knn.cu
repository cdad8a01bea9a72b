// pt_knn.cu -- exact k-NN query + fused blend (replaces the per-corner
// `K_neighbor_search search(tree, q, K)` loop, /root/reference src/pointsTransfer.cpp:470-479,
// metric src/Distance.h:6-11, pruning bound src/Distance.h:27-57).
//
// Four kernels share the helpers in this file:
//   variant 6 ("grid",   pt_knn_grid.cuh, pt_knn_span.cuh): one warp per sample (two at k <= 16)
//     over the uniform-grid cell tables, candidate runs staged in shared memory by bulk async
//     copies; the default first stage -- samples it cannot prove final go to the kernels below;
//   variant 5 ("scan",   pt_knn_scan.cuh)  : one thread per sample, unsorted top-k slots;
//   variant 2 ("thread", pt_knn_thread.cuh): one thread per sample, top-k heap;
//     both walk the box pyramid with pt_knn_traverse.cuh, state in shared-memory columns;
//   variant 0 ("warp",   below)            : one warp per sample, 32-wide levels, nearest-child-
//     first DFS, top-k as a sorted list distributed one entry per lane.  Most instructions per
//     sample but the shortest latency and no per-sample state limits: it answers small launches
//     and re-runs the samples the other two hand over (exact fallback).
#include <type_traits>
#include <cub/device/device_scan.cuh>
#include "pt_index.cuh"

namespace pt {

// ---- programmatic dependent launch (the hand-over chain of launch_chain) ---------------------
// A kernel launched with programmatic stream serialization may start before the kernel ahead of
// it in the stream has finished; griddepcontrol.wait then blocks until that kernel has completed
// and its writes are visible (a no-op in a kernel launched the ordinary way).  A kernel lets its
// dependents launch once all of its blocks have executed launch_dependents or exited.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// kern<<<grid, block, smem, s>>>(args...), as a programmatic dependent of the kernel before it
// when `pdl` is set
template <typename... KArgs, typename... Args>
static cudaError_t launch_maybe_pdl(bool pdl, void (*kern)(KArgs...), unsigned grid, unsigned block, size_t smem,
                                    cudaStream_t s, Args... args)
{
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(block);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    cfg.attrs = at;
    cfg.numAttrs = pdl ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kern, args...);
}

// ---- blend (frozen definition, DESIGN.md "blend") --------------------------------------------
// weights 1/d2 (exact hits: only d2 == 0 neighbours, weight 1); sums accumulated sequentially
// in neighbour order, fp64, never contracted; colour truncated, normal normalised -> fp32.
struct BlendAcc {
    double s[7];
    __device__ __forceinline__ void reset()
    {
#pragma unroll
        for (int a = 0; a < 7; ++a) s[a] = 0.0;
    }
    __device__ __forceinline__ void add(double w, uint32_t rgba, float nx, float ny, float nz)
    {
        s[0] = __dadd_rn(s[0], w);
        s[1] = __dadd_rn(s[1], __dmul_rn(w, (double)(rgba & 0xffu)));
        s[2] = __dadd_rn(s[2], __dmul_rn(w, (double)((rgba >> 8) & 0xffu)));
        s[3] = __dadd_rn(s[3], __dmul_rn(w, (double)((rgba >> 16) & 0xffu)));
        s[4] = __dadd_rn(s[4], __dmul_rn(w, (double)nx));
        s[5] = __dadd_rn(s[5], __dmul_rn(w, (double)ny));
        s[6] = __dadd_rn(s[6], __dmul_rn(w, (double)nz));
    }
    __device__ __forceinline__ bool weight_ok() const { return s[0] > 0.0 && s[0] < INFINITY; }
    __device__ __forceinline__ void store(uint8_t *rgba_out, float *normal_out) const
    {
        if (rgba_out) {
            int r = __double2int_rz(__ddiv_rn(s[1], s[0]));
            int g = __double2int_rz(__ddiv_rn(s[2], s[0]));
            int b = __double2int_rz(__ddiv_rn(s[3], s[0]));
            uchar4 o;
            o.x = (unsigned char)min(max(r, 0), 255);
            o.y = (unsigned char)min(max(g, 0), 255);
            o.z = (unsigned char)min(max(b, 0), 255);
            o.w = 255;
            *reinterpret_cast<uchar4 *>(rgba_out) = o;
        }
        if (normal_out) {
            double len = __dsqrt_rn(__dadd_rn(
                __dadd_rn(__dmul_rn(s[4], s[4]), __dmul_rn(s[5], s[5])), __dmul_rn(s[6], s[6])));
            if (len > 0.0 && len < INFINITY) {
                normal_out[0] = __double2float_rn(__ddiv_rn(s[4], len));
                normal_out[1] = __double2float_rn(__ddiv_rn(s[5], len));
                normal_out[2] = __double2float_rn(__ddiv_rn(s[6], len));
            } else {
                normal_out[0] = normal_out[1] = normal_out[2] = 0.0f;
            }
        }
    }
};

__device__ __forceinline__ void store_empty_blend(uint8_t *rgba_out, float *normal_out)
{
    if (rgba_out) *reinterpret_cast<uchar4 *>(rgba_out) = make_uchar4(0, 0, 0, 0);
    if (normal_out) normal_out[0] = normal_out[1] = normal_out[2] = 0.0f;
}

struct AttrRaw {   // pt_attr as loaded: 3 floats + packed rgba
    float nx, ny, nz;
    uint32_t rgba;
};
__device__ __forceinline__ AttrRaw load_attr(const pt_attr *p)
{
    int4 v = __ldg(reinterpret_cast<const int4 *>(p));
    AttrRaw a;
    a.nx = __int_as_float(v.x); a.ny = __int_as_float(v.y); a.nz = __int_as_float(v.z);
    a.rgba = (uint32_t)v.w;
    return a;
}
__device__ __forceinline__ void store_cand(pt_cand *dst, double d2, int id, const AttrRaw &a)
{
    // pt_cand: d2 | id | rgba | nx ny nz | pad  -> two 16-byte stores
    int4 lo, hi;
    lo.x = __double2loint(d2); lo.y = __double2hiint(d2); lo.z = id; lo.w = (int)a.rgba;
    hi.x = __float_as_int(a.nx); hi.y = __float_as_int(a.ny); hi.z = __float_as_int(a.nz); hi.w = 0;
    int4 *o = reinterpret_cast<int4 *>(dst);
    o[0] = lo;
    o[1] = hi;
}

// ---- point records ---------------------------------------------------------------------------
template <typename PT> struct PointLoad;
template <> struct PointLoad<PointF> {
    struct Raw { float4 v; };
    static __device__ __forceinline__ Raw load_raw(const void *base, uint32_t i)
    {
        Raw r;
        r.v = __ldg(reinterpret_cast<const float4 *>(base) + i);
        return r;
    }
    static __device__ __forceinline__ void decode(const Raw &r, double &x, double &y, double &z, int &idx)
    {
        x = (double)r.v.x; y = (double)r.v.y; z = (double)r.v.z;
        idx = __float_as_int(r.v.w);
    }
    static __device__ __forceinline__ void load(const void *base, uint32_t i, double &x, double &y,
                                                double &z, int &idx)
    {
        float4 v = __ldg(reinterpret_cast<const float4 *>(base) + i);
        x = (double)v.x; y = (double)v.y; z = (double)v.z;
        idx = __float_as_int(v.w);
    }
};
template <> struct PointLoad<PointD> {
    struct Raw { double2 a, b; };
    static __device__ __forceinline__ Raw load_raw(const void *base, uint32_t i)
    {
        const double2 *p = reinterpret_cast<const double2 *>(base) + 2 * (size_t)i;
        Raw r;
        r.a = __ldg(p); r.b = __ldg(p + 1);
        return r;
    }
    static __device__ __forceinline__ void decode(const Raw &r, double &x, double &y, double &z, int &idx)
    {
        x = r.a.x; y = r.a.y; z = r.b.x;
        idx = __double2loint(r.b.y);
    }
    static __device__ __forceinline__ void load(const void *base, uint32_t i, double &x, double &y,
                                                double &z, int &idx)
    {
        const double2 *p = reinterpret_cast<const double2 *>(base) + 2 * (size_t)i;
        double2 a = __ldg(p), b = __ldg(p + 1);
        x = a.x; y = a.y; z = b.x;
        idx = __double2loint(b.y);
    }
};

__device__ __forceinline__ Box load_box(const Box *p)
{
    const int4 *bp = reinterpret_cast<const int4 *>(p);
    int4 b0 = __ldg(bp), b1 = __ldg(bp + 1);
    Box b;
    b.lox = __int_as_float(b0.x); b.loy = __int_as_float(b0.y);
    b.loz = __int_as_float(b0.z); b.hix = __int_as_float(b0.w);
    b.hiy = __int_as_float(b1.x); b.hiz = __int_as_float(b1.y);
    b.pad0 = 0.f; b.pad1 = 0.f;
    return b;
}

// ==============================================================================================
// Variant 0: warp per sample (also the overflow fallback and the K5 merge building block)
// ==============================================================================================
struct WarpList {
    double d;     // lane j holds the j-th best (ascending); +inf when empty
    int    i;     // local point index; IDX_NONE when empty
    double kd;    // replicated: current k-th entry (the acceptance threshold)
    int    ki;
};

__device__ __forceinline__ double shfl_f64(double v, int src)
{
    return __shfl_sync(0xffffffffu, v, src);
}

// Offer one candidate per lane (pass = lane has a candidate that beats the k-th entry).
// `tag` rides along with the entry (merge kernel: where the candidate came from).
// DEDUPE: skip a candidate whose id is already in the list (slab indexes that carry ghost
// points can return the same global point from two ranks).
template <bool DEDUPE = false>
__device__ __forceinline__ void warp_list_offer(WarpList &L, int &tag_list, int k, unsigned lane,
                                                bool pass, double d, int idx, int tag)
{
    unsigned m = __ballot_sync(0xffffffffu, pass);
    while (m) {
        int c = __ffs(m) - 1;
        m &= m - 1;
        double cd = shfl_f64(d, c);
        int ci = __shfl_sync(0xffffffffu, idx, c);
        int ct = __shfl_sync(0xffffffffu, tag, c);
        if (!key_less(cd, ci, L.kd, L.ki)) continue;  // threshold moved since the ballot
        if (DEDUPE && __any_sync(0xffffffffu, L.i == ci)) continue;
        unsigned before = __ballot_sync(0xffffffffu, key_less(L.d, L.i, cd, ci));
        unsigned pos = __popc(before);
        double ud = __shfl_up_sync(0xffffffffu, L.d, 1);
        int ui = __shfl_up_sync(0xffffffffu, L.i, 1);
        int ut = __shfl_up_sync(0xffffffffu, tag_list, 1);
        if (lane > pos) { L.d = ud; L.i = ui; tag_list = ut; }
        else if (lane == pos) { L.d = cd; L.i = ci; tag_list = ct; }
        L.kd = shfl_f64(L.d, k - 1);
        L.ki = __shfl_sync(0xffffffffu, L.i, k - 1);
    }
}

// Sequential (neighbour-order) blend of a lane-distributed list; every lane runs the same sums.
__device__ __forceinline__ void warp_blend_store(unsigned lane, int k, bool has, double d2,
                                                 const AttrRaw &at, uint8_t *rgba_out,
                                                 float *normal_out)
{
    unsigned any = __ballot_sync(0xffffffffu, has);
    if (any == 0) {
        if (lane == 0) store_empty_blend(rgba_out, normal_out);
        return;
    }
    const int cnt = __popc(any);   // valid entries are a prefix of the lanes
    int mode = shfl_f64(d2, 0) == 0.0 ? 1 : 0;
    BlendAcc acc;
    for (int pass = 0; pass < 2; ++pass) {
        acc.reset();
        for (int j = 0; j < cnt; ++j) {
            double dj = shfl_f64(d2, j);
            uint32_t cj = __shfl_sync(0xffffffffu, at.rgba, j);
            float nx = __shfl_sync(0xffffffffu, at.nx, j);
            float ny = __shfl_sync(0xffffffffu, at.ny, j);
            float nz = __shfl_sync(0xffffffffu, at.nz, j);
            acc.add(blend_weight(mode, dj, j), cj, nx, ny, nz);
        }
        if (acc.weight_ok()) break;
        mode = 2;
    }
    (void)k;
    if (lane == 0) acc.store(rgba_out, normal_out);
}

constexpr int WARPS_PER_BLOCK = 8;

template <typename PT>
__device__ __forceinline__ void warp_query(const QueryParams &P, uint32_t q, unsigned lane,
                                           float (*s_lb)[32])
{
    const int k = P.k;
    const double qx = __ldg(P.queries + 3 * (size_t)q);
    const double qy = __ldg(P.queries + 3 * (size_t)q + 1);
    const double qz = __ldg(P.queries + 3 * (size_t)q + 2);
    const float qdn[3] = {__double2float_rd(qx), __double2float_rd(qy), __double2float_rd(qz)};
    const float qup[3] = {__double2float_ru(qx), __double2float_ru(qy), __double2float_ru(qz)};
    const double r2 = P.r2_per_query ? __ldg(P.r2_per_query + q) : P.r2;

    WarpList L;
    L.d = INFINITY; L.i = IDX_NONE; L.kd = INFINITY; L.ki = IDX_NONE;
    int tag = 0;
    float bound = __double2float_ru(r2);   // prune a box iff its lower bound > bound

    // per-level traversal state: lane l keeps level l's group id and pending-children mask
    uint32_t st_group = 0, st_mask = 0;
    int lvl = P.w_levels - 1;

    auto enter = [&](int level, uint32_t group) {
        const int pl = level * WLOG;
        const uint32_t node = group * 32 + lane;
        float lb = INFINITY;
        bool valid = node < P.pyr.count[pl];
        if (valid) lb = box_lower_bound(qdn, qup, load_box(P.pyr.level[pl] + node));
        s_lb[level][lane] = lb;
        unsigned mask = __ballot_sync(0xffffffffu, valid && lb <= bound);
        if (lane == (unsigned)level) { st_group = group; st_mask = mask; }
    };

    if (lvl >= 0) enter(lvl, 0);
    while (lvl < P.w_levels && lvl >= 0) {
        unsigned mask = __shfl_sync(0xffffffffu, st_mask, lvl);
        if (mask == 0) { ++lvl; continue; }
        // nearest pending child first
        float lb = s_lb[lvl][lane];
        unsigned bits = ((mask >> lane) & 1u) ? __float_as_uint(lb) : 0xffffffffu;
        unsigned mn = __reduce_min_sync(0xffffffffu, bits);
        if (__uint_as_float(mn) > bound) {  // nearest pending child is already too far
            if (lane == (unsigned)lvl) st_mask = 0;
            ++lvl;
            continue;
        }
        int c = __ffs(__ballot_sync(0xffffffffu, bits == mn)) - 1;
        if (lane == (unsigned)lvl) st_mask = mask & ~(1u << c);
        uint32_t node = __shfl_sync(0xffffffffu, st_group, lvl) * 32 + c;
        if (lvl > 0) {
            --lvl;
            enter(lvl, node);
            continue;
        }
        // leaf scan: one point per lane, exact metric (src/Distance.h:6-11)
        uint32_t i = node * LEAF + lane;
        double px, py, pz;
        int pidx;
        PointLoad<PT>::load(P.pts, i, px, py, pz, pidx);
        double d = dist2_exact(qx, qy, qz, px, py, pz);
        bool pass = i < P.n && d <= r2 && key_less(d, pidx, L.kd, L.ki);
        warp_list_offer(L, tag, k, lane, pass, d, pidx, 0);
        bound = __double2float_ru(fmin(L.kd, r2));
    }

    // outputs
    bool has = lane < (unsigned)k && L.i != IDX_NONE;
    int gid = has ? (P.ids ? __ldg(P.ids + L.i) : L.i) : -1;
    bool need_attr = (P.rgba_out || P.normal_out || P.cand_out) && P.attrs;
    AttrRaw at{0.f, 0.f, 0.f, 0u};
    if (need_attr && has) at = load_attr(P.attrs + L.i);
    if (lane < (unsigned)k) {
        size_t o = (size_t)q * k + lane;
        if (P.idx_out) P.idx_out[o] = gid;
        if (P.d2_out) P.d2_out[o] = has ? L.d : INFINITY;
        if (P.cand_out) store_cand(P.cand_out + o, has ? L.d : INFINITY, gid, at);
    }
    if (P.rgba_out || P.normal_out)
        warp_blend_store(lane, k, has, L.d, at, P.rgba_out ? P.rgba_out + 4 * (size_t)q : nullptr,
                         P.normal_out ? P.normal_out + 3 * (size_t)q : nullptr);
}

template <typename PT>
__global__ void __launch_bounds__(WARPS_PER_BLOCK * 32) knn_warp_kernel(const QueryParams P)
{
    __shared__ float s_lb[WARPS_PER_BLOCK][MAX_W_LEVELS][32];
    const unsigned lane = threadIdx.x & 31;
    const unsigned wib = threadIdx.x >> 5;
    const uint32_t q = blockIdx.x * WARPS_PER_BLOCK + wib;
    if (q >= P.m) return;
    warp_query<PT>(P, q, lane, s_lb[wib]);
}

// Re-runs the samples listed by the thread kernel (queue overflow), grid-stride over the list.
// Launched as a programmatic dependent: it lets the next kernel of the chain launch at once (its
// blocks wait for this grid to complete) and waits for the kernel that wrote the list.
template <typename PT>
__global__ void __launch_bounds__(WARPS_PER_BLOCK * 32)
knn_warp_list_kernel(const QueryParams P, const uint32_t *count, const uint32_t *list,
                     uint32_t *stat_out, const uint32_t *count_stage1, uint32_t only_up_to)
{
    __shared__ float s_lb[WARPS_PER_BLOCK][MAX_W_LEVELS][32];
    const unsigned lane = threadIdx.x & 31;
    const unsigned wib = threadIdx.x >> 5;
    pdl_launch_dependents();
    pdl_wait();
    uint32_t n = min(*count, P.m);
    if (stat_out && blockIdx.x == 0 && threadIdx.x == 0) {   // pt_index_info / pt_index_fallback_counts
        stat_out[0] = n;
        stat_out[1] = count_stage1 ? *count_stage1 : 0u;
    }
    if (n > only_up_to) return;          // a long list belongs to the scan / thread kernel
    for (uint32_t w = blockIdx.x * WARPS_PER_BLOCK + wib; w < n; w += gridDim.x * WARPS_PER_BLOCK)
        warp_query<PT>(P, list[w], lane, s_lb[wib]);
}

__global__ void __launch_bounds__(256) empty_result_kernel(const QueryParams P)
{
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    size_t total = (size_t)P.m * P.k;
    if (i < total) {
        if (P.idx_out) P.idx_out[i] = -1;
        if (P.d2_out) P.d2_out[i] = INFINITY;
        if (P.cand_out) store_cand(P.cand_out + i, INFINITY, -1, AttrRaw{0.f, 0.f, 0.f, 0u});
    }
    if (i < P.m) store_empty_blend(P.rgba_out ? P.rgba_out + 4 * i : nullptr,
                                   P.normal_out ? P.normal_out + 3 * i : nullptr);
}

}  // namespace pt
#include "pt_knn_traverse.cuh"
#include "pt_knn_thread.cuh"
#include "pt_knn_scan.cuh"
#include "pt_knn_grid.cuh"
#include "pt_knn_span.cuh"
namespace pt {

// Block runs (pt_knn_span.cuh) for the level a k = 16 search plans its first attempt on, when that
// attempt is one the span kernel runs (a 3^3 block expected to fit a half-warp).  Count pass,
// exclusive scan, fill pass.  The runs store each point once per block that holds it (about nine
// times the cloud's records on a scanned surface), so they are built only when table and runs fit
// a quarter of the device memory free at this point -- the rest stays for the queries'
// workspaces, the normals' lists and a second index -- and their offsets fit 32 bits of 16-byte
// units.  Otherwise the index has none and every query stages spans as before.
constexpr size_t BLOCK_FREE_SHARE = 4;    // the runs may take 1 / this of the free device memory

int build_blocks(pt_index *ix)
{
    ix->blk_mem = nullptr;
    ix->blk_bytes = 0;
    GridParams gp;
    if (ix->coord_f64 || grid_plan(ix, 16, INFINITY, gp) == 0 || gp.att_rc[0] != 1 ||
        gp.expect_cand > 0.74f * (float)PAIR_CAP)
        return PT_OK;
    cudaStream_t s = ix->stream;
    const GridTable T = gp.tab[gp.att_tab[0]];
    const uint64_t cells = ix->level_cells[T.level];
    const uint64_t tab_cap = (3 * cells + 8) & ~3ull;           // load <= 1/3, whole 4-slot groups
    if (tab_cap > 0xfffffff0ull) return PT_OK;
    const PointF *pts = reinterpret_cast<const PointF *>(ix->pts);
    const unsigned blocks = (unsigned)(((uint64_t)T.cap * 16 + 255) / 256);
    // units[b]: 16-byte units of bucket b's runs; off = their exclusive sum, off[cap] = all units
    unsigned long long *units = nullptr;
    PT_TRY(pool_alloc((void **)&units, sizeof(unsigned long long) * 2 * ((size_t)T.cap + 1), s));
    unsigned long long *off = units + T.cap + 1;
    struct Free {
        void *p; cudaStream_t s;
        ~Free() { pool_free(p, s); }
    } units_guard{units, s};
    PT_CUDA(cudaMemsetAsync(units + T.cap, 0, sizeof(unsigned long long), s));
    block_run_kernel<true><<<blocks, 256, 0, s>>>(T, units, nullptr, pts, nullptr, nullptr, 0);
    count_launch();
    PT_CUDA(cudaGetLastError());
    size_t tmp_bytes = 0;
    PT_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, units, off, (int)T.cap + 1, s));
    void *tmp = nullptr;
    PT_TRY(pool_alloc(&tmp, tmp_bytes, s));
    const cudaError_t e = cub::DeviceScan::ExclusiveSum(tmp, tmp_bytes, units, off, (int)T.cap + 1, s);
    pool_free(tmp, s);
    PT_CUDA(e);
    unsigned long long total_units = 0;
    PT_CUDA(cudaMemcpyAsync(&total_units, off + T.cap, sizeof total_units, cudaMemcpyDeviceToHost, s));
    PT_CUDA(cudaStreamSynchronize(s));
    const size_t tab_bytes = sizeof(BlockSlot) * tab_cap, bytes = tab_bytes + sizeof(uint4) * total_units;
    size_t free_b = 0, total_b = 0;
    PT_CUDA(cudaMemGetInfo(&free_b, &total_b));
    if (verbose())
        fprintf(stderr, "[points_transfer] block runs level %d: %llu cells, %llu units, %.3f GB (free %.3f GB)\n",
                T.level, (unsigned long long)cells, total_units, (double)bytes * 1e-9, (double)free_b * 1e-9);
    if (total_units > 0xffffffffull || bytes > free_b / BLOCK_FREE_SHARE) return PT_OK;
    void *mem = nullptr;
    PT_TRY(pool_alloc(&mem, bytes, s));
    ix->blk_mem = mem;
    ix->blk_bytes = bytes;
    BlockSlot *tab = reinterpret_cast<BlockSlot *>(mem);
    uint4 *runs = reinterpret_cast<uint4 *>(reinterpret_cast<char *>(mem) + tab_bytes);
    PT_CUDA(cudaMemsetAsync(tab, 0xff, tab_bytes, s));
    block_run_kernel<false><<<blocks, 256, 0, s>>>(T, nullptr, off, pts, runs, tab, (uint32_t)tab_cap);
    count_launch();
    PT_CUDA(cudaGetLastError());
    ix->grid.blk = tab;
    ix->grid.blk_runs = runs;
    ix->grid.blk_cap = (uint32_t)tab_cap;
    ix->grid.blk_level = T.level;
    return PT_OK;
}

// Launch plan.  Every launch gets its OWN hand-over workspace (two sample lists with their
// counters) from the library's stream-ordered pool, so launches of one index that are in flight
// on different streams never share state:
//   grid kernel          --(samples it cannot prove final: list 1)-->
//   scan / thread kernel --(samples whose queue proof obligation failed: list 2)-->
//   warp kernel over list 2.
constexpr uint32_t SHORT_LIST = 2048;   // hand-over lists up to this size go to the warp kernel

template <typename PT>
static int launch_chain(pt_index *ix, const QueryParams &qp, int variant, cudaStream_t s)
{
    uint32_t *ws = nullptr;
    PT_TRY(pool_alloc((void **)&ws, sizeof(uint32_t) * (8 + 2 * (size_t)qp.m), s));
    // ws[1]: the span kernel's pair-claim counter, zeroed with the two list counters
    uint32_t *count1 = ws, *count2 = ws + 4, *list1 = ws + 8, *list2 = list1 + qp.m;
    int rc = PT_OK;
    cudaError_t e = cudaMemsetAsync(ws, 0, 8 * sizeof(uint32_t), s);     // both counters at once
    if (e != cudaSuccess) rc = map_cuda_error(e);
    QueryParams q2 = qp;
    const bool grid_first = variant == 6;
    // Behind a grid kernel the three hand-over kernels are programmatic dependents: each launches
    // while the kernel ahead of it still runs and waits (griddepcontrol.wait) before it reads a
    // counter or a list.  Most launches hand nothing over, and the three then only read a counter.
    const bool pdl = grid_first && opt_chain_pdl() != 0;
    if (rc == PT_OK && variant == 6) {
        // two samples per warp with one look-up per parent cell and one copy per span where the
        // pair kernel would run (pt_knn_span.cuh); otherwise launch_grid picks
        const bool span = grid_span_applies<PT>(qp);
        const bool block = span && grid_block_applies(qp);
        note_grid_span_used(span ? 1 : 0);
        note_grid_block_used(block ? 1 : 0);
        if (span) {
            note_grid_pair_used(0);
            rc = launch_grid_span(qp, block, ix->sm_count, count1, list1, ws + 1, s);
        } else {
            rc = launch_grid<PT>(qp, ix->sm_count, count1, list1, s);
        }
        // A short hand-over list is answered by the warp kernel (one warp per sample: a few
        // samples cost ~30 us there, but a whole ~110 us block latency in the scan / thread
        // kernels); a long one by the scan / thread kernel in list mode (min_count).
        if (rc == PT_OK) {
            e = launch_maybe_pdl(pdl, knn_warp_list_kernel<PT>, ix->sm_count * 4, WARPS_PER_BLOCK * 32, 0, s, qp,
                                 (const uint32_t *)count1, (const uint32_t *)list1, (uint32_t *)nullptr,
                                 (const uint32_t *)nullptr, SHORT_LIST);
            count_launch();
            if (e != cudaSuccess) rc = map_cuda_error(e);
        }
        q2.qlist = list1;
        q2.qcount = count1;
        q2.qlist_min = SHORT_LIST + 1;
        const bool bounded = qp.r2_per_query != nullptr || qp.r2 < INFINITY;
        variant = (qp.k > 16 || !bounded) ? 5 : 2;
    }
    if (rc == PT_OK)
        rc = variant == 5 ? launch_scan<PT>(q2, ix->sm_count, pdl, count2, list2, s)
                          : launch_thread<PT>(q2, ix->sm_count, pdl, count2, list2, s);
    if (rc == PT_OK) {
        e = launch_maybe_pdl(pdl, knn_warp_list_kernel<PT>, ix->sm_count * 4, WARPS_PER_BLOCK * 32, 0, s, qp,
                             (const uint32_t *)count2, (const uint32_t *)list2, ix->fallback_word,
                             (const uint32_t *)(grid_first ? count1 : nullptr), 0xffffffffu);
        count_launch();
        if (e != cudaSuccess) rc = map_cuda_error(e);
    }
    pool_free(ws, s);
    return rc;
}

int launch_query(pt_index *ix, const QueryParams &qp_in, cudaStream_t s)
{
    if (qp_in.m == 0) return PT_OK;
    if (qp_in.k < 1 || qp_in.k > PT_MAX_K) return PT_ERR_UNSUPPORTED;
    QueryParams qp = qp_in;
    qp.qlist = nullptr;
    qp.qcount = nullptr;
    qp.qlist_min = 0;
    if (ix->n == 0) {
        size_t total = (size_t)qp.m * qp.k;
        empty_result_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(qp);
        count_launch();
        PT_CUDA(cudaGetLastError());
        return PT_OK;
    }
    int variant = opt_knn_variant();
    const bool bounded = qp.r2_per_query != nullptr || qp.r2 < INFINITY;
    const bool have_grid = (variant < 0 || variant == 6) && grid_plan(ix, qp.k, qp.r2, qp.grid) > 0;
    if (!have_grid) qp.grid.n_attempts = 0;
    if (have_grid && verbose()) {
        fprintf(stderr, "[points_transfer] grid plan k=%d:", qp.k);
        for (int a = 0; a < qp.grid.n_attempts; ++a) {
            const int L = qp.grid.tab[qp.grid.att_tab[a]].level;
            fprintf(stderr, " (level %d, rc %d, occ %.1f)", L, (int)qp.grid.att_rc[a],
                    (double)ix->n / (double)ix->level_cells[L]);
        }
        fprintf(stderr, "; ~%.0f candidates expected in the first\n", (double)qp.grid.expect_cand);
    }
    if (variant == 6 && !have_grid) variant = -1;
    if (variant < 0) {
        // auto (measured, DESIGN.md section 4): the grid kernel first whenever the index has
        // cell tables.  Without them (tiny clouds, kd-refined order):
        //  * up to ~12 k samples a launch is one partial wave and pays a thread-kernel block's
        //    full latency; the warp kernel -- 32 lanes per sample -- answers it sooner;
        //  * the scan kernel is 3-9 % ahead of the thread kernel on launches that fill the GPU
        //    and 23 % at k = 32;
        //  * on mid-size launches, on radius-bounded searches, which mostly end with short
        //    lists, and on slab indexes with an id map the thread kernel wins at k <= 16.
        if (have_grid) variant = 6;
        else if (qp.m <= 12288u) variant = 0;
        else variant = (qp.k > 16 || (!bounded && qp.m >= 100000u && qp.ids == nullptr)) ? 5 : 2;
    }
    if (variant == 0) {
        unsigned blocks = (qp.m + WARPS_PER_BLOCK - 1) / WARPS_PER_BLOCK;
        if (ix->coord_f64)
            knn_warp_kernel<PointD><<<blocks, WARPS_PER_BLOCK * 32, 0, s>>>(qp);
        else
            knn_warp_kernel<PointF><<<blocks, WARPS_PER_BLOCK * 32, 0, s>>>(qp);
        count_launch();
        PT_CUDA(cudaGetLastError());
        return PT_OK;
    }
    return ix->coord_f64 ? launch_chain<PointD>(ix, qp, variant, s) : launch_chain<PointF>(ix, qp, variant, s);
}

// ---- K5: merge per-slab candidate lists (multi-GPU exchange epilogue) -------------------------
__global__ void __launch_bounds__(WARPS_PER_BLOCK * 32)
merge_kernel(const pt_cand *lists, int n_lists, uint32_t m, int k, int32_t *idx_out,
             double *d2_out, uint8_t *rgba_out, float *normal_out, pt_cand *cand_out)
{
    const unsigned lane = threadIdx.x & 31;
    const uint32_t q = blockIdx.x * WARPS_PER_BLOCK + (threadIdx.x >> 5);
    if (q >= m) return;
    WarpList L;
    L.d = INFINITY; L.i = IDX_NONE; L.kd = INFINITY; L.ki = IDX_NONE;
    int src = -1;  // where this lane's entry came from: list * 32 + slot
    for (int l = 0; l < n_lists; ++l) {
        const pt_cand *c = lists + ((size_t)l * m + q) * k + lane;
        double d = INFINITY;
        int id = IDX_NONE;
        if (lane < (unsigned)k) {
            d = c->d2;
            id = c->id;
            if (id < 0) { id = IDX_NONE; d = INFINITY; }
        }
        bool pass = id != IDX_NONE && key_less(d, id, L.kd, L.ki);
        warp_list_offer<true>(L, src, k, lane, pass, d, id, l * 32 + (int)lane);
    }
    bool has = lane < (unsigned)k && L.i != IDX_NONE;
    AttrRaw at{0.f, 0.f, 0.f, 0u};
    if (has) {
        const pt_cand *c = lists + ((size_t)(src >> 5) * m + q) * k + (src & 31);
        at.nx = c->nx; at.ny = c->ny; at.nz = c->nz;
        at.rgba = (uint32_t)c->r | ((uint32_t)c->g << 8) | ((uint32_t)c->b << 16) | ((uint32_t)c->a << 24);
    }
    if (lane < (unsigned)k) {
        size_t o = (size_t)q * k + lane;
        if (idx_out) idx_out[o] = has ? L.i : -1;
        if (d2_out) d2_out[o] = has ? L.d : INFINITY;
        if (cand_out) store_cand(cand_out + o, has ? L.d : INFINITY, has ? L.i : -1, at);
    }
    if (rgba_out || normal_out)
        warp_blend_store(lane, k, has, L.d, at, rgba_out ? rgba_out + 4 * (size_t)q : nullptr,
                         normal_out ? normal_out + 3 * (size_t)q : nullptr);
}

int launch_merge(const pt_cand *lists, int n_lists, uint32_t m, int k, int32_t *idx_out,
                 double *d2_out, uint8_t *rgba_out, float *normal_out, pt_cand *cand_out,
                 cudaStream_t s)
{
    if (m == 0) return PT_OK;
    if (k < 1 || k > PT_MAX_K || n_lists < 1) return PT_ERR_UNSUPPORTED;
    unsigned blocks = (m + WARPS_PER_BLOCK - 1) / WARPS_PER_BLOCK;
    merge_kernel<<<blocks, WARPS_PER_BLOCK * 32, 0, s>>>(lists, n_lists, m, k, idx_out, d2_out,
                                                         rgba_out, normal_out, cand_out);
    count_launch();
    PT_CUDA(cudaGetLastError());
    return PT_OK;
}

// ---- halo exchange kernels (multi-GPU, DESIGN.md section 6) -------------------------------------
// Fixed-capacity routing so the whole exchange runs without a host synchronisation: every rank
// keeps, per peer, a send block of (cap + 1) rows of 4 doubles -- row 0 is the header
// (count, overflow flag), rows 1.. are (x, y, z, bound) of the samples whose k-th-neighbour ball
// reaches that peer's slab box -- plus the sample index of each row.
__global__ void __launch_bounds__(256)
halo_route_kernel(const double *q, const pt_cand *own, uint32_t m, int k, double r2,
                  const double *boxes, int n_ranks, int self, uint32_t cap, double *send,
                  int32_t *sel, uint32_t *counts)
{
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= m) return;
    const double x = q[3 * (size_t)s], y = q[3 * (size_t)s + 1], z = q[3 * (size_t)s + 2];
    if (x != x) return;                       // NaN row: an unused slot of a routing block
    const double bound = fmin(own[(size_t)s * k + (k - 1)].d2, r2);   // +inf while the list is short
    for (int r = 0; r < n_ranks; ++r) {
        if (r == self) continue;
        const double *b = boxes + 6 * r;
        const double ex = fmax(fmax(b[0] - x, x - b[3]), 0.0);
        const double ey = fmax(fmax(b[1] - y, y - b[4]), 0.0);
        const double ez = fmax(fmax(b[2] - z, z - b[5]), 0.0);
        // shrunk by 1e-12 relative so rounding can never exclude a slab that holds a neighbour
        const double lb = (ex * ex + ey * ey + ez * ez) * (1.0 - 1e-12);
        if (lb <= bound && lb < INFINITY) {   // an empty slab has an inverted box: lb = inf
            const uint32_t pos = atomicAdd(&counts[r], 1u);
            if (pos < cap) {
                double *row = send + ((size_t)r * (cap + 1) + 1 + pos) * 4;
                row[0] = x; row[1] = y; row[2] = z; row[3] = bound;
                sel[(size_t)r * cap + pos] = (int32_t)s;
            }
        }
    }
}

__global__ void halo_header_kernel(const uint32_t *counts, int n_ranks, uint32_t cap, double *send,
                                   uint32_t *overflow_flag)
{
    const int r = threadIdx.x;
    if (r >= n_ranks) return;
    const uint32_t c = counts[r];
    double *row = send + (size_t)r * (cap + 1) * 4;
    row[0] = (double)(c < cap ? c : cap);
    row[1] = c > cap ? 1.0 : 0.0;
    row[2] = 0.0; row[3] = 0.0;
    if (c > cap) atomicOr(overflow_flag, 1u);
}

// Received blocks -> query rows for the bounded halo search; rows past a block's count get a
// negative bound, which the query kernels treat as "no candidates" at once.
__global__ void __launch_bounds__(256)
halo_prepare_kernel(const double *recv, int n_ranks, uint32_t cap, double *q_out, double *r2_out)
{
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (uint32_t)n_ranks * cap) return;
    const uint32_t r = t / cap, j = t % cap;
    const double *blk = recv + (size_t)r * (cap + 1) * 4;
    const bool valid = (double)j < blk[0];
    const double *row = blk + (size_t)(1 + j) * 4;
    q_out[3 * (size_t)t] = valid ? row[0] : 0.0;
    q_out[3 * (size_t)t + 1] = valid ? row[1] : 0.0;
    q_out[3 * (size_t)t + 2] = valid ? row[2] : 0.0;
    r2_out[t] = valid ? row[3] : -1.0;
}

// Merges one peer's returned candidate lists into the owner's lists (in place) and re-blends.
// One warp per routed sample; count_ptr is the device-side number of rows sent to that peer.
__global__ void __launch_bounds__(WARPS_PER_BLOCK * 32)
halo_merge_kernel(pt_cand *own, const pt_cand *back, const int32_t *sel, const uint32_t *count_ptr,
                  uint32_t cap, int k, int32_t *idx_out, double *d2_out, uint8_t *rgba_out,
                  float *normal_out)
{
    const unsigned lane = threadIdx.x & 31;
    const uint32_t j = blockIdx.x * WARPS_PER_BLOCK + (threadIdx.x >> 5);
    const uint32_t cnt = min(*count_ptr, cap);
    if (j >= cnt) return;
    const uint32_t q = (uint32_t)sel[j];
    WarpList L;
    L.d = INFINITY; L.i = IDX_NONE; L.kd = INFINITY; L.ki = IDX_NONE;
    int src = -1;
    const pt_cand *lists[2] = {own + (size_t)q * k, back + (size_t)j * k};
    for (int l = 0; l < 2; ++l) {
        double d = INFINITY;
        int id = IDX_NONE;
        if (lane < (unsigned)k) {
            d = lists[l][lane].d2;
            id = lists[l][lane].id;
            if (id < 0) { id = IDX_NONE; d = INFINITY; }
        }
        bool pass = id != IDX_NONE && key_less(d, id, L.kd, L.ki);
        warp_list_offer<true>(L, src, k, lane, pass, d, id, l * 32 + (int)lane);
    }
    const bool has = lane < (unsigned)k && L.i != IDX_NONE;
    AttrRaw at{0.f, 0.f, 0.f, 0u};
    if (has) {
        const pt_cand *c = lists[src >> 5] + (src & 31);
        at.nx = c->nx; at.ny = c->ny; at.nz = c->nz;
        at.rgba = (uint32_t)c->r | ((uint32_t)c->g << 8) | ((uint32_t)c->b << 16) | ((uint32_t)c->a << 24);
    }
    __syncwarp();   // every lane has read its source record before the in-place update below
    if (lane < (unsigned)k) {
        const size_t o = (size_t)q * k + lane;
        store_cand(own + o, has ? L.d : INFINITY, has ? L.i : -1, at);
        if (idx_out) idx_out[o] = has ? L.i : -1;
        if (d2_out) d2_out[o] = has ? L.d : INFINITY;
    }
    if (rgba_out || normal_out)
        warp_blend_store(lane, k, has, L.d, at, rgba_out ? rgba_out + 4 * (size_t)q : nullptr,
                         normal_out ? normal_out + 3 * (size_t)q : nullptr);
}

// Ghost-zone check (DESIGN.md section 6): flags the step if some sample's k-th-neighbour ball
// both reaches another slab's box and may stick out of the ghost zone around this slab.
__global__ void __launch_bounds__(256)
ghost_check_kernel(const double *q, const double *d2, uint32_t m, int k, double r2,
                   const double *boxes, int n_ranks, int self, double halo, uint32_t *flag)
{
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    bool viol = false;
    if (s < m && q[3 * (size_t)s] == q[3 * (size_t)s]) {     // NaN row: an unused slot of a routing block
        const double x = q[3 * (size_t)s], y = q[3 * (size_t)s + 1], z = q[3 * (size_t)s + 2];
        const double bound = fmin(d2[(size_t)s * k + (k - 1)], r2);
        const double *ob = boxes + 6 * self;
        const double ox = fmax(fmax(ob[0] - x, x - ob[3]), 0.0);
        const double oy = fmax(fmax(ob[1] - y, y - ob[4]), 0.0);
        const double oz = fmax(fmax(ob[2] - z, z - ob[5]), 0.0);
        const bool leaves = (sqrt(bound) + sqrt(ox * ox + oy * oy + oz * oz)) * (1.0 + 1e-9) > halo;
        if (leaves) {
            for (int r = 0; r < n_ranks && !viol; ++r) {
                if (r == self) continue;
                const double *b = boxes + 6 * r;
                const double ex = fmax(fmax(b[0] - x, x - b[3]), 0.0);
                const double ey = fmax(fmax(b[1] - y, y - b[4]), 0.0);
                const double ez = fmax(fmax(b[2] - z, z - b[5]), 0.0);
                const double lb = (ex * ex + ey * ey + ez * ez) * (1.0 - 1e-12);
                viol = lb <= bound && lb < INFINITY;
            }
        }
    }
    if (__any_sync(0xffffffffu, viol) && (threadIdx.x & 31) == 0) atomicOr(flag, 1u);
}

// ---- sample routing for slab-sharded clouds (DESIGN.md section 6) --------------------------------
// Samples arrive in arbitrary order on any rank; the slab that owns a sample is the one whose
// x-range [cuts[r], cuts[r + 1]) holds it.  Fixed-capacity blocks per destination, so the
// all_to_all that follows needs no host synchronisation: row = (x, y, z, +inf) -- the 4th word
// is the per-query squared bound of pt_query_device -- and rows past a block's count keep the
// NaN bound the caller memsets (0xff), which every query kernel answers with an empty list.
// Row numbers come from three levels of counting, so that half a million samples do not queue
// up on n_ranks global counters (one atomic per sample: 200 us at 2 ranks): lanes with the same
// destination are ranked by __match_any_sync, warps add to the block's shared counters, and one
// thread per destination reserves the block's range with a single global atomic.
constexpr int ROUTE_SMEM_RANKS = 64;
__global__ void __launch_bounds__(256)
route_samples_kernel(const double *q, uint32_t m, const double *cuts, int n_ranks, uint32_t cap,
                     double *send, int32_t *sel, uint32_t *counts, uint32_t *overflow_flag)
{
    __shared__ uint32_t s_cnt[ROUTE_SMEM_RANKS], s_base[ROUTE_SMEM_RANKS];
    const bool block_level = n_ranks <= ROUTE_SMEM_RANKS;
    const unsigned lane = threadIdx.x & 31;
    if (block_level) {
        if (threadIdx.x < ROUTE_SMEM_RANKS) s_cnt[threadIdx.x] = 0;
        __syncthreads();
    }
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    const bool valid = s < m;
    double x = 0.0;
    int lo = 0;
    if (valid) {
        x = q[3 * (size_t)s];
        int hi = n_ranks - 1;                    // last r with cuts[r] <= x (cuts[0] = -inf)
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (cuts[mid] <= x) lo = mid; else hi = mid - 1;
        }
    }
    const unsigned peers = __match_any_sync(0xffffffffu, valid ? lo : -1);
    const int leader = __ffs(peers) - 1;
    const uint32_t in_warp = (uint32_t)__popc(peers & ((1u << lane) - 1u));
    uint32_t wbase = 0;
    if (valid && (int)lane == leader)
        wbase = block_level ? atomicAdd(&s_cnt[lo], (uint32_t)__popc(peers))
                            : atomicAdd(&counts[lo], (uint32_t)__popc(peers));
    wbase = __shfl_sync(0xffffffffu, wbase, leader);
    uint32_t pos = wbase + in_warp;
    if (block_level) {
        __syncthreads();
        if ((int)threadIdx.x < n_ranks)
            s_base[threadIdx.x] = s_cnt[threadIdx.x] ? atomicAdd(&counts[threadIdx.x], s_cnt[threadIdx.x]) : 0u;
        __syncthreads();
        pos += s_base[lo];
    }
    if (!valid) return;
    if (pos >= cap) { atomicOr(overflow_flag, 1u); return; }
    double *row = send + ((size_t)lo * cap + pos) * 4;
    row[0] = x; row[1] = q[3 * (size_t)s + 1]; row[2] = q[3 * (size_t)s + 2]; row[3] = INFINITY;
    sel[(size_t)lo * cap + pos] = (int32_t)s;
}

// dst[sel[t]] = src[t] for every row t with sel[t] >= 0; rows are row_words 4-byte words.
__global__ void __launch_bounds__(256)
scatter_rows_kernel(const uint32_t *src, const int32_t *sel, uint32_t rows, uint32_t row_words,
                    uint32_t *dst)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)rows * row_words) return;
    const uint32_t t = (uint32_t)(i / row_words), w = (uint32_t)(i % row_words);
    const int32_t d = sel[t];
    if (d >= 0) dst[(size_t)d * row_words + w] = src[i];
}

int launch_route_samples(const double *q, uint32_t m, const double *cuts, int n_ranks, uint32_t cap,
                         double *send, int32_t *sel, uint32_t *counts, uint32_t *overflow_flag,
                         cudaStream_t s)
{
    if (n_ranks < 1 || n_ranks > 4096 || cap == 0) return PT_ERR_INVALID_ARG;
    const size_t rows = (size_t)n_ranks * cap;
    PT_CUDA(cudaMemsetAsync(send, 0xff, sizeof(double) * 4 * rows, s));       // NaN rows
    PT_CUDA(cudaMemsetAsync(sel, 0xff, sizeof(int32_t) * rows, s));           // -1
    PT_CUDA(cudaMemsetAsync(counts, 0, sizeof(uint32_t) * n_ranks, s));
    PT_CUDA(cudaMemsetAsync(overflow_flag, 0, sizeof(uint32_t), s));
    if (m) {
        route_samples_kernel<<<(m + 255) / 256, 256, 0, s>>>(q, m, cuts, n_ranks, cap, send, sel, counts,
                                                            overflow_flag);
        count_launch();
    }
    PT_CUDA(cudaGetLastError());
    return PT_OK;
}

int launch_scatter_rows(const void *src, const int32_t *sel, uint32_t rows, uint32_t row_bytes, void *dst,
                        cudaStream_t s)
{
    if (row_bytes == 0 || row_bytes % 4 != 0) return PT_ERR_INVALID_ARG;
    const size_t total = (size_t)rows * (row_bytes / 4);
    if (total == 0) return PT_OK;
    scatter_rows_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(
        (const uint32_t *)src, sel, rows, row_bytes / 4, (uint32_t *)dst);
    count_launch();
    PT_CUDA(cudaGetLastError());
    return PT_OK;
}

int launch_ghost_check(const double *q, const double *d2, uint32_t m, int k, double r2,
                       const double *boxes, int n_ranks, int self, double halo, uint32_t *flag,
                       cudaStream_t s)
{
    if (m == 0) return PT_OK;
    if (k < 1 || k > PT_MAX_K || self < 0 || self >= n_ranks) return PT_ERR_INVALID_ARG;
    ghost_check_kernel<<<(m + 255) / 256, 256, 0, s>>>(q, d2, m, k, r2, boxes, n_ranks, self, halo, flag);
    count_launch();
    PT_CUDA(cudaGetLastError());
    return PT_OK;
}

int launch_halo_route(const double *q, const pt_cand *own, uint32_t m, int k, double r2,
                      const double *boxes, int n_ranks, int self, uint32_t cap, double *send,
                      int32_t *sel, uint32_t *counts, uint32_t *overflow_flag, cudaStream_t s)
{
    if (n_ranks < 1 || n_ranks > 1024 || k < 1 || k > PT_MAX_K) return PT_ERR_INVALID_ARG;
    PT_CUDA(cudaMemsetAsync(counts, 0, sizeof(uint32_t) * n_ranks, s));
    if (m) {
        halo_route_kernel<<<(m + 255) / 256, 256, 0, s>>>(q, own, m, k, r2, boxes, n_ranks, self, cap,
                                                         send, sel, counts);
        count_launch();
    }
    halo_header_kernel<<<1, 1024, 0, s>>>(counts, n_ranks, cap, send, overflow_flag);
    count_launch();
    PT_CUDA(cudaGetLastError());
    return PT_OK;
}

int launch_halo_prepare(const double *recv, int n_ranks, uint32_t cap, double *q_out, double *r2_out,
                        cudaStream_t s)
{
    const uint32_t total = (uint32_t)n_ranks * cap;
    if (total == 0) return PT_OK;
    halo_prepare_kernel<<<(total + 255) / 256, 256, 0, s>>>(recv, n_ranks, cap, q_out, r2_out);
    count_launch();
    PT_CUDA(cudaGetLastError());
    return PT_OK;
}

int launch_halo_merge(pt_cand *own, const pt_cand *back, const int32_t *sel, const uint32_t *count_ptr,
                      uint32_t cap, int k, int32_t *idx_out, double *d2_out, uint8_t *rgba_out,
                      float *normal_out, cudaStream_t s)
{
    if (cap == 0) return PT_OK;
    if (k < 1 || k > PT_MAX_K) return PT_ERR_UNSUPPORTED;
    halo_merge_kernel<<<(cap + WARPS_PER_BLOCK - 1) / WARPS_PER_BLOCK, WARPS_PER_BLOCK * 32, 0, s>>>(
        own, back, sel, count_ptr, cap, k, idx_out, d2_out, rgba_out, normal_out);
    count_launch();
    PT_CUDA(cudaGetLastError());
    return PT_OK;
}

}  // namespace pt

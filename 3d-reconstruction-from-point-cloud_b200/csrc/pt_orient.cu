// pt_orient.cu -- consistent orientation of the index's normals by propagation along the minimum
// spanning forest of the k-NN graph (DESIGN.md section 8, "Normal orientation"; Hoppe et al. 1992,
// CGAL's mst_orient_normals, Open3D's orient_normals_consistent_tangent_plane).
//
// Vertices are sorted records (rows), so neighbouring points sit close in every array.
//  1. self_query_chunks keeps every row's k-NN list.
//  2. orient_unit_kernel: the unit normal of every row that takes part (x = NaN otherwise).
//     orient_mask_kernel: a bit per list entry that is kept as an undirected edge (each pair once);
//     an exclusive scan of the bit counts places them and orient_edges_kernel writes them.
//  3. Boruvka.  lab[v] = rep | bit << 31: the row that represents v's component and v's sign relative
//     to it.  Each round: every component's lightest outgoing edge under (w, lo, hi) by two integer
//     atomicMin passes (w >= +0, so its bits order like its values), a hook along it (on an edge both
//     ends picked, the lower label stays the root), pointer jumping that composes the bits, and the
//     edges now inside a component dropped (cub::DeviceSelect in place).  Every hook adds one edge of
//     the unique minimum spanning forest, so a row's bit is the XOR of the edge signs on its forest path.
//  4. Each component's top point (largest z, lowest id) by two integer atomic passes; its rule gives
//     sigma_root, and sigma_v = sigma_root * (-1)^(bit_v xor bit_root).
// No floating-point atomics: the result does not depend on the schedule.
#include <algorithm>
#include <cmath>
#include <vector>

#include <cub/device/device_scan.cuh>
#include <cub/device/device_select.cuh>

#include "pt_bake.cuh"
#include "pt_fp64.cuh"

namespace pt {

constexpr uint32_t LAB_BIT = 0x80000000u;   // sign relative to the representative / edge sign d < 0
constexpr uint32_t LAB_REP = 0x7fffffffu;

struct OrientEdge {
    unsigned long long w;     // bits of w = 1 - |d| >= +0
    unsigned long long key;   // lo << 32 | hi (point ids)
    uint32_t u, v;            // rows; v's LAB_BIT: d < 0
};

static inline unsigned ocdiv(size_t a, size_t b) { return (unsigned)std::min<size_t>((a + b - 1) / b, 148 * 32); }

#define PT_GRID_STRIDE(i, n) \
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < (n); i += (size_t)gridDim.x * blockDim.x)

__device__ __forceinline__ bool takes_part(const D3 *nh, uint32_t r) { return !isnan(nh[r].x); }

template <typename PT>
__global__ void __launch_bounds__(256) orient_unit_kernel(const PT *pts, const pt_attr *attrs, uint32_t n, D3 *nh,
                                                          uint32_t *lab)
{
    PT_GRID_STRIDE(r, n) {
        const pt_attr m = attrs[pts[r].idx];
        const D3 md = {(double)m.nx, (double)m.ny, (double)m.nz};
        nh[r] = d3_usable(md) ? d3_normalise(md) : D3{NAN, 0.0, 0.0};
        lab[r] = (uint32_t)r;
    }
}

// bit s of mask[r]: entry s of row r's list is kept as the edge {i, j}.  A list ends at its first -1.
// Both ends must take part, and a pair in both lists is kept by its lower id only.
template <typename PT>
__global__ void __launch_bounds__(256)
orient_mask_kernel(const PT *pts, const uint32_t *inv, const D3 *nh, const int32_t *lists, uint32_t n, int k,
                   uint32_t *mask, uint32_t *count)
{
    PT_GRID_STRIDE(r, n) {
        uint32_t bits = 0;
        if (takes_part(nh, (uint32_t)r)) {
            const int32_t i = pts[r].idx;
            const int32_t *li = lists + r * k;
            for (int s = 0; s < k; ++s) {
                const int32_t j = li[s];
                if (j < 0 || (uint32_t)j >= n) break;
                if (j == i) continue;
                const uint32_t rj = inv[j];
                if (!takes_part(nh, rj)) continue;
                bool keep = i < j;
                if (!keep) {
                    const int32_t *lj = lists + (size_t)rj * k;
                    keep = true;
                    for (int t = 0; t < k; ++t) {
                        const int32_t x = lj[t];
                        if (x < 0 || (uint32_t)x >= n) break;
                        if (x == i) { keep = false; break; }
                    }
                }
                if (keep) bits |= 1u << s;
            }
        }
        mask[r] = bits;
        count[r] = __popc(bits);
    }
}

template <typename PT>
__global__ void __launch_bounds__(256)
orient_edges_kernel(const PT *pts, const uint32_t *inv, const D3 *nh, const int32_t *lists, uint32_t n, int k,
                    const uint32_t *mask, const uint32_t *first, OrientEdge *edges)
{
    PT_GRID_STRIDE(r, n) {
        uint32_t bits = mask[r], e = first[r];
        if (!bits) continue;
        const int32_t i = pts[r].idx;
        const D3 a = nh[r];
        while (bits) {
            const int s = __ffs(bits) - 1;
            bits &= bits - 1;
            const int32_t j = lists[r * k + s];
            const uint32_t rj = inv[j];
            const double d = d3_dot(a, nh[rj]);
            double w = __dsub_rn(1.0, fabs(d));
            if (w < 0.0) w = 0.0;
            const unsigned long long lo = (unsigned long long)min(i, j), hi = (unsigned long long)max(i, j);
            edges[e++] = OrientEdge{(unsigned long long)__double_as_longlong(w), lo << 32 | hi, (uint32_t)r,
                                    rj | (d < 0.0 ? LAB_BIT : 0u)};
        }
    }
}

__device__ __forceinline__ uint32_t rep_of(const uint32_t *lab, uint32_t r) { return lab[r] & LAB_REP; }

__global__ void __launch_bounds__(256) orient_min_w_kernel(const OrientEdge *edges, size_t m, const uint32_t *lab,
                                                           unsigned long long *best_w)
{
    PT_GRID_STRIDE(e, m) {
        const OrientEdge x = edges[e];
        atomicMin(best_w + rep_of(lab, x.u), x.w);
        atomicMin(best_w + rep_of(lab, x.v & LAB_REP), x.w);
    }
}

__global__ void __launch_bounds__(256) orient_min_key_kernel(const OrientEdge *edges, size_t m, const uint32_t *lab,
                                                             const unsigned long long *best_w, unsigned long long *best_key)
{
    PT_GRID_STRIDE(e, m) {
        const OrientEdge x = edges[e];
        const uint32_t cu = rep_of(lab, x.u), cv = rep_of(lab, x.v & LAB_REP);
        if (best_w[cu] == x.w) atomicMin(best_key + cu, x.key);
        if (best_w[cv] == x.w) atomicMin(best_key + cv, x.key);
    }
}

// hook[c] = the component c hooks to, with c's representative's sign relative to it in LAB_BIT
__global__ void __launch_bounds__(256) orient_hook_kernel(const OrientEdge *edges, size_t m, const uint32_t *lab,
                                                          const unsigned long long *best_w,
                                                          const unsigned long long *best_key, uint32_t *hook)
{
    PT_GRID_STRIDE(e, m) {
        const OrientEdge x = edges[e];
        const uint32_t v = x.v & LAB_REP, lu = lab[x.u], lv = lab[v];
        const uint32_t cu = lu & LAB_REP, cv = lv & LAB_REP;
        const bool by_u = best_w[cu] == x.w && best_key[cu] == x.key;
        const bool by_v = best_w[cv] == x.w && best_key[cv] == x.key;
        const uint32_t bit = (lu ^ lv ^ x.v) & LAB_BIT;
        if (by_u && !(by_v && cu < cv)) hook[cu] = cv | bit;
        if (by_v && !(by_u && cv < cu)) hook[cv] = cu | bit;
    }
}

__global__ void __launch_bounds__(256) orient_apply_hooks_kernel(const uint32_t *hook, uint32_t n, uint32_t *lab)
{
    PT_GRID_STRIDE(r, n) {
        const uint32_t h = hook[r];
        if (h != 0xffffffffu) lab[r] = h;
    }
}

// One pointer jump per row, in place: every word read is a valid (ancestor, sign relative to it)
// pair whenever it is read, so racing rows only converge sooner.
__global__ void __launch_bounds__(256) orient_jump_kernel(uint32_t n, uint32_t *lab, uint32_t *changed)
{
    PT_GRID_STRIDE(r, n) {
        const uint32_t a = lab[r], p = a & LAB_REP;
        const uint32_t b = lab[p], q = b & LAB_REP;
        if (q != p) {
            lab[r] = q | ((a ^ b) & LAB_BIT);
            *changed = 1u;
        }
    }
}

struct OrientCrossing {   // cub select: the edge still joins two components
    const uint32_t *lab;
    __device__ __forceinline__ bool operator()(const OrientEdge &x) const
    {
        return (lab[x.u] & LAB_REP) != (lab[x.v & LAB_REP] & LAB_REP);
    }
};

// fp64 -> uint64 with the same order; -0 is taken as +0 (the root rule compares values)
__device__ __forceinline__ unsigned long long z_key(double z)
{
    const unsigned long long u = (unsigned long long)__double_as_longlong(z == 0.0 ? 0.0 : z);
    return (u >> 63) ? ~u : (u | 0x8000000000000000ull);
}

template <typename PT>
__global__ void __launch_bounds__(256) orient_top_z_kernel(const PT *pts, const D3 *nh, uint32_t n, const uint32_t *lab,
                                                           unsigned long long *top_z)
{
    PT_GRID_STRIDE(r, n) {
        if (takes_part(nh, (uint32_t)r)) atomicMax(top_z + rep_of(lab, (uint32_t)r), z_key((double)pts[r].z));
    }
}

template <typename PT>
__global__ void __launch_bounds__(256) orient_top_id_kernel(const PT *pts, const D3 *nh, uint32_t n, const uint32_t *lab,
                                                            const unsigned long long *top_z, uint32_t *top_id)
{
    PT_GRID_STRIDE(r, n) {
        if (!takes_part(nh, (uint32_t)r)) continue;
        const PT p = pts[r];
        const uint32_t c = rep_of(lab, (uint32_t)r);
        if (top_z[c] == z_key((double)p.z)) atomicMin(top_id + c, (uint32_t)p.idx);
    }
}

struct OrientOut {
    pt_attr *attrs;           // the index's attributes (original order)
    pt_attr *store_curve;     // store: attrs_curve (sorted order) where the index has it, else null
    int store, has_view;
    double vx, vy, vz;
    float *normal;            // n x 3, original order
    int32_t *root;            // n, original order
    unsigned long long *counts;   // += oriented, flipped, components
};

template <typename PT>
__global__ void __launch_bounds__(256) orient_signs_kernel(const PT *pts, const uint32_t *inv, const D3 *nh, uint32_t n,
                                                           const uint32_t *lab, const uint32_t *top_id, const OrientOut o)
{
    PT_GRID_STRIDE(r, n) {
        const uint32_t orig = (uint32_t)pts[r].idx;
        pt_attr m = o.attrs[orig];
        const bool part = takes_part(nh, (uint32_t)r);
        int32_t root = -1;
        bool flip = false;
        if (part) {
            const uint32_t c = rep_of(lab, (uint32_t)r);
            root = (int32_t)top_id[c];
            const uint32_t rr = inv[root];
            const D3 nr = nh[rr];
            bool neg;
            if (o.has_view) {
                const PT p = pts[rr];
                neg = d3_dot(nr, d3_sub(D3{o.vx, o.vy, o.vz}, D3{(double)p.x, (double)p.y, (double)p.z})) < 0.0;
            } else if (nr.z != 0.0) {
                neg = nr.z < 0.0;
            } else {
                const double ax = fabs(nr.x), ay = fabs(nr.y), az = fabs(nr.z);
                neg = (ax >= ay && ax >= az) ? nr.x < 0.0 : (ay >= az ? nr.y < 0.0 : nr.z < 0.0);
            }
            flip = neg != (((lab[r] ^ lab[rr]) & LAB_BIT) != 0);
            if (flip) { m.nx = -m.nx; m.ny = -m.ny; m.nz = -m.nz; }
            if (o.store) {
                o.attrs[orig].nx = m.nx; o.attrs[orig].ny = m.ny; o.attrs[orig].nz = m.nz;
                if (o.store_curve) { o.store_curve[r].nx = m.nx; o.store_curve[r].ny = m.ny; o.store_curve[r].nz = m.nz; }
            }
        }
        if (o.normal) {
            o.normal[3 * (size_t)orig] = m.nx;
            o.normal[3 * (size_t)orig + 1] = m.ny;
            o.normal[3 * (size_t)orig + 2] = m.nz;
        }
        if (o.root) o.root[orig] = root;
        const unsigned act = __activemask();
        const int lead = __ffs(act) - 1;
        const unsigned a = __ballot_sync(act, part), f = __ballot_sync(act, flip),
                       c = __ballot_sync(act, part && rep_of(lab, (uint32_t)r) == (uint32_t)r);
        if ((int)(threadIdx.x & 31u) == lead) {
            if (a) atomicAdd(o.counts, (unsigned long long)__popc(a));
            if (f) atomicAdd(o.counts + 1, (unsigned long long)__popc(f));
            if (c) atomicAdd(o.counts + 2, (unsigned long long)__popc(c));
        }
    }
}

template <typename PT>
static int orient_run(pt_index *ix, int k, double radius, OrientOut o, uint64_t *n_edges, std::vector<cudaEvent_t> &marks,
                      cudaStream_t s)
{
    const uint32_t n = ix->n;
    const PT *pts = (const PT *)ix->pts;
    int32_t *d_lists = nullptr;
    D3 *d_nh = nullptr;
    uint32_t *d_lab = nullptr, *d_mask = nullptr, *d_first = nullptr, *d_hook = nullptr, *d_changed = nullptr;
    unsigned long long *d_best_w = nullptr, *d_best_key = nullptr;
    OrientEdge *d_edges = nullptr;
    int64_t *d_num = nullptr;
    void *d_tmp = nullptr;
    uint32_t n_e = 0;
    int rc = PT_OK;
    auto fail = [&](cudaError_t e) { if (e != cudaSuccess && rc == PT_OK) rc = map_cuda_error(e); return e != cudaSuccess; };
    auto oom = [&](bool bad) { if (bad && rc == PT_OK) rc = PT_ERR_OUT_OF_MEMORY; return bad; };
    auto launched = [&]() { count_launch(); return fail(cudaGetLastError()); };
    const unsigned gn = ocdiv(n, 256);
    do {
        if (oom(pool_alloc((void **)&d_lists, sizeof(int32_t) * (size_t)k * n, s))) break;
        if ((rc = self_query_chunks(ix, k, radius, d_lists, true, [](uint32_t, uint32_t, const int32_t *) { return PT_OK; },
                                    &marks, s)) != PT_OK)
            break;
        const uint32_t *inv = ix->inv_perm;
        // ---- edges
        if (oom(pool_alloc((void **)&d_nh, sizeof(D3) * n, s) || pool_alloc((void **)&d_lab, sizeof(uint32_t) * n, s) ||
                pool_alloc((void **)&d_mask, sizeof(uint32_t) * n, s) ||
                pool_alloc((void **)&d_first, sizeof(uint32_t) * ((size_t)n + 1), s) ||
                pool_alloc((void **)&d_num, sizeof(int64_t) + sizeof(uint32_t), s)))
            break;
        d_changed = (uint32_t *)(d_num + 1);
        orient_unit_kernel<PT><<<gn, 256, 0, s>>>(pts, ix->attrs, n, d_nh, d_lab);
        if (launched()) break;
        orient_mask_kernel<PT><<<gn, 256, 0, s>>>(pts, inv, d_nh, d_lists, n, k, d_mask, d_first);
        if (launched() || fail(cudaMemsetAsync(d_first + n, 0, sizeof(uint32_t), s))) break;
        size_t scan_bytes = 0, select_bytes = 0;
        if (fail(cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, d_first, d_first, (int)n + 1, s))) break;
        if (fail(cub::DeviceSelect::If(nullptr, select_bytes, d_edges, d_num, (int64_t)n * k, OrientCrossing{d_lab}, s)))
            break;
        if (oom(pool_alloc(&d_tmp, std::max(scan_bytes, select_bytes), s))) break;
        if (fail(cub::DeviceScan::ExclusiveSum(d_tmp, scan_bytes, d_first, d_first, (int)n + 1, s))) break;
        if (fail(cudaMemcpyAsync(&n_e, d_first + n, sizeof n_e, cudaMemcpyDeviceToHost, s)) || fail(cudaStreamSynchronize(s)))
            break;
        *n_edges = n_e;
        if (oom(pool_alloc((void **)&d_edges, sizeof(OrientEdge) * std::max<uint32_t>(n_e, 1), s))) break;
        orient_edges_kernel<PT><<<gn, 256, 0, s>>>(pts, inv, d_nh, d_lists, n, k, d_mask, d_first, d_edges);
        if (launched()) break;
        pool_free(d_lists, s);
        pool_free(d_mask, s);
        pool_free(d_first, s);
        d_lists = nullptr; d_mask = d_first = nullptr;
        // ---- Boruvka
        if (oom(pool_alloc((void **)&d_best_w, sizeof(unsigned long long) * n, s) ||
                pool_alloc((void **)&d_best_key, sizeof(unsigned long long) * n, s) ||
                pool_alloc((void **)&d_hook, sizeof(uint32_t) * n, s)))
            break;
        size_t m = n_e;
        while (m > 0 && rc == PT_OK) {
            const unsigned ge = ocdiv(m, 256);
            if (fail(cudaMemsetAsync(d_best_w, 0xff, sizeof(unsigned long long) * n, s)) ||
                fail(cudaMemsetAsync(d_best_key, 0xff, sizeof(unsigned long long) * n, s)) ||
                fail(cudaMemsetAsync(d_hook, 0xff, sizeof(uint32_t) * n, s)))
                break;
            orient_min_w_kernel<<<ge, 256, 0, s>>>(d_edges, m, d_lab, d_best_w);
            if (launched()) break;
            orient_min_key_kernel<<<ge, 256, 0, s>>>(d_edges, m, d_lab, d_best_w, d_best_key);
            if (launched()) break;
            orient_hook_kernel<<<ge, 256, 0, s>>>(d_edges, m, d_lab, d_best_w, d_best_key, d_hook);
            if (launched()) break;
            orient_apply_hooks_kernel<<<gn, 256, 0, s>>>(d_hook, n, d_lab);
            if (launched()) break;
            for (uint32_t changed = 1; changed && rc == PT_OK;) {
                if (fail(cudaMemsetAsync(d_changed, 0, sizeof(uint32_t), s))) break;
                orient_jump_kernel<<<gn, 256, 0, s>>>(n, d_lab, d_changed);
                if (launched() || fail(cudaMemcpyAsync(&changed, d_changed, sizeof changed, cudaMemcpyDeviceToHost, s)) ||
                    fail(cudaStreamSynchronize(s)))
                    break;
            }
            if (rc != PT_OK) break;
            int64_t left = 0;
            if (fail(cub::DeviceSelect::If(d_tmp, select_bytes, d_edges, d_num, (int64_t)m, OrientCrossing{d_lab}, s)) ||
                fail(cudaMemcpyAsync(&left, d_num, sizeof left, cudaMemcpyDeviceToHost, s)) || fail(cudaStreamSynchronize(s)))
                break;
            m = (size_t)left;
        }
        if (rc != PT_OK) break;
        // ---- roots and signs (best_w holds the top z keys, hook the top ids)
        if (fail(cudaMemsetAsync(d_best_w, 0, sizeof(unsigned long long) * n, s)) ||
            fail(cudaMemsetAsync(d_hook, 0xff, sizeof(uint32_t) * n, s)))
            break;
        orient_top_z_kernel<PT><<<gn, 256, 0, s>>>(pts, d_nh, n, d_lab, d_best_w);
        if (launched()) break;
        orient_top_id_kernel<PT><<<gn, 256, 0, s>>>(pts, d_nh, n, d_lab, d_best_w, d_hook);
        if (launched()) break;
        orient_signs_kernel<PT><<<gn, 256, 0, s>>>(pts, inv, d_nh, n, d_lab, d_hook, o);
        if (launched() || fail(record_mark(&marks, s))) break;
    } while (0);
    pool_free(d_lists, s);
    pool_free(d_nh, s);
    pool_free(d_lab, s);
    pool_free(d_mask, s);
    pool_free(d_first, s);
    pool_free(d_num, s);
    pool_free(d_tmp, s);
    pool_free(d_edges, s);
    pool_free(d_best_w, s);
    pool_free(d_best_key, s);
    pool_free(d_hook, s);
    return rc;
}

}  // namespace pt

using namespace pt;

extern "C" int pt_index_orient_normals(pt_index *ix, int k, double radius, const double *viewpoint, int store,
                                       float *normal_out, int32_t *root_out, pt_orient_stats *stats)
{
    if (!ix || (!normal_out && !root_out && !store)) return PT_ERR_INVALID_ARG;
    if (viewpoint && !(std::isfinite(viewpoint[0]) && std::isfinite(viewpoint[1]) && std::isfinite(viewpoint[2])))
        return PT_ERR_INVALID_ARG;
    if (k < 2) return PT_ERR_INVALID_ARG;             // a list of one holds only the point itself
    if (k > PT_MAX_K) return PT_ERR_UNSUPPORTED;
    if (!ix->attrs && ix->n) return PT_ERR_INVALID_ARG;
    // edge offsets are uint32 and rows carry a sign bit: n k must fit an int
    if ((uint64_t)ix->n * (uint64_t)k > (uint64_t)INT32_MAX) return PT_ERR_UNSUPPORTED;
    if (pt_device_count() == 0) return PT_ERR_NO_DEVICE;
    if (stats) *stats = pt_orient_stats{0, 0, 0, 0, 0.0f, 0.0f};
    if (ix->n == 0) return PT_OK;
    PT_CUDA(cudaSetDevice(ix->device));
    cudaStream_t s = ix->stream;
    const size_t n = ix->n;
    float *d_normal = nullptr;
    int32_t *d_root = nullptr;
    unsigned long long *d_counts = nullptr, counts[3] = {0, 0, 0};
    uint64_t n_edges = 0;
    std::vector<cudaEvent_t> marks;
    int rc = PT_OK;
    auto fail = [&](cudaError_t e) { if (e != cudaSuccess && rc == PT_OK) rc = map_cuda_error(e); return e != cudaSuccess; };
    do {
        if ((normal_out && pool_alloc((void **)&d_normal, sizeof(float) * 3 * n, s)) ||
            (root_out && pool_alloc((void **)&d_root, sizeof(int32_t) * n, s)) ||
            pool_alloc((void **)&d_counts, sizeof counts, s)) {
            rc = PT_ERR_OUT_OF_MEMORY;
            break;
        }
        if (fail(cudaMemsetAsync(d_counts, 0, sizeof counts, s))) break;
        OrientOut o{};
        o.attrs = ix->attrs;
        o.store = store != 0;
        o.store_curve = store ? ix->attrs_curve : nullptr;
        o.has_view = viewpoint ? 1 : 0;
        if (viewpoint) { o.vx = viewpoint[0]; o.vy = viewpoint[1]; o.vz = viewpoint[2]; }
        o.normal = d_normal;
        o.root = d_root;
        o.counts = d_counts;
        rc = ix->coord_f64 ? orient_run<PointD>(ix, k, radius, o, &n_edges, marks, s)
                           : orient_run<PointF>(ix, k, radius, o, &n_edges, marks, s);
        if (rc != PT_OK) break;
        if (normal_out && fail(cudaMemcpyAsync(normal_out, d_normal, sizeof(float) * 3 * n, cudaMemcpyDeviceToHost, s))) break;
        if (root_out && fail(cudaMemcpyAsync(root_out, d_root, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, s))) break;
        if (fail(cudaMemcpyAsync(counts, d_counts, sizeof counts, cudaMemcpyDeviceToHost, s))) break;
        if (fail(cudaStreamSynchronize(s))) break;
        if (stats) {
            stats->oriented = counts[0];
            stats->flipped = counts[1];
            stats->components = counts[2];
            stats->edges = n_edges;
            // marks: start, one per chunk's query, then the end of the signs
            const size_t q = marks.size() - 2;
            if (cudaEventElapsedTime(&stats->knn_ms, marks[0], marks[q]) != cudaSuccess) stats->knn_ms = 0.0f;
            if (cudaEventElapsedTime(&stats->mst_ms, marks[q], marks.back()) != cudaSuccess) stats->mst_ms = 0.0f;
        }
    } while (0);
    cudaStreamSynchronize(s);
    pool_free(d_normal, s);
    pool_free(d_root, s);
    pool_free(d_counts, s);
    for (auto &e : marks) if (e) cudaEventDestroy(e);
    cudaStreamSynchronize(s);
    cudaGetLastError();
    return rc;
}

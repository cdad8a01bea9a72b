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

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <cub/device/device_select.cuh>

#include "pt_bake.cuh"
#include "pt_fp64.cuh"

namespace pt {

constexpr uint32_t LAB_BIT = 0x80000000u;   // sign relative to the representative / edge sign d < 0
constexpr uint32_t LAB_REP = 0x7fffffffu;

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

// The edge {i, j} between unit normals a and b, joining vertices u and v
__device__ __forceinline__ OrientEdge orient_edge(D3 a, D3 b, int32_t i, int32_t j, uint32_t u, uint32_t v)
{
    const double d = d3_dot(a, b);
    double w = __dsub_rn(1.0, fabs(d));
    if (w < 0.0) w = 0.0;
    const unsigned long long lo = (unsigned long long)min(i, j), hi = (unsigned long long)max(i, j);
    return OrientEdge{(unsigned long long)__double_as_longlong(w), lo << 32 | hi, u, v | (d < 0.0 ? LAB_BIT : 0u)};
}

// whether point i is missing from the list lj (it ends at its first entry outside 0 .. n - 1)
__device__ __forceinline__ bool not_in_list(const int32_t *lj, int k, uint32_t n, int32_t i)
{
    for (int t = 0; t < k; ++t) {
        const int32_t x = lj[t];
        if (x < 0 || (uint32_t)x >= n) break;
        if (x == i) return false;
    }
    return true;
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
            edges[e++] = orient_edge(a, nh[rj], i, j, (uint32_t)r, rj);
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

// Boruvka's per-vertex arrays and scratch: lab (initialised lab[v] = v), hook, best_w, best_key (n
// each); changed, num (two counters); tmp, enough for a cub select over the edges.
struct OrientWork {
    uint32_t *lab, *hook, *changed;
    unsigned long long *best_w, *best_key;
    int64_t *num;
    void *tmp;
    size_t tmp_bytes;
};

// Every edge a hook of orient_hook_kernel takes, by its predicate: flag[e] = 1
__global__ void __launch_bounds__(256) orient_mark_kernel(const OrientEdge *edges, size_t m, const uint32_t *lab,
                                                          const unsigned long long *best_w,
                                                          const unsigned long long *best_key, uint8_t *flag)
{
    PT_GRID_STRIDE(e, m) {
        const OrientEdge x = edges[e];
        const uint32_t cu = rep_of(lab, x.u), cv = rep_of(lab, x.v & LAB_REP);
        const bool by_u = best_w[cu] == x.w && best_key[cu] == x.key;
        const bool by_v = best_w[cv] == x.w && best_key[cv] == x.key;
        flag[e] = (by_u && !(by_v && cu < cv)) || (by_v && !(by_u && cv < cu)) ? 1 : 0;
    }
}

// Boruvka on edges[0 .. m) over the vertices 0 .. n - 1, on s (the edges are consumed).  With
// forest: each round appends the edges its hooks take (flag: m bytes of scratch), so forest[0 ..
// *n_forest) ends up as the minimum spanning forest.
static int orient_boruvka(OrientEdge *edges, size_t m, uint32_t n, const OrientWork &w, cudaStream_t s,
                          uint8_t *flag = nullptr, OrientEdge *forest = nullptr, size_t *n_forest = nullptr)
{
    int rc = PT_OK;
    auto fail = [&](cudaError_t e) { if (e != cudaSuccess && rc == PT_OK) rc = map_cuda_error(e); return e != cudaSuccess; };
    auto launched = [&]() { count_launch(); return fail(cudaGetLastError()); };
    const unsigned gn = ocdiv(n, 256);
    while (m > 0 && rc == PT_OK) {
        const unsigned ge = ocdiv(m, 256);
        if (fail(cudaMemsetAsync(w.best_w, 0xff, sizeof(unsigned long long) * n, s)) ||
            fail(cudaMemsetAsync(w.best_key, 0xff, sizeof(unsigned long long) * n, s)) ||
            fail(cudaMemsetAsync(w.hook, 0xff, sizeof(uint32_t) * n, s)))
            break;
        orient_min_w_kernel<<<ge, 256, 0, s>>>(edges, m, w.lab, w.best_w);
        if (launched()) break;
        orient_min_key_kernel<<<ge, 256, 0, s>>>(edges, m, w.lab, w.best_w, w.best_key);
        if (launched()) break;
        orient_hook_kernel<<<ge, 256, 0, s>>>(edges, m, w.lab, w.best_w, w.best_key, w.hook);
        if (launched()) break;
        if (forest) {
            orient_mark_kernel<<<ge, 256, 0, s>>>(edges, m, w.lab, w.best_w, w.best_key, flag);
            if (launched()) break;
            size_t bytes = w.tmp_bytes;
            if (fail(cub::DeviceSelect::Flagged(w.tmp, bytes, edges, flag, forest + *n_forest, w.num + 1, (int64_t)m, s)))
                break;
        }
        orient_apply_hooks_kernel<<<gn, 256, 0, s>>>(w.hook, n, w.lab);
        if (launched()) break;
        for (uint32_t changed = 1; changed && rc == PT_OK;) {
            if (fail(cudaMemsetAsync(w.changed, 0, sizeof(uint32_t), s))) break;
            orient_jump_kernel<<<gn, 256, 0, s>>>(n, w.lab, w.changed);
            if (launched() || fail(cudaMemcpyAsync(&changed, w.changed, sizeof changed, cudaMemcpyDeviceToHost, s)) ||
                fail(cudaStreamSynchronize(s)))
                break;
        }
        if (rc != PT_OK) break;
        int64_t left[2] = {0, 0};
        size_t bytes = w.tmp_bytes;
        if (fail(cub::DeviceSelect::If(w.tmp, bytes, edges, w.num, (int64_t)m, OrientCrossing{w.lab}, s)) ||
            fail(cudaMemcpyAsync(left, w.num, sizeof(int64_t) * (forest ? 2 : 1), cudaMemcpyDeviceToHost, s)) ||
            fail(cudaStreamSynchronize(s)))
            break;
        m = (size_t)left[0];
        if (forest) *n_forest += (size_t)left[1];
    }
    return rc;
}

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

// The root rule: whether the root's unit normal nr is negated.  pos() gives the root's position; it
// is read only with a viewpoint.
template <typename Pos>
__device__ __forceinline__ bool root_negates(const OrientOut &o, const D3 nr, const Pos &pos)
{
    bool neg;
    if (o.has_view) {
        neg = d3_dot(nr, d3_sub(D3{o.vx, o.vy, o.vz}, pos())) < 0.0;
    } else if (nr.z != 0.0) {
        neg = nr.z < 0.0;
    } else {
        const double ax = fabs(nr.x), ay = fabs(nr.y), az = fabs(nr.z);
        neg = (ax >= ay && ax >= az) ? nr.x < 0.0 : (ay >= az ? nr.y < 0.0 : nr.z < 0.0);
    }
    return neg;
}

// counts += the warp's points that take part, that flip, and that represent their component (rep())
template <typename Rep>
__device__ __forceinline__ void orient_tally(const OrientOut &o, bool part, bool flip, const Rep &rep)
{
    const unsigned act = __activemask();
    const int lead = __ffs(act) - 1;
    const unsigned a = __ballot_sync(act, part), f = __ballot_sync(act, flip), c = __ballot_sync(act, rep());
    if ((int)(threadIdx.x & 31u) == lead) {
        if (a) atomicAdd(o.counts, (unsigned long long)__popc(a));
        if (f) atomicAdd(o.counts + 1, (unsigned long long)__popc(f));
        if (c) atomicAdd(o.counts + 2, (unsigned long long)__popc(c));
    }
}

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
            const bool neg = root_negates(o, nr, [&] {
                const PT p = pts[rr];
                return D3{(double)p.x, (double)p.y, (double)p.z};
            });
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
        orient_tally(o, part, flip, [&] { return part && rep_of(lab, (uint32_t)r) == (uint32_t)r; });
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
        if ((rc = orient_boruvka(d_edges, n_e, n, OrientWork{d_lab, d_hook, d_changed, d_best_w, d_best_key, d_num, d_tmp,
                                                             select_bytes},
                                 s)) != PT_OK)
            break;
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

// ---- sharded clouds (DESIGN.md section 8, "Sharded normal orientation") ----------------------------
constexpr uint32_t NOT_OWN = 0xffffffffu;

// own[local id of the record at rows[j]] = j: the position of an own point among the own rows
template <typename PT>
__global__ void __launch_bounds__(256) orient_own_kernel(const PT *pts, const uint32_t *rows, uint32_t n_rows, uint32_t *own)
{
    PT_GRID_STRIDE(j, n_rows) own[pts[rows[j]].idx] = (uint32_t)j;
}

// orient_mask_kernel over a slab's own rows (own row j: sorted record rows[j], list at lists + j k):
// intra[j] marks the edges to other own points under the same rule, cross[j] every edge to a point
// that takes part and is owned elsewhere (its owner may emit the same pair: orient_home drops one)
template <typename PT>
__global__ void __launch_bounds__(256)
orient_slab_mask_kernel(const PT *pts, const uint32_t *inv, const D3 *nh, const int32_t *lists, const uint32_t *rows,
                        const uint32_t *own, uint32_t n, uint32_t n_rows, int k, uint32_t *intra, uint32_t *n_intra,
                        uint32_t *cross, uint32_t *n_cross)
{
    PT_GRID_STRIDE(jr, n_rows) {
        uint32_t bi = 0, bc = 0;
        const uint32_t r = rows[jr];
        if (takes_part(nh, r)) {
            const int32_t i = pts[r].idx;
            const int32_t *li = lists + jr * k;
            for (int s = 0; s < k; ++s) {
                const int32_t j = li[s];
                if (j < 0 || (uint32_t)j >= n) break;
                if (j == i) continue;
                if (!takes_part(nh, inv[j])) continue;
                const uint32_t oj = own[j];
                if (oj == NOT_OWN) bc |= 1u << s;
                else if (i < j || not_in_list(lists + (size_t)oj * k, k, n, i)) bi |= 1u << s;
            }
        }
        intra[jr] = bi;
        n_intra[jr] = __popc(bi);
        cross[jr] = bc;
        n_cross[jr] = __popc(bc);
    }
}

// The marked edges of own row j: intra edges between own rows, keyed by local ids (which ascend with
// the global ids); cross edges between global ids (ids: local id -> global id)
template <typename PT>
__global__ void __launch_bounds__(256)
orient_slab_edges_kernel(const PT *pts, const uint32_t *inv, const D3 *nh, const int32_t *lists, const uint32_t *rows,
                         const uint32_t *own, const int32_t *ids, uint32_t n_rows, int k, const uint32_t *intra,
                         const uint32_t *first_intra, const uint32_t *cross, const uint32_t *first_cross,
                         OrientEdge *e_intra, OrientEdge *e_cross)
{
    PT_GRID_STRIDE(jr, n_rows) {
        uint32_t bi = intra[jr], bc = cross[jr], e = first_intra[jr], c = first_cross[jr];
        if (!(bi | bc)) continue;
        const uint32_t r = rows[jr];
        const int32_t i = pts[r].idx;
        const D3 a = nh[r];
        while (bi) {
            const int s = __ffs(bi) - 1;
            bi &= bi - 1;
            const int32_t j = lists[jr * k + s];
            e_intra[e++] = orient_edge(a, nh[inv[j]], i, j, (uint32_t)jr, own[j]);
        }
        while (bc) {
            const int s = __ffs(bc) - 1;
            bc &= bc - 1;
            const int32_t j = lists[jr * k + s], gi = ids[i], gj = ids[j];
            e_cross[c++] = orient_edge(a, nh[inv[j]], gi, gj, (uint32_t)gi, (uint32_t)gj);
        }
    }
}

// A forest edge of own rows and local ids, in global ids
template <typename PT>
__global__ void __launch_bounds__(256)
orient_globalise_kernel(const PT *pts, const uint32_t *rows, const int32_t *ids, size_t m, OrientEdge *edges)
{
    PT_GRID_STRIDE(e, m) {
        OrientEdge x = edges[e];
        const unsigned long long lo = (unsigned long long)ids[x.key >> 32], hi = (unsigned long long)ids[x.key & 0xffffffffu];
        x.key = lo << 32 | hi;
        x.u = (uint32_t)ids[pts[rows[x.u]].idx];
        x.v = (uint32_t)ids[pts[rows[x.v & LAB_REP]].idx] | (x.v & LAB_BIT);
        edges[e] = x;
    }
}

template <typename PT>
static int orient_slab_t(pt_index *ix, int k, double radius, const NormalsSlab &sl, std::vector<OrientEdge> &forest,
                         std::vector<OrientEdge> &cross, uint64_t *intra, int *needs)
{
    cudaStream_t s = ix->stream;
    const uint32_t n = ix->n;
    const PT *pts = (const PT *)ix->pts;
    SlabRows w;
    int32_t *d_lists = nullptr;
    D3 *d_nh = nullptr;
    uint32_t *d_lab = nullptr, *d_own = nullptr, *d_mask = nullptr, *d_first = nullptr, *d_hook = nullptr, *d_changed = nullptr;
    unsigned long long *d_best_w = nullptr, *d_best_key = nullptr;
    OrientEdge *d_intra = nullptr, *d_cross = nullptr, *d_forest = nullptr;
    uint8_t *d_flag = nullptr;
    int64_t *d_num = nullptr;
    void *d_tmp = nullptr;
    int rc = PT_OK;
    auto fail = [&](cudaError_t e) { if (e != cudaSuccess && rc == PT_OK) rc = map_cuda_error(e); return e != cudaSuccess; };
    auto oom = [&](bool bad) { if (bad && rc == PT_OK) rc = PT_ERR_OUT_OF_MEMORY; return bad; };
    auto launched = [&]() { count_launch(); return fail(cudaGetLastError()); };
    do {
        if ((rc = slab_rows_select(ix, sl, w)) != PT_OK) break;
        const uint32_t nr = w.n_rows;
        if (nr == 0) break;
        if (oom(pool_alloc((void **)&d_lists, sizeof(int32_t) * (size_t)k * nr, s))) break;
        if ((rc = slab_rows_query(ix, k, radius, sl, w, d_lists, true,
                                  [](uint32_t, uint32_t, const int32_t *) { return PT_OK; }, nullptr)) != PT_OK)
            break;
        uint32_t flag = 0;
        if (fail(cudaMemcpyAsync(&flag, w.flag, sizeof flag, cudaMemcpyDeviceToHost, s)) || fail(cudaStreamSynchronize(s)))
            break;
        if (sl.check && flag) {             // this attempt is void: the caller widens the halo
            *needs = 1;
            break;
        }
        // ---- edges of the own rows
        const uint32_t *inv = ix->inv_perm;
        if (oom(pool_alloc((void **)&d_nh, sizeof(D3) * n, s) || pool_alloc((void **)&d_lab, sizeof(uint32_t) * n, s) ||
                pool_alloc((void **)&d_own, sizeof(uint32_t) * n, s) ||
                pool_alloc((void **)&d_mask, sizeof(uint32_t) * 2 * (size_t)nr, s) ||
                pool_alloc((void **)&d_first, sizeof(uint32_t) * 2 * ((size_t)nr + 1), s) ||
                pool_alloc((void **)&d_num, sizeof(int64_t) * 2 + sizeof(uint32_t), s)))
            break;
        d_changed = (uint32_t *)(d_num + 2);
        uint32_t *first_c = d_first + nr + 1;
        const unsigned gn = ocdiv(n, 256), gr = ocdiv(nr, 256);
        orient_unit_kernel<PT><<<gn, 256, 0, s>>>(pts, ix->attrs, n, d_nh, d_lab);
        if (launched() || fail(cudaMemsetAsync(d_own, 0xff, sizeof(uint32_t) * n, s))) break;
        orient_own_kernel<PT><<<gr, 256, 0, s>>>(pts, w.rows, nr, d_own);
        if (launched()) break;
        orient_slab_mask_kernel<PT><<<gr, 256, 0, s>>>(pts, inv, d_nh, d_lists, w.rows, d_own, n, nr, k, d_mask, d_first,
                                                       d_mask + nr, first_c);
        if (launched() || fail(cudaMemsetAsync(d_first + nr, 0, sizeof(uint32_t), s)) ||
            fail(cudaMemsetAsync(first_c + nr, 0, sizeof(uint32_t), s)))
            break;
        size_t scan_bytes = 0, select_bytes = 0, flag_bytes = 0;
        if (fail(cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, d_first, d_first, (int)nr + 1, s)) ||
            fail(cub::DeviceSelect::If(nullptr, select_bytes, d_intra, d_num, (int64_t)nr * k, OrientCrossing{d_lab}, s)) ||
            fail(cub::DeviceSelect::Flagged(nullptr, flag_bytes, d_intra, d_flag, d_forest, d_num + 1, (int64_t)nr * k, s)))
            break;
        const size_t tmp_bytes = std::max(scan_bytes, std::max(select_bytes, flag_bytes));
        if (oom(pool_alloc(&d_tmp, tmp_bytes, s))) break;
        if (fail(cub::DeviceScan::ExclusiveSum(d_tmp, scan_bytes, d_first, d_first, (int)nr + 1, s)) ||
            fail(cub::DeviceScan::ExclusiveSum(d_tmp, scan_bytes, first_c, first_c, (int)nr + 1, s)))
            break;
        uint32_t n_i = 0, n_c = 0;
        if (fail(cudaMemcpyAsync(&n_i, d_first + nr, sizeof n_i, cudaMemcpyDeviceToHost, s)) ||
            fail(cudaMemcpyAsync(&n_c, first_c + nr, sizeof n_c, cudaMemcpyDeviceToHost, s)) || fail(cudaStreamSynchronize(s)))
            break;
        *intra = n_i;
        if (oom(pool_alloc((void **)&d_intra, sizeof(OrientEdge) * std::max<uint32_t>(n_i, 1), s) ||
                pool_alloc((void **)&d_cross, sizeof(OrientEdge) * std::max<uint32_t>(n_c, 1), s)))
            break;
        orient_slab_edges_kernel<PT><<<gr, 256, 0, s>>>(pts, inv, d_nh, d_lists, w.rows, d_own, ix->ids, nr, k, d_mask, d_first,
                                                        d_mask + nr, first_c, d_intra, d_cross);
        if (launched()) break;
        cross.resize(n_c);
        if (n_c && fail(cudaMemcpyAsync(cross.data(), d_cross, sizeof(OrientEdge) * n_c, cudaMemcpyDeviceToHost, s))) break;
        void *done[] = {d_lists, d_mask, d_first, d_own, d_cross};
        for (void *p : done) pool_free(p, s);
        d_lists = nullptr; d_mask = d_first = d_own = nullptr; d_cross = nullptr;
        // ---- the minimum spanning forest of the intra edges over the own rows
        if (oom(pool_alloc((void **)&d_best_w, sizeof(unsigned long long) * nr, s) ||
                pool_alloc((void **)&d_best_key, sizeof(unsigned long long) * nr, s) ||
                pool_alloc((void **)&d_hook, sizeof(uint32_t) * nr, s) ||
                pool_alloc((void **)&d_flag, std::max<size_t>(n_i, 1), s) ||
                pool_alloc((void **)&d_forest, sizeof(OrientEdge) * nr, s)))
            break;
        size_t n_f = 0;
        if ((rc = orient_boruvka(d_intra, n_i, nr, OrientWork{d_lab, d_hook, d_changed, d_best_w, d_best_key, d_num, d_tmp,
                                                             tmp_bytes},
                                 s, d_flag, d_forest, &n_f)) != PT_OK)
            break;
        if (n_f) {
            orient_globalise_kernel<PT><<<ocdiv(n_f, 256), 256, 0, s>>>(pts, w.rows, ix->ids, n_f, d_forest);
            if (launched()) break;
        }
        forest.resize(n_f);
        if (n_f && fail(cudaMemcpyAsync(forest.data(), d_forest, sizeof(OrientEdge) * n_f, cudaMemcpyDeviceToHost, s))) break;
        fail(cudaStreamSynchronize(s));
    } while (0);
    cudaStreamSynchronize(s);
    slab_rows_free(w, s);
    void *frees[] = {d_lists, d_nh, d_lab, d_own, d_mask, d_first, d_hook, d_best_w, d_best_key, d_intra, d_cross,
                     d_forest, d_flag, d_num, d_tmp};
    for (void *p : frees) pool_free(p, s);
    cudaStreamSynchronize(s);
    cudaGetLastError();
    return rc;
}

int orient_slab(pt_index *ix, int k, double radius, const NormalsSlab &sl, std::vector<OrientEdge> &forest,
                std::vector<OrientEdge> &cross, uint64_t *intra, int *needs)
{
    forest.clear();
    cross.clear();
    *intra = 0;
    *needs = 0;
    if (!ix) return PT_ERR_INVALID_ARG;
    if (ix->n == 0) return PT_OK;
    if (!ix->attrs || !ix->ids) return PT_ERR_INVALID_ARG;
    // edge offsets are uint32 and own rows carry a sign bit: the slab's records times k must fit an int
    if ((uint64_t)ix->n * (uint64_t)k > (uint64_t)INT32_MAX) return PT_ERR_UNSUPPORTED;
    PT_CUDA(cudaSetDevice(ix->device));
    return ix->coord_f64 ? orient_slab_t<PointD>(ix, k, radius, sl, forest, cross, intra, needs)
                         : orient_slab_t<PointF>(ix, k, radius, sl, forest, cross, intra, needs);
}

// The points of a sharded cloud on the home device, vertex = global id: the normals the slabs'
// records were built from, narrowed here as the build narrows them (NaNs included), and the caller's
// positions (pos: n x 3 with a viewpoint, else the n z values, zs apart)
struct OrientPoints {
    const double *normal;
    const double *pos;
    uint32_t zs;
    __device__ __forceinline__ float mf(size_t g, int a) const { return (float)normal[3 * g + a]; }
    __device__ __forceinline__ D3 m(uint32_t g) const { return D3{(double)mf(g, 0), (double)mf(g, 1), (double)mf(g, 2)}; }
    __device__ __forceinline__ bool part(uint32_t g) const { return d3_usable(m(g)); }
    __device__ __forceinline__ double z(uint32_t g) const { return pos[(size_t)zs * g + (zs - 1)]; }
};

__global__ void __launch_bounds__(256) orient_lab_kernel(uint32_t n, uint32_t *lab)
{
    PT_GRID_STRIDE(g, n) lab[g] = (uint32_t)g;
}

// orient_top_z_kernel / orient_top_id_kernel / orient_signs_kernel by global id
__global__ void __launch_bounds__(256) orient_top_z_points_kernel(const OrientPoints p, uint32_t n, const uint32_t *lab,
                                                                  unsigned long long *top_z)
{
    PT_GRID_STRIDE(g, n) {
        if (p.part((uint32_t)g)) atomicMax(top_z + rep_of(lab, (uint32_t)g), z_key(p.z((uint32_t)g)));
    }
}

__global__ void __launch_bounds__(256) orient_top_id_points_kernel(const OrientPoints p, uint32_t n, const uint32_t *lab,
                                                                   const unsigned long long *top_z, uint32_t *top_id)
{
    PT_GRID_STRIDE(g, n) {
        if (!p.part((uint32_t)g)) continue;
        const uint32_t c = rep_of(lab, (uint32_t)g);
        if (top_z[c] == z_key(p.z((uint32_t)g))) atomicMin(top_id + c, (uint32_t)g);
    }
}

__global__ void __launch_bounds__(256) orient_signs_points_kernel(const OrientPoints p, uint32_t n, const uint32_t *lab,
                                                                  const uint32_t *top_id, const OrientOut o)
{
    PT_GRID_STRIDE(g, n) {
        float mx = p.mf(g, 0), my = p.mf(g, 1), mz = p.mf(g, 2);
        const bool part = p.part((uint32_t)g);
        int32_t root = -1;
        bool flip = false;
        if (part) {
            const uint32_t c = rep_of(lab, (uint32_t)g);
            root = (int32_t)top_id[c];
            const D3 nr = d3_normalise(p.m((uint32_t)root));
            const bool neg = root_negates(o, nr, [&] { return d3_load(p.pos + 3 * (size_t)root); });
            flip = neg != (((lab[g] ^ lab[root]) & LAB_BIT) != 0);
            if (flip) { mx = -mx; my = -my; mz = -mz; }
        }
        o.normal[3 * g] = mx;
        o.normal[3 * g + 1] = my;
        o.normal[3 * g + 2] = mz;
        o.root[g] = root;
        orient_tally(o, part, flip, [&] { return part && rep_of(lab, (uint32_t)g) == (uint32_t)g; });
    }
}

// cross edges: keys[e] = their keys, idx[e] = e
__global__ void __launch_bounds__(256) orient_keys_kernel(const OrientEdge *edges, size_t m, unsigned long long *keys,
                                                          uint32_t *idx)
{
    PT_GRID_STRIDE(e, m) {
        keys[e] = edges[e].key;
        idx[e] = (uint32_t)e;
    }
}

__global__ void __launch_bounds__(256) orient_gather_kernel(const OrientEdge *edges, const uint32_t *idx, const int64_t *m,
                                                            OrientEdge *out)
{
    PT_GRID_STRIDE(e, (size_t)*m) out[e] = edges[idx[e]];
}

int orient_home(const OrientHome &h, const std::vector<std::vector<OrientEdge>> &forest,
                const std::vector<std::vector<OrientEdge>> &cross, uint64_t *unique_cross, unsigned long long counts[3],
                cudaStream_t s)
{
    const uint32_t n = (uint32_t)h.n;
    size_t n_f = 0, n_c = 0;
    for (const auto &f : forest) n_f += f.size();
    for (const auto &c : cross) n_c += c.size();
    if (n_c >= (size_t)INT32_MAX) return PT_ERR_UNSUPPORTED;      // cub's sort counts in an int
    const size_t pos_n = (h.viewpoint ? 3 : 1) * h.n;
    float *d_out = nullptr;
    double *d_normal = nullptr, *d_pos = nullptr;
    int32_t *d_root = nullptr;
    uint32_t *d_lab = nullptr, *d_hook = nullptr, *d_changed = nullptr, *d_idx = nullptr;
    unsigned long long *d_best_w = nullptr, *d_best_key = nullptr, *d_keys = nullptr, *d_counts = nullptr;
    OrientEdge *d_edges = nullptr, *d_cross = nullptr;
    int64_t *d_num = nullptr;
    void *d_tmp = nullptr;
    int rc = PT_OK;
    auto fail = [&](cudaError_t e) { if (e != cudaSuccess && rc == PT_OK) rc = map_cuda_error(e); return e != cudaSuccess; };
    auto oom = [&](bool bad) { if (bad && rc == PT_OK) rc = PT_ERR_OUT_OF_MEMORY; return bad; };
    auto launched = [&]() { count_launch(); return fail(cudaGetLastError()); };
    const unsigned gn = ocdiv(n, 256);
    do {
        if (oom(pool_alloc((void **)&d_edges, sizeof(OrientEdge) * std::max<size_t>(n_f + n_c, 1), s) ||
                pool_alloc((void **)&d_num, sizeof(int64_t) * 2 + sizeof(uint32_t), s)))
            break;
        d_changed = (uint32_t *)(d_num + 2);
        size_t at = 0;
        for (const auto &f : forest) {
            if (!f.empty() && fail(cudaMemcpyAsync(d_edges + at, f.data(), sizeof(OrientEdge) * f.size(),
                                                   cudaMemcpyHostToDevice, s)))
                break;
            at += f.size();
        }
        if (rc != PT_OK) break;
        // ---- the cross edges, sorted by key, each pair once
        size_t sort_bytes = 0, unique_bytes = 0, select_bytes = 0;
        int64_t n_u = 0;
        if (n_c) {
            if (oom(pool_alloc((void **)&d_cross, sizeof(OrientEdge) * n_c, s) ||
                    pool_alloc((void **)&d_keys, sizeof(unsigned long long) * 2 * n_c, s) ||
                    pool_alloc((void **)&d_idx, sizeof(uint32_t) * 2 * n_c, s)))
                break;
            at = 0;
            for (const auto &c : cross) {
                if (!c.empty() && fail(cudaMemcpyAsync(d_cross + at, c.data(), sizeof(OrientEdge) * c.size(),
                                                       cudaMemcpyHostToDevice, s)))
                    break;
                at += c.size();
            }
            if (rc != PT_OK) break;
            if (fail(cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, d_keys, d_keys + n_c, d_idx, d_idx + n_c, (int)n_c,
                                                     0, 64, s)) ||
                fail(cub::DeviceSelect::UniqueByKey(nullptr, unique_bytes, d_keys + n_c, d_idx + n_c, d_keys, d_idx, d_num,
                                                    (int)n_c, s)))
                break;
        }
        if (fail(cub::DeviceSelect::If(nullptr, select_bytes, d_edges, d_num, (int64_t)(n_f + n_c), OrientCrossing{d_lab}, s)))
            break;
        const size_t tmp_bytes = std::max(std::max(sort_bytes, unique_bytes), std::max(select_bytes, (size_t)1));
        if (oom(pool_alloc(&d_tmp, tmp_bytes, s))) break;
        if (n_c) {
            orient_keys_kernel<<<ocdiv(n_c, 256), 256, 0, s>>>(d_cross, n_c, d_keys, d_idx);
            if (launched()) break;
            if (fail(cub::DeviceRadixSort::SortPairs(d_tmp, sort_bytes, d_keys, d_keys + n_c, d_idx, d_idx + n_c, (int)n_c,
                                                     0, 64, s)) ||
                fail(cub::DeviceSelect::UniqueByKey(d_tmp, unique_bytes, d_keys + n_c, d_idx + n_c, d_keys, d_idx, d_num,
                                                    (int)n_c, s)))
                break;
            orient_gather_kernel<<<ocdiv(n_c, 256), 256, 0, s>>>(d_cross, d_idx, d_num, d_edges + n_f);
            if (launched() || fail(cudaMemcpyAsync(&n_u, d_num, sizeof n_u, cudaMemcpyDeviceToHost, s)) ||
                fail(cudaStreamSynchronize(s)))
                break;
            pool_free(d_cross, s);
            pool_free(d_keys, s);
            pool_free(d_idx, s);
            d_cross = nullptr; d_keys = nullptr; d_idx = nullptr;
        }
        *unique_cross = (uint64_t)n_u;
        // ---- the minimum spanning forest of the whole graph over the global ids
        if (oom(pool_alloc((void **)&d_lab, sizeof(uint32_t) * n, s) || pool_alloc((void **)&d_hook, sizeof(uint32_t) * n, s) ||
                pool_alloc((void **)&d_best_w, sizeof(unsigned long long) * n, s) ||
                pool_alloc((void **)&d_best_key, sizeof(unsigned long long) * n, s)))
            break;
        orient_lab_kernel<<<gn, 256, 0, s>>>(n, d_lab);
        if (launched()) break;
        if ((rc = orient_boruvka(d_edges, n_f + (size_t)n_u, n,
                                 OrientWork{d_lab, d_hook, d_changed, d_best_w, d_best_key, d_num, d_tmp, tmp_bytes}, s)) != PT_OK)
            break;
        pool_free(d_edges, s);
        d_edges = nullptr;
        // ---- roots, signs and outputs (best_w holds the top z keys, hook the top ids)
        if (oom(pool_alloc((void **)&d_normal, sizeof(double) * 3 * h.n, s) || pool_alloc((void **)&d_pos, sizeof(double) * pos_n, s) ||
                pool_alloc((void **)&d_out, sizeof(float) * 3 * h.n, s) || pool_alloc((void **)&d_root, sizeof(int32_t) * h.n, s) ||
                pool_alloc((void **)&d_counts, sizeof(unsigned long long) * 3, s)))
            break;
        if (fail(cudaMemcpyAsync(d_normal, h.normal, sizeof(double) * 3 * h.n, cudaMemcpyHostToDevice, s)) ||
            fail(cudaMemcpyAsync(d_pos, h.pos, sizeof(double) * pos_n, cudaMemcpyHostToDevice, s)) ||
            fail(cudaMemsetAsync(d_counts, 0, sizeof(unsigned long long) * 3, s)) ||
            fail(cudaMemsetAsync(d_best_w, 0, sizeof(unsigned long long) * n, s)) ||
            fail(cudaMemsetAsync(d_hook, 0xff, sizeof(uint32_t) * n, s)))
            break;
        const OrientPoints p{d_normal, d_pos, h.viewpoint ? 3u : 1u};
        OrientOut o{};
        o.has_view = h.viewpoint ? 1 : 0;
        if (h.viewpoint) { o.vx = h.viewpoint[0]; o.vy = h.viewpoint[1]; o.vz = h.viewpoint[2]; }
        o.normal = d_out;
        o.root = d_root;
        o.counts = d_counts;
        orient_top_z_points_kernel<<<gn, 256, 0, s>>>(p, n, d_lab, d_best_w);
        if (launched()) break;
        orient_top_id_points_kernel<<<gn, 256, 0, s>>>(p, n, d_lab, d_best_w, d_hook);
        if (launched()) break;
        orient_signs_points_kernel<<<gn, 256, 0, s>>>(p, n, d_lab, d_hook, o);
        if (launched()) break;
        if (fail(cudaMemcpyAsync(h.normal_out, d_out, sizeof(float) * 3 * h.n, cudaMemcpyDeviceToHost, s)) ||
            fail(cudaMemcpyAsync(h.root_out, d_root, sizeof(int32_t) * h.n, cudaMemcpyDeviceToHost, s)) ||
            fail(cudaMemcpyAsync(counts, d_counts, sizeof(unsigned long long) * 3, cudaMemcpyDeviceToHost, s)))
            break;
        fail(cudaStreamSynchronize(s));
    } while (0);
    cudaStreamSynchronize(s);
    void *frees[] = {d_normal, d_out, d_pos, d_root, d_lab, d_hook, d_idx, d_best_w, d_best_key, d_keys, d_counts,
                     d_edges, d_cross, d_num, d_tmp};
    for (void *q : frees) pool_free(q, s);
    cudaStreamSynchronize(s);
    cudaGetLastError();
    return rc;
}

int orient_check_args(int k, const double *viewpoint, bool store, bool any_output)
{
    if (!any_output && !store) return PT_ERR_INVALID_ARG;
    if (viewpoint && !(std::isfinite(viewpoint[0]) && std::isfinite(viewpoint[1]) && std::isfinite(viewpoint[2])))
        return PT_ERR_INVALID_ARG;
    if (k < 2) return PT_ERR_INVALID_ARG;             // a list of one holds only the point itself
    if (k > PT_MAX_K) return PT_ERR_UNSUPPORTED;
    return PT_OK;
}

}  // namespace pt

using namespace pt;

extern "C" int pt_index_orient_normals(pt_index *ix, int k, double radius, const double *viewpoint, int store,
                                       float *normal_out, int32_t *root_out, pt_orient_stats *stats)
{
    if (!ix) return PT_ERR_INVALID_ARG;
    const int arg_rc = orient_check_args(k, viewpoint, store != 0, normal_out || root_out);
    if (arg_rc != PT_OK) return arg_rc;
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

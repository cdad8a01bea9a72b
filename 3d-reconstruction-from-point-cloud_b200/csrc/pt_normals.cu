// pt_normals.cu -- PCA normal estimation over each cloud point's k nearest neighbours (DESIGN.md
// section 8, "Normal estimation"; CGAL's pca_estimate_normals, Open3D's and PCL's estimators).
//
// Per chunk of at most HEIGHT_CHUNK sorted records: the records' positions become the query rows
// (row r = sorted record r, so the k-NN kernels see coherent samples), one launch_query writes the
// neighbour lists, and normals_pca_kernel turns every list into a normal and a surface variation.
// Everything is fp64 with every operation rounded on its own, in the order DESIGN.md states, so
// that oracle/pt_normals_oracle.c equals it bit for bit.  A sharded cloud (pt_sharded.cu) runs the
// same kernels per slab over the rows of the records the slab owns (normals_slab, DESIGN.md
// section 8, "Sharded normal estimation").
#include <algorithm>
#include <cmath>
#include <vector>

#include <cub/device/device_select.cuh>
#include <thrust/iterator/counting_iterator.h>

#include "pt_bake.cuh"
#include "pt_fp64.cuh"

namespace pt {

constexpr uint32_t NORMALS_NAN = 0x7fc00000u;   // the variation of a point without an estimate
constexpr int JACOBI_MAX_SWEEPS = 50;

static inline unsigned ncdiv(size_t a, size_t b) { return (unsigned)((a + b - 1) / b); }

// Query row i of a chunk is sorted record r0 + i, or with LIST sorted record rows[r0 + i].
template <typename PT, bool LIST>
__device__ __forceinline__ void normals_rows(const PT *pts, const uint32_t *rows, uint32_t r0, uint32_t count, double *xyz)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    const PT rec = pts[LIST ? rows[r0 + i] : r0 + i];
    xyz[3 * (size_t)i] = (double)rec.x;
    xyz[3 * (size_t)i + 1] = (double)rec.y;
    xyz[3 * (size_t)i + 2] = (double)rec.z;
}

template <typename PT>
__global__ void __launch_bounds__(256) normals_rows_kernel(const PT *pts, uint32_t r0, uint32_t count, double *xyz)
{
    normals_rows<PT, false>(pts, nullptr, r0, count, xyz);
}

template <typename PT>
__global__ void __launch_bounds__(256)
normals_rows_list_kernel(const PT *pts, const uint32_t *rows, uint32_t r0, uint32_t count, double *xyz)
{
    normals_rows<PT, true>(pts, rows, r0, count, xyz);
}

// ROTATE of Numerical Recipes' jacobi: (g, h) <- (g - s (h + g tau), h + s (g - h tau))
__device__ __forceinline__ void jacobi_rotate(double &gr, double &hr, double s, double tau)
{
    const double g = gr, h = hr;
    gr = __dsub_rn(g, __dmul_rn(s, __dadd_rn(h, __dmul_rn(g, tau))));
    hr = __dadd_rn(h, __dmul_rn(s, __dsub_rn(g, __dmul_rn(h, tau))));
}

// pivot (P, Q) of sweep `sweep` (1-based); a holds the upper triangle
template <int P, int Q>
__device__ __forceinline__ void jacobi_pivot(double a[3][3], double v[3][3], double d[3], double z[3], int sweep,
                                             double tresh)
{
    const double apq = a[P][Q];
    const double g = __dmul_rn(100.0, fabs(apq));
    if (sweep > 4 && __dadd_rn(fabs(d[P]), g) == fabs(d[P]) && __dadd_rn(fabs(d[Q]), g) == fabs(d[Q])) {
        a[P][Q] = 0.0;
        return;
    }
    if (!(fabs(apq) > tresh)) return;
    double h = __dsub_rn(d[Q], d[P]);
    double t;
    if (__dadd_rn(fabs(h), g) == fabs(h)) {
        t = __ddiv_rn(apq, h);
    } else {
        const double theta = __ddiv_rn(__dmul_rn(0.5, h), apq);
        t = __ddiv_rn(1.0, __dadd_rn(fabs(theta), __dsqrt_rn(__dadd_rn(1.0, __dmul_rn(theta, theta)))));
        if (theta < 0.0) t = -t;
    }
    const double c = __ddiv_rn(1.0, __dsqrt_rn(__dadd_rn(1.0, __dmul_rn(t, t))));
    const double s = __dmul_rn(t, c);
    const double tau = __ddiv_rn(s, __dadd_rn(1.0, c));
    h = __dmul_rn(t, apq);
    z[P] = __dsub_rn(z[P], h);
    z[Q] = __dadd_rn(z[Q], h);
    d[P] = __dsub_rn(d[P], h);
    d[Q] = __dadd_rn(d[Q], h);
    a[P][Q] = 0.0;
    if (P == 0 && Q == 1) jacobi_rotate(a[0][2], a[1][2], s, tau);
    if (P == 0 && Q == 2) jacobi_rotate(a[0][1], a[1][2], s, tau);
    if (P == 1 && Q == 2) jacobi_rotate(a[0][1], a[0][2], s, tau);
#pragma unroll
    for (int j = 0; j < 3; ++j) jacobi_rotate(v[j][P], v[j][Q], s, tau);
}

// Cyclic Jacobi on the symmetric scatter matrix: eigenvalues d, eigenvectors in the columns of v.
__device__ __forceinline__ void jacobi3(const double c[6], double d[3], double v[3][3])
{
    double a[3][3] = {{c[0], c[1], c[2]}, {0.0, c[3], c[4]}, {0.0, 0.0, c[5]}};
    double b[3] = {c[0], c[3], c[5]}, z[3] = {0.0, 0.0, 0.0};
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        d[i] = b[i];
#pragma unroll
        for (int j = 0; j < 3; ++j) v[i][j] = i == j ? 1.0 : 0.0;
    }
    for (int sweep = 1; sweep <= JACOBI_MAX_SWEEPS; ++sweep) {
        const double sm = __dadd_rn(__dadd_rn(fabs(a[0][1]), fabs(a[0][2])), fabs(a[1][2]));
        if (sm == 0.0) break;
        const double tresh = sweep < 4 ? __ddiv_rn(__dmul_rn(0.2, sm), 9.0) : 0.0;
        jacobi_pivot<0, 1>(a, v, d, z, sweep, tresh);
        jacobi_pivot<0, 2>(a, v, d, z, sweep, tresh);
        jacobi_pivot<1, 2>(a, v, d, z, sweep, tresh);
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            b[i] = __dadd_rn(b[i], z[i]);
            d[i] = b[i];
            z[i] = 0.0;
        }
    }
}

struct NormalsOut {
    const pt_attr *attrs;     // input normals, original order (may be null: rule (a) never applies)
    pt_attr *store;           // store: attrs (original order), else null
    pt_attr *store_curve;     // store: attrs_curve (sorted order) where the index has it, else null
    int has_view;
    double vx, vy, vz;
    float *normal;            // n x 3, original order (may be null)
    float *variation;         // n, original order (may be null)
    unsigned long long *estimated;   // += points with an estimate (may be null)
};

// A warp takes 32 consecutive rows (sorted records r0 + base ..).  It walks them in `width` rounds, a
// group of `width` (the power of two >= k) lanes per row: lane j of a group gathers neighbour j
// through the inverse permutation (independent random reads, in parallel), and the group forms the
// centroid and then the six scatter sums in neighbour order through shuffles.  The sums go to the
// row's own lane, and after the rounds every lane solves its row's 3 x 3 on its own, so the Jacobi
// sweeps run 32 rows wide.  Every lane runs the same loops, so the shuffles see the full warp.
// With LIST, row r0 + i of the chunk is sorted record rows[r0 + i] instead of r0 + i.
template <typename PT, bool LIST>
__device__ __forceinline__ void normals_pca(const PT *pts, const uint32_t *inv, uint32_t n_points, const uint32_t *rows,
                                            uint32_t r0, uint32_t count, const int32_t *idx, int k, int width,
                                            const NormalsOut &o)
{
    const unsigned lane = threadIdx.x & 31u;
    const uint32_t base = (uint32_t)(((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5) * 32u;
    if (base >= count) return;                                    // warp-uniform
    const bool mine = base + lane < count;
    const PosSorted<PT> pos{pts, inv};
    double c[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    int my_cnt = 0;
    const unsigned per_round = 32u / (unsigned)width;
    const unsigned g = lane / (unsigned)width, j = lane % (unsigned)width, g0 = g * (unsigned)width;
    const int from = (int)((lane % per_round) * (unsigned)width);  // a lane of the group that sums my row
    for (unsigned r = 0; r < (unsigned)width; ++r) {
        const uint32_t s = base + r * per_round + g;
        bool has = false;
        D3 p = {0.0, 0.0, 0.0};
        if (s < count && (int)j < k) {
            const int id = idx[(size_t)s * k + j];
            if (id >= 0 && (uint32_t)id < n_points) {
                double x[3];
                pos.get(id, x);
                p = D3{x[0], x[1], x[2]};
                has = true;
            }
        }
        // the list is its leading run of valid entries
        const unsigned seg = (__ballot_sync(0xffffffffu, has) >> g0) & (width == 32 ? 0xffffffffu : ((1u << width) - 1u));
        const int cnt = __ffsll(~(unsigned long long)seg) - 1;
        D3 sum = {0.0, 0.0, 0.0};
        for (int jj = 0; jj < k; ++jj) {
            const D3 q = {shfl_d(p.x, (int)g0 + jj), shfl_d(p.y, (int)g0 + jj), shfl_d(p.z, (int)g0 + jj)};
            if (jj < cnt) sum = d3_add(sum, q);
        }
        const double dc = (double)cnt;
        const D3 e = d3_sub(p, D3{__ddiv_rn(sum.x, dc), __ddiv_rn(sum.y, dc), __ddiv_rn(sum.z, dc)});
        const double t[6] = {__dmul_rn(e.x, e.x), __dmul_rn(e.x, e.y), __dmul_rn(e.x, e.z),
                             __dmul_rn(e.y, e.y), __dmul_rn(e.y, e.z), __dmul_rn(e.z, e.z)};
        double acc[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
        for (int jj = 0; jj < k; ++jj) {
#pragma unroll
            for (int a = 0; a < 6; ++a) {
                const double tj = shfl_d(t[a], (int)g0 + jj);
                if (jj < cnt) acc[a] = __dadd_rn(acc[a], tj);
            }
        }
        const bool take = lane / per_round == r;
#pragma unroll
        for (int a = 0; a < 6; ++a) {
            const double v = shfl_d(acc[a], from);
            if (take) c[a] = v;
        }
        const int tc = __shfl_sync(0xffffffffu, cnt, from);
        if (take) my_cnt = tc;
    }
    if (!mine) return;

    const uint32_t row = LIST ? rows[r0 + base + lane] : r0 + base + lane;
    const PT rec = pts[row];
    const uint32_t orig = (uint32_t)rec.idx;
    const D3 pi = {(double)rec.x, (double)rec.y, (double)rec.z};
    const double trace = __dadd_rn(__dadd_rn(c[0], c[3]), c[5]);
    bool est = my_cnt >= 3 && trace > 0.0 && trace < INFINITY;
    D3 n = {0.0, 0.0, 0.0};
    double lam0 = 0.0;
    if (est) {
        double d[3], v[3][3];
        jacobi3(c, d, v);
        // the smallest eigenvalue, the lower column on ties (selects, not a dynamic index: no local memory)
        lam0 = d[0];
        D3 col = {v[0][0], v[1][0], v[2][0]};
        if (d[1] < lam0) { lam0 = d[1]; col = D3{v[0][1], v[1][1], v[2][1]}; }
        if (d[2] < lam0) { lam0 = d[2]; col = D3{v[0][2], v[1][2], v[2][2]}; }
        n = d3_normalise(col);
        est = d3_usable(n);
    }
    if (est) {
        bool flip;
        const pt_attr m = o.attrs ? o.attrs[orig] : pt_attr{};
        const D3 md = {(double)m.nx, (double)m.ny, (double)m.nz};
        if (o.attrs && d3_usable(md)) {
            flip = d3_dot(n, md) < 0.0;                                             // (a) input normal
        } else if (o.has_view) {
            flip = d3_dot(n, d3_sub(D3{o.vx, o.vy, o.vz}, pi)) < 0.0;               // (b) viewpoint
        } else {
            const double ax = fabs(n.x), ay = fabs(n.y), az = fabs(n.z);      // (c) largest component
            flip = (ax >= ay && ax >= az) ? n.x < 0.0 : (ay >= az ? n.y < 0.0 : n.z < 0.0);
        }
        if (flip) n = D3{-n.x, -n.y, -n.z};
    }
    const float fx = __double2float_rn(n.x), fy = __double2float_rn(n.y), fz = __double2float_rn(n.z);
    if (o.normal) {
        o.normal[3 * (size_t)orig] = fx;
        o.normal[3 * (size_t)orig + 1] = fy;
        o.normal[3 * (size_t)orig + 2] = fz;
    }
    if (o.variation)
        o.variation[orig] = est ? __double2float_rn(__ddiv_rn(lam0 > 0.0 ? lam0 : 0.0, trace)) : __uint_as_float(NORMALS_NAN);
    if (est && o.store) {
        o.store[orig].nx = fx; o.store[orig].ny = fy; o.store[orig].nz = fz;
        if (o.store_curve) { o.store_curve[row].nx = fx; o.store_curve[row].ny = fy; o.store_curve[row].nz = fz; }
    }
    if (o.estimated) {
        const unsigned act = __activemask();
        const unsigned got = __ballot_sync(act, est);
        if (got && lane == (unsigned)(__ffs(act) - 1)) atomicAdd(o.estimated, (unsigned long long)__popc(got));
    }
}

template <typename PT>
__global__ void __launch_bounds__(256)
normals_pca_kernel(const PT *pts, const uint32_t *inv, uint32_t n_points, uint32_t r0, uint32_t count,
                   const int32_t *idx, int k, int width, const NormalsOut o)
{
    normals_pca<PT, false>(pts, inv, n_points, nullptr, r0, count, idx, k, width, o);
}

template <typename PT>
__global__ void __launch_bounds__(256)
normals_pca_list_kernel(const PT *pts, const uint32_t *inv, uint32_t n_points, const uint32_t *rows, uint32_t r0,
                        uint32_t count, const int32_t *idx, int k, int width, const NormalsOut o)
{
    normals_pca<PT, true>(pts, inv, n_points, rows, r0, count, idx, k, width, o);
}

static int normals_width(int k)
{
    int w = 1;
    while (w < k) w <<= 1;
    return w;
}

cudaError_t record_mark(std::vector<cudaEvent_t> *marks, cudaStream_t s)
{
    if (!marks) return cudaSuccess;
    marks->emplace_back();
    const cudaError_t e = cudaEventCreate(&marks->back());
    return e != cudaSuccess ? e : cudaEventRecord(marks->back(), s);
}

template <typename PT>
static int self_query_chunks_t(pt_index *ix, int k, double radius, int32_t *lists, bool keep, const ChunkThen &then,
                               std::vector<cudaEvent_t> *marks, cudaStream_t s, const uint32_t *rows, uint32_t n_rows,
                               const BakeGhost *ghost)
{
    const uint32_t n = rows ? n_rows : ix->n;
    const size_t chunk = std::min((size_t)HEIGHT_CHUNK, (size_t)n);
    double *d_q = nullptr, *d_d2 = nullptr;
    int rc = PT_OK;
    auto fail = [&](cudaError_t e) { if (e != cudaSuccess && rc == PT_OK) rc = map_cuda_error(e); return e != cudaSuccess; };
    do {
        if (fail(record_mark(marks, s))) break;
        // built once per index on its own stream, which every later user of it is ordered after
        const bool fresh = ix->inv_perm == nullptr;
        if ((rc = index_inverse_perm(ix)) != PT_OK) break;
        if (fresh && s != ix->stream && fail(cudaStreamSynchronize(ix->stream))) break;
        if (pool_alloc((void **)&d_q, sizeof(double) * 3 * chunk, s) ||
            (ghost && pool_alloc((void **)&d_d2, sizeof(double) * k * chunk, s))) {
            rc = PT_ERR_OUT_OF_MEMORY;
            break;
        }
        QueryParams qp{};
        fill_params(ix, qp);
        qp.ids = nullptr;          // the index's own ids: the callers read its records by them
        qp.k = k;
        qp.r2 = radius_to_r2(radius);
        qp.queries = d_q;
        qp.d2_out = d_d2;
        const PT *pts = (const PT *)ix->pts;
        for (size_t c0 = 0; c0 < n; c0 += chunk) {
            const uint32_t cm = (uint32_t)std::min(chunk, (size_t)n - c0);
            if (rows)
                normals_rows_list_kernel<PT><<<ncdiv(cm, 256), 256, 0, s>>>(pts, rows, (uint32_t)c0, cm, d_q);
            else
                normals_rows_kernel<PT><<<ncdiv(cm, 256), 256, 0, s>>>(pts, (uint32_t)c0, cm, d_q);
            count_launch();
            qp.m = cm;
            qp.idx_out = keep ? lists + c0 * (size_t)k : lists;
            if ((rc = launch_query(ix, qp, s)) != PT_OK) break;
            if (ghost && (rc = launch_ghost_check(d_q, d_d2, cm, k, qp.r2, ghost->boxes, ghost->n_ranks, ghost->self,
                                                  ghost->halo, ghost->flag, s)) != PT_OK)
                break;
            if (fail(record_mark(marks, s))) break;
            if ((rc = then((uint32_t)c0, cm, qp.idx_out)) != PT_OK) break;
        }
    } while (0);
    pool_free(d_q, s);
    pool_free(d_d2, s);
    return rc;
}

int self_query_chunks(pt_index *ix, int k, double radius, int32_t *lists, bool keep, const ChunkThen &then,
                      std::vector<cudaEvent_t> *marks, cudaStream_t s, const uint32_t *rows, uint32_t n_rows,
                      const BakeGhost *ghost)
{
    return ix->coord_f64 ? self_query_chunks_t<PointD>(ix, k, radius, lists, keep, then, marks, s, rows, n_rows, ghost)
                         : self_query_chunks_t<PointF>(ix, k, radius, lists, keep, then, marks, s, rows, n_rows, ghost);
}

// All points of ix in chunks, asynchronous on s.  marks (may be null): an event before the first
// chunk and after each chunk's query and PCA kernel.
template <typename PT>
static int normals_run(pt_index *ix, int k, double radius, const NormalsOut &o, std::vector<cudaEvent_t> *marks,
                       cudaStream_t s)
{
    const uint32_t n = ix->n;
    int32_t *d_idx = nullptr;
    if (pool_alloc((void **)&d_idx, sizeof(int32_t) * k * std::min((size_t)HEIGHT_CHUNK, (size_t)n), s))
        return PT_ERR_OUT_OF_MEMORY;
    const int rc = self_query_chunks(
        ix, k, radius, d_idx, false,
        [&](uint32_t c0, uint32_t cm, const int32_t *idx) {
            normals_pca_kernel<PT><<<ncdiv(cm, 256), 256, 0, s>>>((const PT *)ix->pts, ix->inv_perm, n, c0, cm, idx, k,
                                                                  normals_width(k), o);
            count_launch();
            cudaError_t e = cudaGetLastError();
            if (e == cudaSuccess) e = record_mark(marks, s);
            return e == cudaSuccess ? PT_OK : map_cuda_error(e);
        },
        marks, s);
    pool_free(d_idx, s);
    return rc;
}

int normals_check_args(int k, const double *viewpoint, bool store, bool any_output)
{
    if (!any_output && !store) return PT_ERR_INVALID_ARG;
    if (viewpoint && !(std::isfinite(viewpoint[0]) && std::isfinite(viewpoint[1]) && std::isfinite(viewpoint[2])))
        return PT_ERR_INVALID_ARG;
    if (k < 3) return PT_ERR_INVALID_ARG;             // a plane needs three points
    if (k > PT_MAX_K) return PT_ERR_UNSUPPORTED;
    return PT_OK;
}

static int normals_check(const pt_index *ix, int k, const double *viewpoint, bool store, bool any_output)
{
    if (!ix) return PT_ERR_INVALID_ARG;
    const int rc = normals_check_args(k, viewpoint, store, any_output);
    if (rc != PT_OK) return rc;
    if (store && !ix->attrs && ix->n) return PT_ERR_INVALID_ARG;
    if (pt_device_count() == 0) return PT_ERR_NO_DEVICE;
    return PT_OK;
}

static NormalsOut normals_out(pt_index *ix, const double *viewpoint, bool store, float *normal, float *variation,
                              unsigned long long *estimated)
{
    NormalsOut o{};
    o.attrs = ix->attrs;
    o.store = store ? ix->attrs : nullptr;
    o.store_curve = store ? ix->attrs_curve : nullptr;
    o.has_view = viewpoint ? 1 : 0;
    if (viewpoint) { o.vx = viewpoint[0]; o.vy = viewpoint[1]; o.vz = viewpoint[2]; }
    o.normal = normal;
    o.variation = variation;
    o.estimated = estimated;
    return o;
}

static int normals_device(pt_index *ix, int k, double radius, const NormalsOut &o, std::vector<cudaEvent_t> *marks,
                          cudaStream_t s)
{
    return ix->coord_f64 ? normals_run<PointD>(ix, k, radius, o, marks, s) : normals_run<PointF>(ix, k, radius, o, marks, s);
}

// ---- sharded clouds (DESIGN.md section 8, "Sharded normal estimation") ------------------------------
// A slab's own records: the host's cut rule on the stored x, which widens to the caller's x exactly
// in both storage modes, so this is the owner build_slabs gave the point.
template <typename PT>
struct SlabOwnRow {
    const PT *pts;
    const double *cuts;       // device, n_cuts ascending
    int n_cuts, self;
    __device__ __forceinline__ bool operator()(uint32_t r) const
    {
        const double x = (double)pts[r].x;
        int slab = 0;
        for (int j = 0; j < n_cuts; ++j) slab += !(x < cuts[j]) ? 1 : 0;
        return slab == self;
    }
};

// ... and the same rule by local id i (the record at sorted position inv[i])
template <typename PT>
struct SlabOwnLocal {
    SlabOwnRow<PT> own;
    const uint32_t *inv;
    __device__ __forceinline__ bool operator()(uint32_t i) const { return own(inv[i]); }
};

// row j of the compact outputs takes the results of local id own[j]
__global__ void __launch_bounds__(256)
normals_compact_kernel(const uint32_t *own, uint32_t m, const float *normal, const float *variation, float *c_normal,
                       float *c_variation)
{
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= m) return;
    const uint32_t i = own[j];
    c_normal[3 * (size_t)j] = normal[3 * (size_t)i];
    c_normal[3 * (size_t)j + 1] = normal[3 * (size_t)i + 1];
    c_normal[3 * (size_t)j + 2] = normal[3 * (size_t)i + 2];
    c_variation[j] = variation[i];
}

// attrs[i] and attrs_curve[inv[i]] take the normal values[i] where its x is not NaN
__global__ void __launch_bounds__(256)
normals_store_kernel(const float *values, uint32_t n, const uint32_t *inv, pt_attr *attrs, pt_attr *attrs_curve)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float x = values[3 * (size_t)i];
    if (x != x) return;
    const float y = values[3 * (size_t)i + 1], z = values[3 * (size_t)i + 2];
    attrs[i].nx = x; attrs[i].ny = y; attrs[i].nz = z;
    if (attrs_curve) {
        const uint32_t r = inv[i];
        attrs_curve[r].nx = x; attrs_curve[r].ny = y; attrs_curve[r].nz = z;
    }
}

template <typename PT>
static int slab_rows_select_t(pt_index *ix, const NormalsSlab &sl, SlabRows &w)
{
    cudaStream_t s = ix->stream;
    const uint32_t n = ix->n;
    int rc = PT_OK;
    auto fail = [&](cudaError_t e) { if (e != cudaSuccess && rc == PT_OK) rc = map_cuda_error(e); return e != cudaSuccess; };
    do {
        if (sl.n_slabs < 1 || sl.n_slabs > BAKE_MAX_SLABS || sl.self < 0 || sl.self >= sl.n_slabs) {
            rc = PT_ERR_INVALID_ARG;
            break;
        }
        const int R = sl.n_slabs;
        if (pool_alloc((void **)&w.boxes, sizeof(double) * (7 * R - 1), s) ||
            pool_alloc((void **)&w.rows, sizeof(uint32_t) * n, s) || pool_alloc((void **)&w.count, sizeof(uint32_t), s) ||
            pool_alloc((void **)&w.flag, sizeof(uint32_t), s)) {
            rc = PT_ERR_OUT_OF_MEMORY;
            break;
        }
        if (fail(cudaMemcpyAsync(w.boxes, sl.boxes, sizeof(double) * 6 * R, cudaMemcpyHostToDevice, s)) ||
            (R > 1 && fail(cudaMemcpyAsync(w.boxes + 6 * R, sl.cuts, sizeof(double) * (R - 1), cudaMemcpyHostToDevice, s))) ||
            fail(cudaMemsetAsync(w.flag, 0, sizeof(uint32_t), s)))
            break;
        // the own records in ascending sorted position, so the self-queries stay curve-coherent
        const SlabOwnRow<PT> own{(const PT *)ix->pts, w.boxes + 6 * R, R - 1, sl.self};
        thrust::counting_iterator<uint32_t> ids(0);
        size_t row_bytes = 0, local_bytes = 0;
        if (fail(cub::DeviceSelect::If(nullptr, row_bytes, ids, w.rows, w.count, (int)n, own, s)) ||
            fail(cub::DeviceSelect::If(nullptr, local_bytes, ids, w.rows, w.count, (int)n, SlabOwnLocal<PT>{own, nullptr}, s)))
            break;
        w.tmp_bytes = std::max(std::max(row_bytes, local_bytes), (size_t)1);
        if (pool_alloc(&w.tmp, w.tmp_bytes, s)) {
            rc = PT_ERR_OUT_OF_MEMORY;
            break;
        }
        if (fail(cub::DeviceSelect::If(w.tmp, row_bytes, ids, w.rows, w.count, (int)n, own, s))) break;
        count_launch();
        if (fail(cudaMemcpyAsync(&w.n_rows, w.count, sizeof w.n_rows, cudaMemcpyDeviceToHost, s)) ||
            fail(cudaStreamSynchronize(s)))
            break;
        // the records this rule selects are the ones build_slabs counted as the slab's own
        if (w.n_rows != sl.n_own) rc = PT_ERR_UNSUPPORTED;
    } while (0);
    return rc;
}

int slab_rows_select(pt_index *ix, const NormalsSlab &sl, SlabRows &w)
{
    return ix->coord_f64 ? slab_rows_select_t<PointD>(ix, sl, w) : slab_rows_select_t<PointF>(ix, sl, w);
}

int slab_rows_query(pt_index *ix, int k, double radius, const NormalsSlab &sl, const SlabRows &w, int32_t *lists,
                    bool keep, const ChunkThen &then, std::vector<cudaEvent_t> *marks)
{
    const BakeGhost ghost{w.boxes, sl.n_slabs, sl.self, sl.halo, w.flag};
    return self_query_chunks(ix, k, radius, lists, keep, then, marks, ix->stream, w.rows, w.n_rows,
                             sl.check ? &ghost : nullptr);
}

void slab_rows_free(SlabRows &w, cudaStream_t s)
{
    void *frees[] = {w.boxes, w.rows, w.count, w.flag, w.tmp};
    for (void *p : frees) pool_free(p, s);
    w = SlabRows{};
}

template <typename PT>
static int normals_slab_t(pt_index *ix, int k, double radius, const double *viewpoint, const NormalsSlab &sl,
                          float *normal_out, float *variation_out, unsigned long long *estimated, float *pca_ms,
                          int *needs)
{
    cudaStream_t s = ix->stream;
    const uint32_t n = ix->n;
    SlabRows w;
    int32_t *d_idx = nullptr;
    float *d_normal = nullptr, *d_var = nullptr, *d_cnormal = nullptr, *d_cvar = nullptr;
    unsigned long long *d_est = nullptr, est = 0;
    uint32_t flag = 0;
    std::vector<cudaEvent_t> marks;
    int rc = PT_OK;
    auto fail = [&](cudaError_t e) { if (e != cudaSuccess && rc == PT_OK) rc = map_cuda_error(e); return e != cudaSuccess; };
    do {
        if ((rc = slab_rows_select_t<PT>(ix, sl, w)) != PT_OK) break;
        const uint32_t n_rows = w.n_rows;
        if (n_rows == 0) break;
        const size_t chunk = std::min((size_t)HEIGHT_CHUNK, (size_t)n_rows);
        if (pool_alloc((void **)&d_idx, sizeof(int32_t) * k * chunk, s) ||
            pool_alloc((void **)&d_normal, sizeof(float) * 3 * n, s) || pool_alloc((void **)&d_var, sizeof(float) * n, s) ||
            pool_alloc((void **)&d_cnormal, sizeof(float) * 3 * n_rows, s) ||
            pool_alloc((void **)&d_cvar, sizeof(float) * n_rows, s) || pool_alloc((void **)&d_est, sizeof(unsigned long long), s)) {
            rc = PT_ERR_OUT_OF_MEMORY;
            break;
        }
        if (fail(cudaMemsetAsync(d_est, 0, sizeof(unsigned long long), s))) break;
        // no store here: the caller stores once every slab has passed its check
        const NormalsOut o = normals_out(ix, viewpoint, false, d_normal, d_var, d_est);
        rc = slab_rows_query(
            ix, k, radius, sl, w, d_idx, false,
            [&](uint32_t c0, uint32_t cm, const int32_t *idx) {
                normals_pca_list_kernel<PT><<<ncdiv(cm, 256), 256, 0, s>>>((const PT *)ix->pts, ix->inv_perm, n, w.rows, c0,
                                                                           cm, idx, k, normals_width(k), o);
                count_launch();
                cudaError_t e = cudaGetLastError();
                if (e == cudaSuccess) e = record_mark(&marks, s);
                return e == cudaSuccess ? PT_OK : map_cuda_error(e);
            },
            &marks);
        if (rc != PT_OK) break;
        // only the own records' results travel to the host, in ascending local id (the order of their
        // global ids); the row list is free again in stream order and takes their local ids
        const SlabOwnRow<PT> own{(const PT *)ix->pts, w.boxes + 6 * sl.n_slabs, sl.n_slabs - 1, sl.self};
        if (fail(cub::DeviceSelect::If(w.tmp, w.tmp_bytes, thrust::counting_iterator<uint32_t>(0), w.rows, w.count, (int)n,
                                       SlabOwnLocal<PT>{own, ix->inv_perm}, s)))
            break;
        count_launch();
        normals_compact_kernel<<<ncdiv(n_rows, 256), 256, 0, s>>>(w.rows, n_rows, d_normal, d_var, d_cnormal, d_cvar);
        count_launch();
        if (fail(cudaGetLastError())) break;
        if (fail(cudaMemcpyAsync(normal_out, d_cnormal, sizeof(float) * 3 * n_rows, cudaMemcpyDeviceToHost, s)) ||
            fail(cudaMemcpyAsync(variation_out, d_cvar, sizeof(float) * n_rows, cudaMemcpyDeviceToHost, s)) ||
            fail(cudaMemcpyAsync(&est, d_est, sizeof est, cudaMemcpyDeviceToHost, s)) ||
            fail(cudaMemcpyAsync(&flag, w.flag, sizeof flag, cudaMemcpyDeviceToHost, s)) || fail(cudaStreamSynchronize(s)))
            break;
        *estimated += est;
        *needs = sl.check && flag ? 1 : 0;
        // marks: start, then per chunk (after the query and check, after the PCA kernel)
        float t = 0.0f;
        for (size_t c = 1; c + 1 < marks.size(); c += 2)
            if (cudaEventElapsedTime(&t, marks[c], marks[c + 1]) == cudaSuccess) *pca_ms += t;
    } while (0);
    cudaStreamSynchronize(s);
    slab_rows_free(w, s);
    void *frees[] = {d_idx, d_normal, d_var, d_cnormal, d_cvar, d_est};
    for (void *p : frees) pool_free(p, s);
    for (auto &e : marks) if (e) cudaEventDestroy(e);
    cudaStreamSynchronize(s);
    cudaGetLastError();
    return rc;
}

int normals_slab(pt_index *ix, int k, double radius, const double *viewpoint, const NormalsSlab &sl,
                 float *normal_out, float *variation_out, unsigned long long *estimated, float *pca_ms, int *needs)
{
    *pca_ms = 0.0f;
    *needs = 0;
    if (!ix) return PT_ERR_INVALID_ARG;
    if (ix->n == 0) return PT_OK;
    PT_CUDA(cudaSetDevice(ix->device));
    return ix->coord_f64
               ? normals_slab_t<PointD>(ix, k, radius, viewpoint, sl, normal_out, variation_out, estimated, pca_ms, needs)
               : normals_slab_t<PointF>(ix, k, radius, viewpoint, sl, normal_out, variation_out, estimated, pca_ms, needs);
}

int normals_store(pt_index *ix, const float *values)
{
    if (!ix) return PT_ERR_INVALID_ARG;
    if (ix->n == 0) return PT_OK;             // an empty index (a slab that owns nothing) has no attrs
    if (!ix->attrs) return PT_ERR_INVALID_ARG;
    PT_CUDA(cudaSetDevice(ix->device));
    cudaStream_t s = ix->stream;
    const uint32_t n = ix->n;
    float *d_values = nullptr;
    int rc = index_inverse_perm(ix);
    auto fail = [&](cudaError_t e) { if (e != cudaSuccess && rc == PT_OK) rc = map_cuda_error(e); return e != cudaSuccess; };
    do {
        if (rc != PT_OK) break;
        if (pool_alloc((void **)&d_values, sizeof(float) * 3 * n, s)) {
            rc = PT_ERR_OUT_OF_MEMORY;
            break;
        }
        if (fail(cudaMemcpyAsync(d_values, values, sizeof(float) * 3 * n, cudaMemcpyHostToDevice, s))) break;
        normals_store_kernel<<<ncdiv(n, 256), 256, 0, s>>>(d_values, n, ix->inv_perm, ix->attrs, ix->attrs_curve);
        count_launch();
        if (fail(cudaGetLastError())) break;
        fail(cudaStreamSynchronize(s));
    } while (0);
    cudaStreamSynchronize(s);
    pool_free(d_values, s);
    cudaStreamSynchronize(s);
    cudaGetLastError();
    return rc;
}

}  // namespace pt

using namespace pt;

extern "C" int pt_estimate_normals_device(pt_index *ix, int k, double radius, const double *viewpoint, int store,
                                          float *normal_out, float *variation_out, void *stream)
{
    const int rc = normals_check(ix, k, viewpoint, store != 0, normal_out || variation_out);
    if (rc != PT_OK) return rc;
    if (ix->n == 0) return PT_OK;
    PT_CUDA(cudaSetDevice(ix->device));
    return normals_device(ix, k, radius, normals_out(ix, viewpoint, store != 0, normal_out, variation_out, nullptr),
                          nullptr, (cudaStream_t)stream);
}

extern "C" int pt_index_estimate_normals(pt_index *ix, int k, double radius, const double *viewpoint, int store,
                                         float *normal_out, float *variation_out, pt_normals_stats *stats)
{
    int rc = normals_check(ix, k, viewpoint, store != 0, normal_out || variation_out);
    if (rc != PT_OK) return rc;
    if (stats) *stats = pt_normals_stats{0, 0.0f, 0.0f};
    if (ix->n == 0) return PT_OK;
    PT_CUDA(cudaSetDevice(ix->device));
    cudaStream_t s = ix->stream;
    const size_t n = ix->n;
    float *d_normal = nullptr, *d_var = nullptr;
    unsigned long long *d_est = nullptr, est = 0;
    std::vector<cudaEvent_t> marks;
    auto fail = [&](cudaError_t e) { if (e != cudaSuccess && rc == PT_OK) rc = map_cuda_error(e); return e != cudaSuccess; };
    do {
        if ((normal_out && pool_alloc((void **)&d_normal, sizeof(float) * 3 * n, s)) ||
            (variation_out && pool_alloc((void **)&d_var, sizeof(float) * n, s)) ||
            pool_alloc((void **)&d_est, sizeof(unsigned long long), s)) {
            rc = PT_ERR_OUT_OF_MEMORY;
            break;
        }
        if (fail(cudaMemsetAsync(d_est, 0, sizeof(unsigned long long), s))) break;
        if ((rc = normals_device(ix, k, radius, normals_out(ix, viewpoint, store != 0, d_normal, d_var, d_est), &marks, s)) !=
            PT_OK)
            break;
        if (normal_out && fail(cudaMemcpyAsync(normal_out, d_normal, sizeof(float) * 3 * n, cudaMemcpyDeviceToHost, s))) break;
        if (variation_out && fail(cudaMemcpyAsync(variation_out, d_var, sizeof(float) * n, cudaMemcpyDeviceToHost, s))) break;
        if (fail(cudaMemcpyAsync(&est, d_est, sizeof est, cudaMemcpyDeviceToHost, s))) break;
        if (fail(cudaStreamSynchronize(s))) break;
        if (stats) {
            stats->estimated = est;
            // marks: start, then per chunk (after the query, after the PCA kernel)
            float t = 0.0f;
            for (size_t c = 1; c + 1 < marks.size(); c += 2) {
                if (cudaEventElapsedTime(&t, marks[c - 1], marks[c]) == cudaSuccess) stats->knn_ms += t;
                if (cudaEventElapsedTime(&t, marks[c], marks[c + 1]) == cudaSuccess) stats->pca_ms += t;
            }
        }
    } while (0);
    cudaStreamSynchronize(s);
    pool_free(d_normal, s);
    pool_free(d_var, s);
    pool_free(d_est, s);
    for (auto &e : marks) if (e) cudaEventDestroy(e);
    cudaStreamSynchronize(s);
    cudaGetLastError();
    return rc;
}

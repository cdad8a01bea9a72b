// pt_sharded.cu -- a cloud sharded over several GPUs of one box behind the C ABI, host side in
// C++ (north_star: "host code stays C++"; "each GPU indexes a spatial slab of the cloud plus a
// halo sized to the search radius; queries are ... routed by slab").  One process, one host
// thread per slab; built only on the single-index entry points of this library:
//
//   build   : x-cuts at point-count quantiles -> per slab its own points plus the GHOST ZONE
//             (the other slabs' points within `halo` of the slab's box), global ids ascending,
//             one pt_index per slab on its device (pt_index_build)
//   transfer: samples routed to the slab whose x-range holds them; every slab answers its
//             samples with pt_transfer_slab -- k-NN + blend + the ghost-zone check fused per
//             pipeline chunk -- and the results land in the caller's arrays in sample order.
//             A step is final iff no sample's k-th-neighbour ball can leave its slab's ghost
//             zone towards another slab (exactness argument: DESIGN.md section 6).  If some
//             slab reports needs_exchange the halo is widened (widen_and_rebuild), the slabs are
//             rebuilt and the call is repeated, so the result is always exact; `rebuilds` counts that.
//   bake    : the per-texel bake of pt_texture_bake_height on the sharded cloud (DESIGN.md section
//             8, "Sharded bake"): raster, frames, composition and padding on slab 0's device (the
//             home device, pt_bake.cuh pieces); the samples are partitioned by slab there, each
//             slab answers its rows on its own device (k-NN + blend + ghost check + heights from
//             its own records) and the results are scattered back into sample order.
//   normals : pt_index_estimate_normals on the sharded cloud (DESIGN.md section 8, "Sharded normal
//             estimation"): every slab estimates the points it owns on its own device, from its
//             own records with the ghost-zone check on those rows, and the host scatters the
//             results into the caller's point order.  A store reaches every copy of a point (the
//             live slab indexes, and the records of every later rebuild).
//   orient  : pt_index_orient_normals on the sharded cloud (DESIGN.md section 8, "Sharded normal
//             orientation"): every slab builds the edges of the points it owns and the minimum
//             spanning forest of its intra-slab edges on its own device; the home device joins
//             those forests and the cross-slab edges into the global forest and orients from it.
//
// The reference has no multi-GPU path (its query loop is src/pointsTransfer.cpp:465-479); the
// torch.distributed / NCCL form of the same sharding (one process per GPU, unsorted samples
// routed over all_to_all) is sharded.py.  Devices may repeat in the device list: several slabs
// then share one GPU, which is how the single-GPU test box exercises this file.
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstring>
#include <functional>
#include <new>
#include <thread>
#include <vector>

#include "points_transfer.h"
#include "pt_bake.cuh"

namespace {

struct Rec80 {
    double ver[3];
    double normal[3];
    int    color[3];
    int    pad;
    double U, V;
};
static_assert(sizeof(Rec80) == PT_POINT_STRIDE, "Point must be 80 bytes");

struct Slab {
    pt_index *index = nullptr;
    int device = 0;
    size_t n_own = 0, n_ghost = 0;
    double box[6] = {INFINITY, INFINITY, INFINITY, -INFINITY, -INFINITY, -INFINITY};   // own points
    std::vector<int32_t> ids;         // the global id of every record, in the index's local order
    std::vector<uint8_t> own;         // 1 where that record is one of the slab's own points
};

}  // namespace

struct pt_sharded {
    std::vector<Slab> slabs;
    std::vector<double> cuts;         // n_slabs + 1, first -inf, last +inf
    std::vector<double> boxes;        // n_slabs x 6, the slabs' OWN boxes
    const Rec80 *points = nullptr;    // the caller's cloud (must outlive the handle)
    size_t n = 0;
    double halo = 0.0;
    double halo_auto = 0.0;           // the bounding-box estimate (4x the expected k-th neighbour distance)
    int coord_mode = PT_COORD_AUTO;
    int rebuilds = 0;
    // the normals pt_sharded_estimate_normals / pt_sharded_orient_normals stored, n x 3 in point
    // order (x NaN: none, the point keeps its input normal); empty until the first store.
    // build_slabs puts them in the records.
    std::vector<float> stored;
};

namespace {

void free_slabs(pt_sharded *S)
{
    for (auto &s : S->slabs) {
        if (s.index) pt_index_free(s.index);
        s.index = nullptr;
        std::vector<int32_t>().swap(s.ids);
        std::vector<uint8_t>().swap(s.own);
    }
}

// The normal point i's records hold where it is stored, else null: its input normal
const float *stored_normal(const pt_sharded *S, size_t i)
{
    const float *m = S->stored.empty() ? nullptr : &S->stored[3 * i];
    return m && m[0] == m[0] ? m : nullptr;
}

// (re)builds every slab index for the current halo
int build_slabs(pt_sharded *S)
{
    const int R = (int)S->slabs.size();
    free_slabs(S);
    const Rec80 *P = S->points;
    const size_t n = S->n;
    // owner of every point, own boxes
    std::vector<int> owner(n);
    for (auto &s : S->slabs) {
        s.n_own = s.n_ghost = 0;
        for (int a = 0; a < 3; ++a) { s.box[a] = INFINITY; s.box[3 + a] = -INFINITY; }
    }
    for (size_t i = 0; i < n; ++i) {
        const double x = P[i].ver[0];
        const int r = (int)(std::upper_bound(S->cuts.begin() + 1, S->cuts.end() - 1, x) - (S->cuts.begin() + 1));
        owner[i] = r;
        Slab &s = S->slabs[r];
        ++s.n_own;
        for (int a = 0; a < 3; ++a) {
            s.box[a] = std::min(s.box[a], P[i].ver[a]);
            s.box[3 + a] = std::max(s.box[3 + a], P[i].ver[a]);
        }
    }
    // A slab below the last that owns no point gets an empty x-range, so every path (the host
    // routing of sharded_query, bake_partition, the own rows of the normals) sends what falls in
    // its range to the next slab that owns points.  Its index has no records, and the ghost check
    // of an empty box would flag every attempt.  No point changes owner (no point lies in that
    // range), and once applied the rule changes nothing on later builds.  Every cut is some point's
    // x, so the last slab owns a point unless the cloud is empty.
    for (int r = 0; r + 1 < R; ++r)
        if (S->slabs[r].n_own == 0) S->cuts[r + 1] = S->cuts[r];
    S->boxes.assign((size_t)R * 6, 0.0);
    for (int r = 0; r < R; ++r) memcpy(&S->boxes[(size_t)r * 6], S->slabs[r].box, sizeof(double) * 6);
    std::vector<int> status(R, PT_OK);
    std::vector<std::thread> th;
    const double h2 = S->halo * S->halo * (1.0 + 1e-9);
    auto work = [&](int r) {
          try {
            Slab &s = S->slabs[r];
            std::vector<Rec80> rec;
            std::vector<int32_t> ids;
            std::vector<uint8_t> own;
            rec.reserve(s.n_own + s.n_own / 16 + 1024);
            ids.reserve(s.n_own + s.n_own / 16 + 1024);
            own.reserve(s.n_own + s.n_own / 16 + 1024);
            const double *b = s.box;
            for (size_t i = 0; i < n; ++i) {          // index order: global ids ascending
                bool take = owner[i] == r;
                if (!take && s.n_own) {
                    const double ex = std::max(std::max(b[0] - P[i].ver[0], P[i].ver[0] - b[3]), 0.0);
                    const double ey = std::max(std::max(b[1] - P[i].ver[1], P[i].ver[1] - b[4]), 0.0);
                    const double ez = std::max(std::max(b[2] - P[i].ver[2], P[i].ver[2] - b[5]), 0.0);
                    take = ex * ex + ey * ey + ez * ez <= h2;
                }
                if (take) {
                    rec.push_back(P[i]);
                    ids.push_back((int32_t)i);
                    own.push_back(owner[i] == r ? 1 : 0);
                    // a stored normal, widened: the build narrows it back to the same float
                    const float *m = stored_normal(S, i);
                    if (m)
                        for (int a = 0; a < 3; ++a) rec.back().normal[a] = (double)m[a];
                }
            }
            s.n_ghost = rec.size() - s.n_own;
            pt_build_opts o;
            memset(&o, 0, sizeof o);
            o.device = s.device;
            o.coord_mode = S->coord_mode;
            o.ids = ids.data();
            status[r] = pt_index_build(rec.data(), rec.size(), &o, &s.index);
            s.ids = std::move(ids);
            s.own = std::move(own);
          } catch (...) { status[r] = PT_ERR_OUT_OF_MEMORY; }     // nothing is thrown across the ABI
    };
    for (int r = 0; r < R; ++r) {
        try { th.emplace_back(work, r); } catch (...) { work(r); }      // no thread to be had: inline
    }
    for (auto &t : th) t.join();
    for (int r = 0; r < R; ++r)
        if (status[r] != PT_OK) { free_slabs(S); return status[r]; }
    return PT_OK;
}

constexpr int ATTEMPTS = 8;           // answers per call: the first, then one per widening

// A slab whose index holds the whole cloud answers every sample exactly: its ghost check is moot.
bool holds_cloud(const pt_sharded *S, const Slab &s) { return s.n_own + s.n_ghost == S->n; }

// After attempt `attempt` found some ghost zone too narrow: widen the halo and rebuild the slabs.
// x4, at least the bounding-box estimate, at most the diagonal of the cloud's bounding box (the
// union of the own boxes), and that diagonal for the last attempt.  At the diagonal every slab that
// owns a point holds the whole cloud (holds_cloud) and the others receive nothing (build_slabs), so
// the last attempt is final whatever the cloud's units and however far the samples lie.
int widen_and_rebuild(pt_sharded *S, int attempt)
{
    double lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
    for (const Slab &s : S->slabs)
        for (int a = 0; a < 3; ++a) { lo[a] = std::min(lo[a], s.box[a]); hi[a] = std::max(hi[a], s.box[3 + a]); }
    double diag2 = 0.0;
    for (int a = 0; a < 3; ++a) {
        const double e = std::max(hi[a] - lo[a], 0.0);
        diag2 += e * e;
    }
    const double diag = std::sqrt(diag2);
    S->halo = attempt + 2 >= ATTEMPTS ? diag : std::min(std::max(4.0 * S->halo, S->halo_auto), diag);
    ++S->rebuilds;
    return build_slabs(S);
}

int sharded_query(pt_sharded *S, const void *queries, size_t m, int k, double radius, int32_t *idx_out,
                  double *d2_out, uint8_t *rgba_out, float *normal_out)
{
    if (!S || (!queries && m)) return PT_ERR_INVALID_ARG;
    if (k < 1 || k > PT_MAX_K) return PT_ERR_UNSUPPORTED;
    if (m == 0) return PT_OK;
    const int R = (int)S->slabs.size();
    const Rec80 *Q = (const Rec80 *)queries;
    // route: the slab whose x-range holds the sample
    std::vector<std::vector<uint32_t>> mine(R);
    for (size_t i = 0; i < m; ++i) {
        const double x = Q[i].ver[0];
        const int r = (int)(std::upper_bound(S->cuts.begin() + 1, S->cuts.end() - 1, x) - (S->cuts.begin() + 1));
        mine[r].push_back((uint32_t)i);
    }
    for (int attempt = 0; attempt < ATTEMPTS; ++attempt) {
        std::vector<int> status(R, PT_OK), needs(R, 0);
        std::vector<std::thread> th;
        auto work = [&](int r) {
              try {
                const std::vector<uint32_t> &sel = mine[r];
                const size_t mr = sel.size();
                if (mr == 0) return;
                std::vector<Rec80> q(mr);
                for (size_t j = 0; j < mr; ++j) q[j] = Q[sel[j]];
                std::vector<int32_t> idx(idx_out ? mr * k : 0);
                std::vector<double> d2(d2_out ? mr * k : 0);
                std::vector<uint8_t> rgba(rgba_out ? mr * 4 : 0);
                std::vector<float> nrm(normal_out ? mr * 3 : 0);
                int need = 0;
                int rc;
                if (S->slabs[r].index == nullptr) { status[r] = PT_ERR_INVALID_ARG; return; }
                if (rgba_out || normal_out)
                    rc = pt_transfer_slab(S->slabs[r].index, q.data(), 0, mr, k, radius, S->boxes.data(), R, r, S->halo,
                                          idx_out ? idx.data() : nullptr, d2_out ? d2.data() : nullptr,
                                          rgba_out ? rgba.data() : nullptr, normal_out ? nrm.data() : nullptr, &need);
                else {       // k-NN only: the slab entry needs a blend output to run; use a scratch one
                    rgba.resize(mr * 4);
                    rc = pt_transfer_slab(S->slabs[r].index, q.data(), 0, mr, k, radius, S->boxes.data(), R, r, S->halo,
                                          idx_out ? idx.data() : nullptr, d2_out ? d2.data() : nullptr, rgba.data(),
                                          nullptr, &need);
                }
                status[r] = rc;
                needs[r] = holds_cloud(S, S->slabs[r]) ? 0 : need;
                if (rc != PT_OK || needs[r]) return;
                for (size_t j = 0; j < mr; ++j) {          // results back into sample order
                    const size_t d = sel[j];
                    if (idx_out) memcpy(idx_out + d * k, idx.data() + j * k, sizeof(int32_t) * k);
                    if (d2_out) memcpy(d2_out + d * k, d2.data() + j * k, sizeof(double) * k);
                    if (rgba_out) memcpy(rgba_out + d * 4, rgba.data() + j * 4, 4);
                    if (normal_out) memcpy(normal_out + d * 3, nrm.data() + j * 3, sizeof(float) * 3);
                }
              } catch (...) { status[r] = PT_ERR_OUT_OF_MEMORY; }
        };
        for (int r = 0; r < R; ++r) {
            try { th.emplace_back(work, r); } catch (...) { work(r); }
        }
        for (auto &t : th) t.join();
        bool again = false;
        for (int r = 0; r < R; ++r) {
            if (status[r] != PT_OK) return status[r];
            again |= needs[r] != 0;
        }
        if (!again) return PT_OK;
        if (attempt + 1 == ATTEMPTS) break;
        // some k-th-neighbour ball may leave a ghost zone: widen it and answer the call again
        const int rc = widen_and_rebuild(S, attempt);
        if (rc != PT_OK) return rc;
    }
    return PT_ERR_UNSUPPORTED;        // a guard: the last attempt is final for finite input
}

// Sample rows in slab order on the home device (struct of arrays, so a slab's rows are one range
// of each), or one slab's rows on its own device.
struct BakeRows {
    double *xyz = nullptr;
    uint32_t *texel = nullptr;
    int32_t *face = nullptr;      // heights only
    uint8_t *rgba = nullptr;
    float *normal = nullptr;
    float *height = nullptr;      // heights only
    double *mesh = nullptr;       // heights on another device: mesh rows | frames (n_vertices x 8 each)
    int32_t *faces = nullptr;     //   and faces
};

// Buffers that a peer copy reads or writes are cudaMalloc memory (`peer`: dev_alloc), since the
// library's memory pools grant no access to other devices; the others come from the pool on s.
int rows_alloc(BakeRows &B, size_t m, bool heights, size_t mesh_rows, size_t n_faces, bool peer, cudaStream_t s)
{
    auto dev_alloc = [&](void **p, size_t bytes) { return peer ? pt::dev_alloc(p, bytes) : pt::pool_alloc(p, bytes, s); };
    if (dev_alloc((void **)&B.xyz, sizeof(double) * 3 * m) || dev_alloc((void **)&B.texel, sizeof(uint32_t) * m) ||
        dev_alloc((void **)&B.rgba, 4 * m) || dev_alloc((void **)&B.normal, sizeof(float) * 3 * m) ||
        (heights && (dev_alloc((void **)&B.face, sizeof(int32_t) * m) || dev_alloc((void **)&B.height, sizeof(float) * m))) ||
        (mesh_rows && (dev_alloc((void **)&B.mesh, sizeof(double) * 2 * pt::BAKE_ROW * mesh_rows) ||
                       dev_alloc((void **)&B.faces, sizeof(int32_t) * 3 * n_faces))))
        return PT_ERR_OUT_OF_MEMORY;
    return PT_OK;
}

void rows_free(BakeRows &B, bool peer, cudaStream_t s)
{
    void *frees[] = {B.xyz, B.texel, B.face, B.rgba, B.normal, B.height, B.mesh, B.faces};
    for (void *p : frees) {
        if (peer) pt::dev_free(p);
        else pt::pool_free(p, s);
    }
    B = BakeRows{};
}

// One slab's step 3 of the bake, on the slab's own stream and host thread: its rows (home device,
// from row `first`) to its device, k-NN + blend + ghost check + heights there, the per-row results
// back into the home rows.  `copy`: the slab works on copies of its rows (it is on another device,
// or the test option asks for it), else on the home rows in place.  *needs = 1 when the ghost check
// flags the step.
int slab_bake(pt_sharded *S, int r, int home, const pt::BakeJob &J, const BakeRows &rows, size_t first, size_t m,
              bool copy, int k, double radius, int *needs)
{
    using namespace pt;
    const Slab &sl = S->slabs[r];
    pt_index *ix = sl.index;
    if (!ix) return PT_ERR_INVALID_ARG;
    PT_CUDA(cudaSetDevice(sl.device));
    cudaStream_t s = ix->stream;
    const bool heights = J.heights;
    const size_t R = S->slabs.size(), nv = J.n_vertices, nf = J.M.n_faces;
    BakeRows d, mine;
    double *boxes = nullptr;
    uint32_t *flag = nullptr;
    uint32_t h_flag = 0;
    int rc = PT_OK;
    auto fail = [&](cudaError_t e) { if (e != cudaSuccess && rc == PT_OK) rc = map_cuda_error(e); return e != cudaSuccess; };
    auto put = [&](void *dst, int dst_dev, const void *src, int src_dev, size_t bytes) {
        return fail(dst_dev == src_dev ? cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, s)
                                       : cudaMemcpyPeerAsync(dst, dst_dev, src, src_dev, bytes, s));
    };
    do {
        if (pool_alloc((void **)&boxes, sizeof(double) * 6 * R, s) || pool_alloc((void **)&flag, sizeof(uint32_t), s)) {
            rc = PT_ERR_OUT_OF_MEMORY;
            break;
        }
        if (!copy) {
            d.xyz = rows.xyz + 3 * first; d.texel = rows.texel + first; d.rgba = rows.rgba + 4 * first;
            d.normal = rows.normal + 3 * first;
            if (heights) { d.face = rows.face + first; d.height = rows.height + first; }
        } else {
            if ((rc = rows_alloc(mine, m, heights, heights ? nv : 0, nf, true, s)) != PT_OK) break;
            d = mine;
            const int dv = sl.device;
            if (put(d.xyz, dv, rows.xyz + 3 * first, home, sizeof(double) * 3 * m) ||
                put(d.texel, dv, rows.texel + first, home, sizeof(uint32_t) * m))
                break;
            if (heights && (put(d.face, dv, rows.face + first, home, sizeof(int32_t) * m) ||
                            put(d.mesh, dv, rows.mesh, home, sizeof(double) * 2 * BAKE_ROW * nv) ||
                            put(d.faces, dv, rows.faces, home, sizeof(int32_t) * 3 * nf)))
                break;
        }
        if (fail(cudaMemcpyAsync(boxes, S->boxes.data(), sizeof(double) * 6 * R, cudaMemcpyHostToDevice, s)) ||
            fail(cudaMemsetAsync(flag, 0, sizeof(uint32_t), s)))
            break;
        const bool whole = holds_cloud(S, sl);
        const BakeGhost ghost{boxes, (int)R, r, S->halo, flag};
        const BakeMesh M = copy ? BakeMesh{d.mesh, BAKE_ROW, (uint32_t)nv, d.faces, (uint32_t)nf, J.res} : J.M;
        const double *frames = copy ? d.mesh + BAKE_ROW * nv : J.d_frames;
        if ((rc = bake_answer_rows(ix, M, frames, d.xyz, d.texel, d.face, m, k, radius, whole ? nullptr : &ghost, d.rgba,
                                   d.normal, d.height, true, nullptr, s)) != PT_OK)
            break;
        if (copy && (put(rows.rgba + 4 * first, home, d.rgba, sl.device, 4 * m) ||
                     put(rows.normal + 3 * first, home, d.normal, sl.device, sizeof(float) * 3 * m) ||
                     (heights && put(rows.height + first, home, d.height, sl.device, sizeof(float) * m))))
            break;
        if (fail(cudaMemcpyAsync(&h_flag, flag, sizeof h_flag, cudaMemcpyDeviceToHost, s))) break;
        if (fail(cudaStreamSynchronize(s))) break;
        *needs = whole ? 0 : (h_flag ? 1 : 0);
    } while (0);
    cudaStreamSynchronize(s);
    pool_free(boxes, s);
    pool_free(flag, s);
    cudaStreamSynchronize(s);
    rows_free(mine, true, s);
    return rc;
}

// Steps 2-4 of the sharded bake: route the samples, answer them slab by slab until no ghost zone is
// too narrow (widening the halo and rebuilding as sharded_query does), scatter the results into
// J's sample order.  On the home device, current on entry.
int sharded_answer(pt_sharded *S, int home, pt::BakeJob &J, int k, double radius)
{
    using namespace pt;
    const int R = (int)S->slabs.size();
    const size_t count = J.count, nv = J.n_vertices, nf = J.M.n_faces;
    cudaStream_t s = J.s;
    std::vector<char> copy(R, 0);
    bool any_copy = false;
    for (int r = 0; r < R; ++r) {
        copy[r] = S->slabs[r].device != home || opt_sharded_copy();
        any_copy |= copy[r] != 0;
    }
    BakeRows rows;
    int32_t *sel = nullptr;
    std::vector<size_t> starts(R + 1, 0);
    int rc = PT_OK;
    auto fail = [&](cudaError_t e) { if (e != cudaSuccess && rc == PT_OK) rc = map_cuda_error(e); return e != cudaSuccess; };
    do {
        const bool mesh = any_copy && J.heights;
        if (pool_alloc((void **)&sel, sizeof(int32_t) * count, s) ||
            (rc = rows_alloc(rows, count, J.heights, mesh ? nv : 0, nf, any_copy, s)) != PT_OK) {
            rc = PT_ERR_OUT_OF_MEMORY;
            break;
        }
        // the height kernel of a slab on another device reads the mesh rows, frames and faces there
        if (mesh && (fail(cudaMemcpyAsync(rows.mesh, J.d_rows, sizeof(double) * BAKE_ROW * nv, cudaMemcpyDeviceToDevice, s)) ||
                     fail(cudaMemcpyAsync(rows.mesh + BAKE_ROW * nv, J.d_frames, sizeof(double) * BAKE_ROW * nv,
                                          cudaMemcpyDeviceToDevice, s)) ||
                     fail(cudaMemcpyAsync(rows.faces, J.d_faces, sizeof(int32_t) * 3 * nf, cudaMemcpyDeviceToDevice, s))))
            break;
        // samples with a NaN component are routed nowhere: their lists are empty (alpha 0, no height)
        if (fail(cudaMemsetAsync(J.d_rgba, 0, 4 * count, s)) || fail(cudaMemsetAsync(J.d_normal, 0, sizeof(float) * 3 * count, s)))
            break;
        if ((rc = bake_partition(J.d_q, J.d_texels, J.heights ? J.d_sface : nullptr, count, S->cuts.data() + 1, R, sel,
                                 rows.xyz, rows.texel, rows.face, starts.data(), s)) != PT_OK)
            break;
        bool done = false;
        for (int attempt = 0; attempt < ATTEMPTS && !done; ++attempt) {
            std::vector<int> status(R, PT_OK), needs(R, 0);
            std::vector<std::thread> th;
            auto work = [&](int r) {
                const size_t m = starts[r + 1] - starts[r];
                if (m == 0) return;
                try {
                    status[r] = slab_bake(S, r, home, J, rows, starts[r], m, copy[r] != 0, k, radius, &needs[r]);
                } catch (...) { status[r] = PT_ERR_OUT_OF_MEMORY; }
            };
            for (int r = 0; r < R; ++r) {
                try { th.emplace_back(work, r); } catch (...) { work(r); }
            }
            for (auto &t : th) t.join();
            bool again = false;
            for (int r = 0; r < R; ++r) {
                if (status[r] != PT_OK && rc == PT_OK) rc = status[r];
                again |= needs[r] != 0;
            }
            if (rc != PT_OK) break;
            if (!again) { done = true; break; }
            if (attempt + 1 == ATTEMPTS) break;
            // some k-th-neighbour ball may leave a ghost zone: widen it and answer the rows again
            if ((rc = widen_and_rebuild(S, attempt)) != PT_OK) break;
        }
        if (rc != PT_OK) break;
        if (!done) { rc = PT_ERR_UNSUPPORTED; break; }          // a guard, as in sharded_query
        if (fail(cudaSetDevice(home))) break;
        const uint32_t routed = (uint32_t)starts[R];
        if ((rc = launch_scatter_rows(rows.rgba, sel, routed, 4, J.d_rgba, s)) != PT_OK ||
            (rc = launch_scatter_rows(rows.normal, sel, routed, 12, J.d_normal, s)) != PT_OK)
            break;
        // a row's height goes straight to its texel of the image
        if (J.heights && (rc = launch_scatter_rows(rows.height, (const int32_t *)rows.texel, routed, 4, J.d_height, s)) != PT_OK)
            break;
        fail(cudaStreamSynchronize(s));
    } while (0);
    cudaSetDevice(home);
    cudaStreamSynchronize(s);
    pool_free(sel, s);
    cudaStreamSynchronize(s);
    rows_free(rows, any_copy, s);
    return rc;
}

int sharded_bake(pt_sharded *S, const void *vertices, size_t n_vertices, const int32_t *faces, size_t n_faces, int k,
                 double radius, int res, int pad, const pt_bake_outputs &o, pt_bake_height *hb, pt_bake_stats *st)
{
    using namespace pt;
    const int home = S->slabs[0].device;
    PT_CUDA(cudaSetDevice(home));
    cudaStream_t s = nullptr;
    PT_CUDA(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
    BakeJob J;
    float knn_ms = 0.0f;
    int rc = bake_prepare(J, s, vertices, n_vertices, faces, n_faces, res, o, hb);
    if (rc == PT_OK && J.count) {
        const auto t0 = std::chrono::steady_clock::now();
        rc = sharded_answer(S, home, J, k, radius);
        knn_ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
    }
    if (rc == PT_OK) rc = bake_finish(J, pad, o, hb, st);
    if (rc == PT_OK && st) st->knn_ms = knn_ms;
    bake_release(J);
    cudaStreamDestroy(s);
    return rc;
}

// f(r) for r = 0 .. R - 1, one host thread each (one per slab): the first error, else PT_OK
int on_threads(int R, const std::function<int(int)> &f)
{
    std::vector<int> status(R, PT_OK);
    std::vector<std::thread> th;
    auto work = [&](int r) {
        try {
            status[r] = f(r);
        } catch (...) { status[r] = PT_ERR_OUT_OF_MEMORY; }
    };
    for (int r = 0; r < R; ++r) {
        try { th.emplace_back(work, r); } catch (...) { work(r); }
    }
    for (auto &t : th) t.join();
    for (int r = 0; r < R; ++r)
        if (status[r] != PT_OK) return status[r];
    return (int)PT_OK;
}

// every copy of every point, own and ghost, takes the stored normals
int store_slabs(pt_sharded *S)
{
    return on_threads((int)S->slabs.size(), [&](int r) {
        const Slab &sl = S->slabs[r];
        if (sl.ids.empty()) return (int)PT_OK;                         // a slab without records
        std::vector<float> values(3 * sl.ids.size());
        for (size_t l = 0; l < sl.ids.size(); ++l)
            memcpy(&values[3 * l], &S->stored[3 * (size_t)sl.ids[l]], sizeof(float) * 3);
        return pt::normals_store(sl.index, values.data());
    });
}

// pt_index_estimate_normals on the sharded cloud; arguments checked, S->n > 0.
int sharded_normals(pt_sharded *S, int k, double radius, const double *viewpoint, bool store, float *normal_out,
                    float *variation_out, pt_normals_stats *stats)
{
    const int R = (int)S->slabs.size();
    const auto t0 = std::chrono::steady_clock::now();
    std::vector<std::vector<float>> nrm(R), var(R);
    std::vector<unsigned long long> est(R, 0);
    std::vector<float> pca(R, 0.0f);
    // every slab estimates its own points; nothing reaches the caller or the slabs before all pass
    int rc = PT_OK;
    bool done = false;
    for (int attempt = 0; attempt < ATTEMPTS && !done; ++attempt) {
        std::vector<int> needs(R, 0);
        rc = on_threads(R, [&](int r) {
            const Slab &sl = S->slabs[r];
            est[r] = 0;
            pca[r] = 0.0f;
            if (!sl.index) return (int)PT_ERR_INVALID_ARG;
            if (sl.n_own == 0) return (int)PT_OK;
            nrm[r].resize(3 * sl.n_own);
            var[r].resize(sl.n_own);
            const pt::NormalsSlab job{S->cuts.data() + 1, R, r, sl.n_own, S->boxes.data(), S->halo, !holds_cloud(S, sl)};
            return pt::normals_slab(sl.index, k, radius, viewpoint, job, nrm[r].data(), var[r].data(), &est[r], &pca[r],
                                    &needs[r]);
        });
        if (rc != PT_OK) return rc;
        done = std::none_of(needs.begin(), needs.end(), [](int v) { return v != 0; });
        if (done || attempt + 1 == ATTEMPTS) break;
        // some k-th-neighbour ball may leave a ghost zone: widen it and estimate again
        if ((rc = widen_and_rebuild(S, attempt)) != PT_OK) return rc;
    }
    if (!done) return PT_ERR_UNSUPPORTED;                     // a guard, as in sharded_query
    // the own entries into the caller's point order (slabs own disjoint points)
    if (store && S->stored.empty()) S->stored.assign(3 * S->n, NAN);
    // each slab's own results come in ascending local id: the i-th goes to the global id of the
    // slab's i-th own record.  Ranges of records over a share of the host's cores.
    const size_t share = std::max(1u, std::thread::hardware_concurrency() / (unsigned)R);
    rc = on_threads(R, [&](int r) {
        const Slab &sl = S->slabs[r];
        if (sl.n_own == 0) return (int)PT_OK;
        const float *nr = nrm[r].data(), *vr = var[r].data();
        const size_t nl = sl.ids.size(), parts = std::min(share, nl / 65536 + 1), step = (nl + parts - 1) / parts;
        std::vector<size_t> first(parts + 1, 0);           // own records before each range
        for (size_t p = 0; p < parts; ++p)
            first[p + 1] = first[p] + (size_t)std::count(sl.own.begin() + std::min(nl, p * step),
                                                         sl.own.begin() + std::min(nl, (p + 1) * step), (uint8_t)1);
        if (first[parts] != sl.n_own) return (int)PT_ERR_UNSUPPORTED;
        auto scatter = [&](size_t p) {
            size_t j = first[p];
            for (size_t l = p * step; l < std::min(nl, (p + 1) * step); ++l) {
                if (!sl.own[l]) continue;                                  // a ghost: its owner writes it
                const size_t g = (size_t)sl.ids[l];
                if (normal_out) memcpy(normal_out + 3 * g, nr + 3 * j, sizeof(float) * 3);
                if (variation_out) variation_out[g] = vr[j];
                if (store && vr[j] == vr[j]) memcpy(&S->stored[3 * g], nr + 3 * j, sizeof(float) * 3);   // estimated
                ++j;
            }
        };
        std::vector<std::thread> th;
        for (size_t p = 1; p < parts; ++p) {
            try { th.emplace_back(scatter, p); } catch (...) { scatter(p); }
        }
        scatter(0);
        for (auto &t : th) t.join();
        return (int)PT_OK;
    });
    if (rc == PT_OK && store) rc = store_slabs(S);
    if (rc != PT_OK) return rc;
    if (stats) {
        stats->knn_ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
        stats->pca_ms = 0.0f;
        stats->estimated = 0;
        for (int r = 0; r < R; ++r) {
            stats->estimated += est[r];
            stats->pca_ms += pca[r];
        }
    }
    return PT_OK;
}

// pt_index_orient_normals on the sharded cloud (DESIGN.md section 8, "Sharded normal orientation");
// arguments checked, S->n > 0.
int sharded_orient(pt_sharded *S, int k, double radius, const double *viewpoint, bool store, float *normal_out,
                   int32_t *root_out, pt_orient_stats *stats)
{
    const int R = (int)S->slabs.size();
    const size_t n = S->n;
    const auto t0 = std::chrono::steady_clock::now();
    std::vector<std::vector<pt::OrientEdge>> forest(R), cross(R);
    std::vector<uint64_t> intra(R, 0);
    // every slab: its own rows' lists, edges and intra-slab forest; nothing reaches the caller or the
    // slabs before all pass their ghost checks
    int rc = PT_OK;
    bool done = false;
    for (int attempt = 0; attempt < ATTEMPTS && !done; ++attempt) {
        std::vector<int> needs(R, 0);
        rc = on_threads(R, [&](int r) {
            const Slab &sl = S->slabs[r];
            forest[r].clear();
            cross[r].clear();
            intra[r] = 0;
            if (!sl.index) return (int)PT_ERR_INVALID_ARG;
            if (sl.n_own == 0) return (int)PT_OK;
            const pt::NormalsSlab job{S->cuts.data() + 1, R, r, sl.n_own, S->boxes.data(), S->halo, !holds_cloud(S, sl)};
            return pt::orient_slab(sl.index, k, radius, job, forest[r], cross[r], &intra[r], &needs[r]);
        });
        if (rc != PT_OK) return rc;
        done = std::none_of(needs.begin(), needs.end(), [](int v) { return v != 0; });
        if (done || attempt + 1 == ATTEMPTS) break;
        // some k-th-neighbour ball may leave a ghost zone: widen it and run the stage again
        if ((rc = widen_and_rebuild(S, attempt)) != PT_OK) return rc;
    }
    if (!done) return PT_ERR_UNSUPPORTED;                     // a guard, as in sharded_query
    const auto t1 = std::chrono::steady_clock::now();
    // the home device's inputs in point order: the normals the records were built from (the device
    // narrows them as the build does), and the caller's z (with a viewpoint, the whole position)
    const int home = S->slabs[0].device;
    const size_t dims = viewpoint ? 3 : 1;
    std::vector<double> normal(3 * n);
    std::vector<float> nrm_tmp(normal_out ? 0 : 3 * n);
    std::vector<double> pos(dims * n);
    std::vector<int32_t> root_tmp(root_out ? 0 : n);
    float *nrm = normal_out ? normal_out : nrm_tmp.data();
    int32_t *root = root_out ? root_out : root_tmp.data();
    const Rec80 *P = S->points;
    const size_t parts = std::max(1u, std::thread::hardware_concurrency()), step = (n + parts - 1) / parts;
    on_threads((int)parts, [&](int p) {
        for (size_t i = p * step; i < std::min(n, (p + 1) * step); ++i) {
            const float *m = stored_normal(S, i);
            for (int a = 0; a < 3; ++a) normal[3 * i + a] = m ? (double)m[a] : P[i].normal[a];
            for (size_t a = 0; a < dims; ++a) pos[dims * i + a] = P[i].ver[3 - dims + a];
        }
        return (int)PT_OK;
    });
    unsigned long long counts[3] = {0, 0, 0};
    uint64_t unique_cross = 0;
    {
        PT_CUDA(cudaSetDevice(home));
        cudaStream_t s = nullptr;
        PT_CUDA(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
        const pt::OrientHome h{n, normal.data(), pos.data(), viewpoint, nrm, root};
        rc = pt::orient_home(h, forest, cross, &unique_cross, counts, s);
        cudaStreamDestroy(s);
        if (rc != PT_OK) return rc;
    }
    // the oriented normals of the points that take part (root >= 0) into every copy of them
    if (store) {
        if (S->stored.empty()) S->stored.assign(3 * n, NAN);
        for (size_t i = 0; i < n; ++i)
            if (root[i] >= 0) memcpy(&S->stored[3 * i], nrm + 3 * i, sizeof(float) * 3);
        if ((rc = store_slabs(S)) != PT_OK) return rc;
    }
    if (stats) {
        stats->oriented = counts[0];
        stats->flipped = counts[1];
        stats->components = counts[2];
        stats->edges = unique_cross;
        for (int r = 0; r < R; ++r) stats->edges += intra[r];
        stats->knn_ms = std::chrono::duration<float, std::milli>(t1 - t0).count();
        stats->mst_ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t1).count();
    }
    return PT_OK;
}

}  // namespace

extern "C" {

int pt_sharded_build(const void *points, size_t n, const pt_sharded_opts *opts, pt_sharded **out)
{
    if (!out || !opts || (!points && n) || n >= 0x7fffffffull || opts->n_devices < 1 || opts->n_devices > 64)
        return PT_ERR_INVALID_ARG;
    *out = nullptr;
    const int avail = pt_device_count();
    if (avail == 0) return PT_ERR_NO_DEVICE;
    pt_sharded *S = new (std::nothrow) pt_sharded();
    if (!S) return PT_ERR_OUT_OF_MEMORY;
    try {
    const int R = opts->n_devices;
    S->slabs.resize(R);
    for (int r = 0; r < R; ++r) {
        S->slabs[r].device = opts->devices ? opts->devices[r] : r % avail;
        if (S->slabs[r].device < 0 || S->slabs[r].device >= avail) { delete S; return PT_ERR_INVALID_ARG; }
    }
    S->points = (const Rec80 *)points;
    S->n = n;
    S->coord_mode = opts->coord_mode;
    // x-cuts at point-count quantiles (of a sample of the cloud: the cuts need not be exact)
    {
        const size_t step = n > 4000000 ? n / 4000000 : 1;
        std::vector<double> xs;
        xs.reserve(n / step + 1);
        for (size_t i = 0; i < n; i += step) xs.push_back(S->points[i].ver[0]);
        S->cuts.assign(R + 1, 0.0);
        S->cuts[0] = -INFINITY;
        S->cuts[R] = INFINITY;
        for (int r = 1; r < R; ++r) {
            const size_t pos = xs.empty() ? 0 : std::min(xs.size() - 1, xs.size() * (size_t)r / R);
            if (!xs.empty()) std::nth_element(xs.begin(), xs.begin() + pos, xs.end());
            S->cuts[r] = xs.empty() ? 0.0 : xs[pos];
        }
        std::sort(S->cuts.begin() + 1, S->cuts.end() - 1);
    }
    // ghost-zone width: given, or a multiple of the expected k-th-neighbour distance estimated
    // from the bounding box (line, surface and volume estimate, the largest one); a call that finds
    // it too small widens it (widen_and_rebuild)
    S->halo = opts->halo;
    {
        double lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
        for (size_t i = 0; i < n; i += (n > 1000000 ? n / 1000000 : 1))
            for (int a = 0; a < 3; ++a) { lo[a] = std::min(lo[a], S->points[i].ver[a]); hi[a] = std::max(hi[a], S->points[i].ver[a]); }
        double e[3] = {std::max(hi[0] - lo[0], 0.0), std::max(hi[1] - lo[1], 0.0), std::max(hi[2] - lo[2], 0.0)};
        std::sort(e, e + 3);
        const double kk = opts->k_hint > 0 ? opts->k_hint : 20;
        const double nn = n ? (double)n : 1.0;
        const double r_surface = std::sqrt(kk * e[1] * e[2] / (M_PI * nn));
        const double r_volume = std::cbrt(3.0 * kk * e[0] * e[1] * e[2] / (4.0 * M_PI * nn));
        const double r_line = kk * e[2] / nn;
        // no wider than the box's diagonal, beyond which a ghost zone takes no more points
        const double diag = std::sqrt(e[0] * e[0] + e[1] * e[1] + e[2] * e[2]);
        S->halo_auto = std::min(4.0 * std::max(std::max(r_surface, r_volume), r_line), diag);
        if (!std::isfinite(S->halo_auto)) S->halo_auto = 0.0;
        if (!(S->halo > 0.0)) S->halo = S->halo_auto;
    }
    const int rc = build_slabs(S);
    if (rc != PT_OK) { delete S; return rc; }
    *out = S;
    return PT_OK;
    } catch (...) {                 // host allocation failure: nothing is thrown across the ABI
        free_slabs(S);
        delete S;
        return PT_ERR_OUT_OF_MEMORY;
    }
}

int pt_sharded_free(pt_sharded *S)
{
    if (!S) return PT_OK;
    free_slabs(S);
    delete S;
    return PT_OK;
}

int pt_sharded_knn(pt_sharded *S, const void *queries, size_t m, int k, double radius, int32_t *idx_out,
                   double *d2_out)
{
    if (!idx_out && m) return PT_ERR_INVALID_ARG;
    try {
        return sharded_query(S, queries, m, k, radius, idx_out, d2_out, nullptr, nullptr);
    } catch (...) { return PT_ERR_OUT_OF_MEMORY; }
}

int pt_sharded_transfer(pt_sharded *S, const void *queries, size_t m, int k, double radius, int32_t *idx_out,
                        double *d2_out, uint8_t *rgba_out, float *normal_out)
{
    if ((!rgba_out && !normal_out) && m) return PT_ERR_INVALID_ARG;
    try {
        return sharded_query(S, queries, m, k, radius, idx_out, d2_out, rgba_out, normal_out);
    } catch (...) { return PT_ERR_OUT_OF_MEMORY; }
}

int pt_sharded_bake(pt_sharded *S, const void *vertices, size_t n_vertices, const int32_t *faces, size_t n_faces,
                    int k, double radius, int resolution, int pad, const pt_bake_outputs *out, pt_bake_height *height,
                    pt_bake_stats *stats)
{
    const pt_bake_outputs none = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    const pt_bake_outputs &o = out ? *out : none;
    if (!S) return PT_ERR_INVALID_ARG;
    const int rc = pt::bake_check_args(vertices, n_vertices, faces, n_faces, k, resolution, o, height);
    if (rc != PT_OK) return rc;
    if (pt_device_count() == 0) return PT_ERR_NO_DEVICE;
    try {
        return sharded_bake(S, vertices, n_vertices, faces, n_faces, k, radius, resolution, pad, o, height, stats);
    } catch (...) { return PT_ERR_OUT_OF_MEMORY; }
}

int pt_sharded_estimate_normals(pt_sharded *S, int k, double radius, const double *viewpoint, int store,
                                float *normal_out, float *variation_out, pt_normals_stats *stats)
{
    if (!S) return PT_ERR_INVALID_ARG;
    const int rc = pt::normals_check_args(k, viewpoint, store != 0, normal_out || variation_out);
    if (rc != PT_OK) return rc;
    if (pt_device_count() == 0) return PT_ERR_NO_DEVICE;
    if (stats) *stats = pt_normals_stats{0, 0.0f, 0.0f};
    if (S->n == 0) return PT_OK;
    try {
        return sharded_normals(S, k, radius, viewpoint, store != 0, normal_out, variation_out, stats);
    } catch (...) { return PT_ERR_OUT_OF_MEMORY; }
}

int pt_sharded_orient_normals(pt_sharded *S, int k, double radius, const double *viewpoint, int store,
                              float *normal_out, int32_t *root_out, pt_orient_stats *stats)
{
    if (!S) return PT_ERR_INVALID_ARG;
    const int rc = pt::orient_check_args(k, viewpoint, store != 0, normal_out || root_out);
    if (rc != PT_OK) return rc;
    if (pt_device_count() == 0) return PT_ERR_NO_DEVICE;
    if (stats) *stats = pt_orient_stats{0, 0, 0, 0, 0.0f, 0.0f};
    if (S->n == 0) return PT_OK;
    try {
        return sharded_orient(S, k, radius, viewpoint, store != 0, normal_out, root_out, stats);
    } catch (...) { return PT_ERR_OUT_OF_MEMORY; }
}

int pt_sharded_get_info(const pt_sharded *S, pt_sharded_info *info)
{
    if (!S || !info) return PT_ERR_INVALID_ARG;
    memset(info, 0, sizeof *info);
    info->n_slabs = (int)S->slabs.size();
    info->halo = S->halo;
    info->rebuilds = S->rebuilds;
    info->n_points = S->n;
    for (size_t r = 0; r < S->slabs.size() && r < 64; ++r) {
        info->slab_points[r] = S->slabs[r].n_own;
        info->slab_ghosts[r] = S->slabs[r].n_ghost;
        info->slab_device[r] = S->slabs[r].device;
    }
    return PT_OK;
}

}  // extern "C"

// pt_common.cuh -- shared device/host definitions of the pointsTransfer hot path (sm_100a).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <atomic>

#include "points_transfer.h"

namespace pt {

// ---- error plumbing (nothing may throw across the C ABI) ------------------------------
extern std::atomic<uint64_t> g_launches;
inline void count_launch(uint64_t n = 1) { g_launches.fetch_add(n, std::memory_order_relaxed); }

int map_cuda_error(cudaError_t e);
#define PT_CUDA(call)                                                              \
    do {                                                                           \
        cudaError_t e__ = (call);                                                  \
        if (e__ != cudaSuccess) {                                                  \
            if (::pt::verbose())                                                   \
                fprintf(stderr, "[points_transfer] %s:%d %s -> %s\n", __FILE__,    \
                        __LINE__, #call, cudaGetErrorString(e__));                 \
            return ::pt::map_cuda_error(e__);                                      \
        }                                                                          \
    } while (0)
#define PT_TRY(call)                   \
    do {                               \
        int s__ = (call);              \
        if (s__ != PT_OK) return s__;  \
    } while (0)
bool verbose();

// ---- data layout in HBM -----------------------------------------------------------------
// The cloud is stored Morton-sorted in 32-point leaves ("buckets"); one leaf is one
// contiguous, 16-byte aligned run: 512 B (F32) or 1 KiB (F64).
constexpr int LEAF = 32;

struct PointF {          // 16 B: float4 with the local point index in .w's bits
    float x, y, z;
    int   idx;
};
struct __align__(16) PointD {  // 32 B
    double x, y, z;
    int    idx;
    int    pad;
};

// Axis-aligned box of a pyramid node, float, rounded outward for F64 clouds.  32 B so a
// lane / thread fetches it with two 16-byte loads.
struct __align__(16) Box {
    float lox, loy, loz, hix;
    float hiy, hiz, pad0, pad1;
};

constexpr int MAX_PYR_LEVELS = 32;  // binary pyramid: level j covers 2^j leaves
constexpr int WLOG = 5;             // the warp traversal is 32-wide: uses levels 0,5,10,...
constexpr int MAX_W_LEVELS = 6;     // 32^6 leaves

struct Pyramid {
    const Box *level[MAX_PYR_LEVELS];
    uint32_t   count[MAX_PYR_LEVELS];
    int        n_levels;
};

// ---- uniform grid over the curve-sorted cloud (pt_grid.cu) ----------------------------------
// A cell of level l is the set of points whose 21-bit lattice coordinates share their top l bits
// per axis: one contiguous run of the sorted cloud (Morton and Hilbert keys are both
// hierarchical).  A table holds one 32-byte bucket per occupied PARENT cell (level l - 1), found
// by hashing the parent's lattice coordinates; the bucket locates the runs of its 8 children.
struct __align__(16) GridBucket {
    unsigned long long key;    // parent coordinates x | y << 21 | z << 42; ~0 = empty slot
    uint32_t           start;  // first point of the parent's run
    uint32_t           perm;   // bits 3o..3o+2: curve rank of child octant o (x&1 | y&1 << 1 | z&1 << 2);
                               // bits 24+o: octant o holds points
    uint16_t           cum[8]; // cum[0] = points of the parent (0xffff: too many, bucket unusable);
                               // cum[r], r >= 1 = points in the children of rank < r
};
static_assert(sizeof(GridBucket) == 32, "one sector per bucket");

// Slot of the block-run table (pt_knn_span.cuh, build_blocks): one per occupied cell of the level
// the runs are built for, found by hashing the cell's lattice coordinates; four slots = one
// aligned 64-byte group.
struct __align__(16) BlockSlot {
    unsigned long long key;    // cell coordinates x | y << 21 | z << 42; ~0 = empty slot
    uint32_t           off;    // first 16-byte unit of the run
    uint32_t           meta;   // records | heads << 16; BLOCK_MISS: the block cannot be staged
};
static_assert(sizeof(BlockSlot) == 16, "four slots per 64-byte group");
constexpr uint32_t BLOCK_MISS = 0x80000000u;

constexpr int GRID_MAX_TABLES = 4;
constexpr int GRID_MAX_ATTEMPTS = 4;
struct GridTable {
    const GridBucket *buckets;
    uint32_t          cap;     // slots (even; linear probing in 2-slot groups, load <= 1/3)
    int               level;   // level of the CHILD cells the table resolves
};
struct GridParams {
    GridTable tab[GRID_MAX_TABLES];   // finest first
    int       n_tables;
    double    lo[3];           // lattice origin (bbox minimum)
    double    inv_cell21;      // 2^21 / extent
    double    cell21;          // extent / 2^21
    double    slack;           // absolute safety margin of the cell-boundary distances
    // search schedule of one launch: attempt a looks at the (2 rc + 1)^3 block of level
    // tab[att_tab[a]].level around the sample; the next attempt runs only if the k-th candidate
    // is not provably final
    int       n_attempts;
    unsigned char att_tab[GRID_MAX_ATTEMPTS], att_rc[GRID_MAX_ATTEMPTS];
    float     expect_cand;     // candidates the first attempt is expected to stage per sample (host estimate)
    // block runs of the cells of level blk_level (null: none)
    const BlockSlot *blk;
    const uint4     *blk_runs;
    uint32_t         blk_cap;  // slots (a multiple of 4; linear probing in 4-slot groups, load <= 1/3)
    int              blk_level;
};

struct QueryParams {
    const void    *pts;        // PointF* or PointD*, n_pad records
    const pt_attr *attrs;      // original (local) order, may be null
    const pt_attr *attrs_curve; // attrs in the order of pts (attrs_curve[i] = attrs[pts[i].idx]), may be null
    const int32_t *ids;        // local -> global id, may be null
    Pyramid        pyr;
    uint32_t       n;          // points
    uint32_t       n_leaves;
    int            w_levels;   // number of 32-wide levels used by the warp traversal
    int            t_levels;   // number of 8-wide levels used by the thread traversal
    int            pq_cap;     // queue entries a sample may hold (<= the compiled capacity)
    GridParams     grid;       // n_tables == 0: no grid
    const uint32_t *qlist;     // optional: the launch answers samples qlist[0 .. *qcount) only
    const uint32_t *qcount;
    uint32_t        qlist_min; // list mode: do nothing unless *qcount >= qlist_min
    const double  *queries;    // m * 3
    const double  *r2_per_query;
    uint32_t       m;
    int            k;
    double         r2;         // squared radius bound (+inf if unbounded)
    int32_t       *idx_out;
    double        *d2_out;
    uint8_t       *rgba_out;
    float         *normal_out;
    pt_cand       *cand_out;
};

// ---- the metric: src/Distance.h:6-11, fp64, (dx*dx + dy*dy) + dz*dz, never contracted ----
__device__ __forceinline__ double dist2_exact(double qx, double qy, double qz, double px,
                                              double py, double pz)
{
    double dx = __dsub_rn(qx, px);
    double dy = __dsub_rn(qy, py);
    double dz = __dsub_rn(qz, pz);
    return __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
}

// Weight of neighbour j in the blend (DESIGN.md "blend"), shared by the blend and the height bake.
// mode 0: 1/d2; 1 (the nearest is an exact hit): exact hits only; 2 (the mode 0 / 1 sum is not in
// (0, inf)): the nearest only.
__device__ __forceinline__ double blend_weight(int mode, double d2, int j)
{
    if (mode == 0) return __ddiv_rn(1.0, d2);
    if (mode == 1) return d2 == 0.0 ? 1.0 : 0.0;
    return j == 0 ? 1.0 : 0.0;
}

// Ordering key (d2, index): lowest index wins ties.
__device__ __forceinline__ bool key_less(double da, int ia, double db, int ib)
{
    return da < db || (da == db && ia < ib);
}

constexpr int IDX_NONE = 0x7fffffff;  // sentinel index of an empty list slot

// Conservative fp32 lower bound of Distance::min_distance_to_rectangle (src/Distance.h:27-57):
// every operation rounds toward the safe side, so lb <= the real bound <= real d2 of any
// point inside the box.  The query is bracketed by [q_dn, q_up] (fp32 round-down / round-up).
__device__ __forceinline__ float box_lower_bound(const float qdn[3], const float qup[3],
                                                 const Box &b)
{
    float ex = fmaxf(fmaxf(__fsub_rd(b.lox, qup[0]), __fsub_rd(qdn[0], b.hix)), 0.0f);
    float ey = fmaxf(fmaxf(__fsub_rd(b.loy, qup[1]), __fsub_rd(qdn[1], b.hiy)), 0.0f);
    float ez = fmaxf(fmaxf(__fsub_rd(b.loz, qup[2]), __fsub_rd(qdn[2], b.hiz)), 0.0f);
    return __fadd_rd(__fadd_rd(__fmul_rd(ex, ex), __fmul_rd(ey, ey)), __fmul_rd(ez, ez));
}

}  // namespace pt

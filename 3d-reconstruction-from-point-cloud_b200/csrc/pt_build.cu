// pt_build.cu -- spatial index build (replaces the lazy CGAL kd-tree build behind
// `Tree tree(points.begin(), points.end())`, /root/reference src/pointsTransfer.cpp:259).
//
//   K1  bounding box + 63-bit Morton key per point        (bbox_kernel, morton_kernel)
//   K2  radix sort of (key, index) pairs                   (sort_pairs)
//       gather into 32-point leaves (16-byte float4 / 32-byte fp64 records)
//       leaf boxes + binary box pyramid ("cell table")    (leaf_box_kernel, pyramid_kernel)
//
// HBM layout: pts[n_leaves*32] sorted records; boxes[level][node] 32-byte AABBs, level j
// node i covering leaves [i*2^j, (i+1)*2^j).  Attributes and ids stay in original order; float4
// clouds with cell tables also keep a sorted-order copy of the attributes (attrs_curve).
#include <cub/device/device_radix_sort.cuh>

#include <cfloat>
#include <chrono>
#include <cmath>
#include <mutex>
#include <unordered_map>

#include "pt_index.cuh"

namespace pt {

// ---- K1: bounding box -------------------------------------------------------------------
__device__ __forceinline__ unsigned long long enc_f64(double d)
{
    unsigned long long u = (unsigned long long)__double_as_longlong(d);
    return (u >> 63) ? ~u : (u | 0x8000000000000000ull);
}
static inline double dec_f64(unsigned long long u)
{
    u = (u >> 63) ? (u & 0x7fffffffffffffffull) : ~u;
    double d;
    memcpy(&d, &u, sizeof d);
    return d;
}

struct BBoxAcc {                 // device-side accumulator
    unsigned long long lo[3];    // encoded minima
    unsigned long long hi[3];    // encoded maxima
    unsigned int       non_finite;
    unsigned int       pad;
};

template <typename In>
__global__ void __launch_bounds__(256) bbox_kernel(In in, uint32_t n, BBoxAcc *acc)
{
    double lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
    bool bad = false;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        double v[3];
        in.load(i, v[0], v[1], v[2]);
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            bad |= !isfinite(v[a]);
            lo[a] = fmin(lo[a], v[a]);
            hi[a] = fmax(hi[a], v[a]);
        }
    }
#pragma unroll
    for (int a = 0; a < 3; ++a) {
#pragma unroll
        for (int s = 16; s > 0; s >>= 1) {
            lo[a] = fmin(lo[a], __shfl_xor_sync(0xffffffffu, lo[a], s));
            hi[a] = fmax(hi[a], __shfl_xor_sync(0xffffffffu, hi[a], s));
        }
    }
    bad = __any_sync(0xffffffffu, bad);
    if ((threadIdx.x & 31) == 0) {
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            atomicMin(&acc->lo[a], enc_f64(lo[a]));
            atomicMax(&acc->hi[a], enc_f64(hi[a]));
        }
        if (bad) atomicOr(&acc->non_finite, 1u);
    }
}

// ---- K1: Morton keys ----------------------------------------------------------------------
__device__ __forceinline__ unsigned long long spread21(unsigned int v)
{
    unsigned long long x = v & 0x1fffffu;
    x = (x | (x << 32)) & 0x001f00000000ffffull;
    x = (x | (x << 16)) & 0x001f0000ff0000ffull;
    x = (x | (x << 8)) & 0x100f00f00f00f00full;
    x = (x | (x << 4)) & 0x10c30c30c30c30c3ull;
    x = (x | (x << 2)) & 0x1249249249249249ull;
    return x;
}

// 3-D Hilbert index of 21-bit cell coordinates (Skilling's transpose algorithm): consecutive
// keys are always face-adjacent cells, so 32-point runs make tighter leaves than Morton order.
__device__ __forceinline__ unsigned long long hilbert63(unsigned int x, unsigned int y,
                                                        unsigned int z)
{
    unsigned int X[3] = {x, y, z};
    const unsigned int M = 1u << 20;
    for (unsigned int Q = M; Q > 1; Q >>= 1) {
        const unsigned int Pm = Q - 1;
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            if (X[i] & Q) X[0] ^= Pm;
            else { unsigned int t = (X[0] ^ X[i]) & Pm; X[0] ^= t; X[i] ^= t; }
        }
    }
    X[1] ^= X[0];
    X[2] ^= X[1];
    unsigned int t = 0;
    for (unsigned int Q = M; Q > 1; Q >>= 1)
        if (X[2] & Q) t ^= Q - 1;
    X[0] ^= t; X[1] ^= t; X[2] ^= t;
    return (spread21(X[0]) << 2) | (spread21(X[1]) << 1) | spread21(X[2]);
}

struct KeyParams {
    double lo[3];
    double inv_cell;   // 2^21 / max extent (0 when the cloud is a single point)
    int    order;      // 0 = Morton, 1 = Hilbert, 2 = Hilbert + in-block kd refinement
};

template <typename In>
__global__ void __launch_bounds__(256) morton_kernel(In in, uint32_t n, KeyParams kp,
                                                     unsigned long long *keys, uint32_t *vals)
{
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double v[3];
    in.load(i, v[0], v[1], v[2]);
    unsigned int c[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        double t = (v[a] - kp.lo[a]) * kp.inv_cell;
        t = fmin(fmax(t, 0.0), 2097151.0);
        c[a] = (unsigned int)t;
    }
    keys[i] = kp.order >= 1 ? hilbert63(c[0], c[1], c[2])
                            : (spread21(c[0]) | (spread21(c[1]) << 1) | (spread21(c[2]) << 2));
    vals[i] = i;
}

// ---- gather into leaves -----------------------------------------------------------------
template <typename In, typename Out>
__global__ void __launch_bounds__(256) gather_kernel(In in, const uint32_t *perm, uint32_t n,
                                                     uint32_t n_pad, Out *out, const pt_attr *attrs,
                                                     pt_attr *attrs_out)
{
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_pad) return;
    Out o;
    if (i < n) {
        uint32_t src = perm[i];
        if (attrs_out) attrs_out[i] = attrs[src];   // the attributes in the same (sorted) order
        double x, y, z;
        in.load(src, x, y, z);
        o.x = x; o.y = y; o.z = z;   // exact: F32 storage is only chosen when representable
        o.idx = (int)src;
    } else {
        o.x = FLT_MAX; o.y = FLT_MAX; o.z = FLT_MAX;
        o.idx = IDX_NONE;
    }
    if constexpr (sizeof(Out) == 32) o.pad = 0;
    out[i] = o;
}

// ---- kd refinement of the curve order (order = 2) ----------------------------------------------
// A run of consecutive Hilbert keys is a compact blob, but a 32-point run inside it is not a
// compact cell.  Each CTA takes one aligned block of BLK sorted records (128 KiB of shared
// memory), and splits it recursively at the count median along the widest axis of the segment
// (a balanced kd-tree by sorting: bitonic sort of every segment, log2(BLK/32) levels), so every
// aligned run of 32*2^j records -- i.e. every pyramid node below the block -- becomes a kd cell.
// In simulation this cuts the leaves a query scans from 5.5 to 3.4 (tools/sim_tree.py).
__device__ __forceinline__ int ord_f32(float f)
{
    int i = __float_as_int(f);
    return i ^ ((i >> 31) & 0x7fffffff);
}

template <typename Out>
__device__ __forceinline__ bool kd_after(const Out &a, const Out &b, int axis)
{
    const auto ka = axis == 0 ? a.x : (axis == 1 ? a.y : a.z);
    const auto kb = axis == 0 ? b.x : (axis == 1 ? b.y : b.z);
    return ka > kb || (ka == kb && a.idx > b.idx);
}

// ---- sorting (key, position) pairs packed in 64 bits ----------------------------------------
__device__ __forceinline__ unsigned long long kd_shfl_xor(unsigned long long v, int lane_mask)
{
    unsigned lo = __shfl_xor_sync(0xffffffffu, (unsigned)v, lane_mask);
    unsigned hi = __shfl_xor_sync(0xffffffffu, (unsigned)(v >> 32), lane_mask);
    return ((unsigned long long)hi << 32) | lo;
}

// A warp owns 32*E consecutive values of the block, lane-interleaved: slot e of lane l is value
// wbase + 32*e + l, so shared-memory accesses are conflict-free, compare-exchange distances
// j < 32 are warp shuffles and distances 32 <= j < 32*E stay inside the thread.
template <int E, int J>   // J = in-thread slot distance (j / 32)
__device__ __forceinline__ void kd_local_step(unsigned long long (&r)[E], int ibase, int sz, int kk)
{
    if constexpr (J < E) {
#pragma unroll
        for (int e = 0; e < E; ++e) {
            if ((e & J) == 0) {
                const bool asc = (((ibase + 32 * e) & (sz - 1)) & kk) == 0;
                const unsigned long long a = r[e], b = r[e | J];
                if ((a > b) == asc) { r[e] = b; r[e | J] = a; }
            }
        }
    }
}

// One bitonic compare-exchange step (stage kk, distance j < 32 E); ibase = wbase + lane.
template <int E>
__device__ __forceinline__ void kd_reg_step(unsigned long long (&r)[E], int ibase, int sz, int kk, int j)
{
    if (j < 32) {   // partner = lane ^ j, same slot
#pragma unroll
        for (int e = 0; e < E; ++e) {
            const int i = ibase + 32 * e;
            const bool keep_min = ((i & j) == 0) == (((i & (sz - 1)) & kk) == 0);
            const unsigned long long p = kd_shfl_xor(r[e], j);
            r[e] = keep_min ? (p < r[e] ? p : r[e]) : (p > r[e] ? p : r[e]);
        }
    } else {        // both values in this thread: static register indices for each distance
        if (j == 128) kd_local_step<E, 4>(r, ibase, sz, kk);
        else if (j == 64) kd_local_step<E, 2>(r, ibase, sz, kk);
        else kd_local_step<E, 1>(r, ibase, sz, kk);
    }
}

template <typename Out, int BLK>
__global__ void __launch_bounds__(1024, 1) kd_refine_kernel(Out *pts, uint32_t n_pad)
{
    constexpr int E = BLK / 1024;       // values per thread
    constexpr int WSPAN = 32 * E;       // values covered by one warp
    extern __shared__ __align__(16) unsigned char kd_smem[];
    Out *s = reinterpret_cast<Out *>(kd_smem);
    unsigned long long *keys = reinterpret_cast<unsigned long long *>(kd_smem + sizeof(Out) * BLK);
    constexpr int MAXSEG = BLK / (2 * LEAF);
    __shared__ int seg_lo[3][MAXSEG], seg_hi[3][MAXSEG];
    __shared__ unsigned char seg_axis[MAXSEG];
    const uint32_t base = blockIdx.x * (uint32_t)BLK;
    const uint32_t cnt = min((uint32_t)BLK, n_pad - base);
    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const int ibase = (tid >> 5) * WSPAN + lane;      // this thread's slot e is value ibase + 32 e
    for (int i = tid; i < BLK; i += 1024) {
        Out p;
        if ((uint32_t)i < cnt) p = pts[base + i];
        else {
            p.x = FLT_MAX; p.y = FLT_MAX; p.z = FLT_MAX; p.idx = IDX_NONE;
            if constexpr (sizeof(Out) == 32) p.pad = 0;
        }
        s[i] = p;
    }
    __syncthreads();
    for (int sz = BLK; sz > LEAF; sz >>= 1) {
        const int nseg = BLK / sz;
        const int shift = __ffs(sz) - 1;
        if (tid < nseg) {
#pragma unroll
            for (int a = 0; a < 3; ++a) { seg_lo[a][tid] = 0x7fffffff; seg_hi[a][tid] = (int)0x80000000; }
        }
        __syncthreads();
        // segment bounding boxes: slots of a thread that fall in the same segment are reduced in
        // registers, then across the warp by shuffles; one lane issues the shared-memory atomics
        {
            const int per = sz >= WSPAN ? E : sz / 32;     // consecutive slots per segment
#pragma unroll
            for (int g0 = 0; g0 < E; ++g0) {
                if (g0 % per != 0) continue;
                int lo[3] = {0x7fffffff, 0x7fffffff, 0x7fffffff};
                int hi[3] = {(int)0x80000000, (int)0x80000000, (int)0x80000000};
#pragma unroll
                for (int e = 0; e < E; ++e) {
                    if (e >= g0 && e < g0 + per) {
                        const Out p = s[ibase + 32 * e];
                        if (p.idx != IDX_NONE) {
                            const int ex = ord_f32((float)p.x), ey = ord_f32((float)p.y), ez = ord_f32((float)p.z);
                            lo[0] = min(lo[0], ex); hi[0] = max(hi[0], ex);
                            lo[1] = min(lo[1], ey); hi[1] = max(hi[1], ey);
                            lo[2] = min(lo[2], ez); hi[2] = max(hi[2], ez);
                        }
                    }
                }
#pragma unroll
                for (int a = 0; a < 3; ++a) {
                    lo[a] = __reduce_min_sync(0xffffffffu, lo[a]);
                    hi[a] = __reduce_max_sync(0xffffffffu, hi[a]);
                }
                if (lane == 0) {
                    const int sg = (ibase + 32 * g0) >> shift;
#pragma unroll
                    for (int a = 0; a < 3; ++a) { atomicMin(&seg_lo[a][sg], lo[a]); atomicMax(&seg_hi[a][sg], hi[a]); }
                }
            }
        }
        __syncthreads();
        if (tid < nseg) {
            float ext[3];
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                int lo = seg_lo[a][tid], hi = seg_hi[a][tid];
                float flo = __int_as_float(lo ^ ((lo >> 31) & 0x7fffffff));
                float fhi = __int_as_float(hi ^ ((hi >> 31) & 0x7fffffff));
                ext[a] = hi >= lo ? fhi - flo : -1.0f;
            }
            int ax = 0;
            if (ext[1] > ext[ax]) ax = 1;
            if (ext[2] > ext[ax]) ax = 2;
            seg_axis[tid] = (unsigned char)ax;
        }
        __syncthreads();
        // Sort (coordinate key, position) pairs of every segment with a bitonic network; the
        // 16/32-byte records move only once per level.
        unsigned long long r[E];
#pragma unroll
        for (int e = 0; e < E; ++e) {
            const int i = ibase + 32 * e;
            const int ax = seg_axis[i >> shift];
            const Out p = s[i];
            const float c = (float)(ax == 0 ? p.x : (ax == 1 ? p.y : p.z));
            unsigned u = __float_as_uint(c);
            u = (u & 0x80000000u) ? ~u : (u | 0x80000000u);
            if (p.idx == IDX_NONE) u = 0xffffffffu;     // padding sorts last
            r[e] = ((unsigned long long)u << 32) | (unsigned)i;
        }
        const int top_reg = sz < WSPAN ? sz : WSPAN;
        for (int kk = 2; kk <= top_reg; kk <<= 1)
            for (int j = kk >> 1; j > 0; j >>= 1) kd_reg_step<E>(r, ibase, sz, kk, j);
        for (int kk = 2 * WSPAN; kk <= sz; kk <<= 1) {
#pragma unroll
            for (int e = 0; e < E; ++e) keys[ibase + 32 * e] = r[e];
            __syncthreads();
            int j = kk >> 1;
            for (; j >= WSPAN; j >>= 1) {
                for (int t = tid; t < BLK / 2; t += 1024) {
                    const int i = ((t & ~(j - 1)) << 1) | (t & (j - 1));
                    const int l = i | j;
                    const bool asc = ((i & (sz - 1)) & kk) == 0;
                    const unsigned long long a = keys[i], b = keys[l];
                    if ((a > b) == asc) { keys[i] = b; keys[l] = a; }
                }
                __syncthreads();
            }
#pragma unroll
            for (int e = 0; e < E; ++e) r[e] = keys[ibase + 32 * e];
            for (; j > 0; j >>= 1) kd_reg_step<E>(r, ibase, sz, kk, j);
        }
        // apply the permutation: each position receives the record the sort put there
        Out rec[E];
#pragma unroll
        for (int e = 0; e < E; ++e) rec[e] = s[(unsigned)(r[e] & 0xffffffffu)];
        __syncthreads();
#pragma unroll
        for (int e = 0; e < E; ++e) s[ibase + 32 * e] = rec[e];
        __syncthreads();
    }
    for (int i = tid; (uint32_t)i < cnt; i += 1024) pts[base + i] = s[i];
}

template <typename Out>
static int kd_refine(Out *pts, uint32_t n_pad, cudaStream_t s)
{
    constexpr int BLK = sizeof(Out) == 16 ? 8192 : 4096;
    const size_t smem = (size_t)BLK * (sizeof(Out) + sizeof(unsigned long long));
    PT_CUDA(cudaFuncSetAttribute(kd_refine_kernel<Out, BLK>,
                                 cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kd_refine_kernel<Out, BLK><<<(n_pad + BLK - 1) / BLK, 1024, smem, s>>>(pts, n_pad);
    count_launch();
    PT_CUDA(cudaGetLastError());
    return PT_OK;
}

// ---- leaf boxes: one warp per 32-point leaf ------------------------------------------------
__device__ __forceinline__ float f_dn(double v) { return __double2float_rd(v); }
__device__ __forceinline__ float f_up(double v) { return __double2float_ru(v); }

template <typename Out>
__global__ void __launch_bounds__(256) leaf_box_kernel(const Out *pts, uint32_t n,
                                                       uint32_t n_leaves, Box *boxes)
{
    uint32_t leaf = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    uint32_t lane = threadIdx.x & 31;
    if (leaf >= n_leaves) return;
    uint32_t i = leaf * LEAF + lane;
    float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
    if (i < n) {
        Out p = pts[i];
        lo[0] = f_dn(p.x); lo[1] = f_dn(p.y); lo[2] = f_dn(p.z);
        hi[0] = f_up(p.x); hi[1] = f_up(p.y); hi[2] = f_up(p.z);
    }
#pragma unroll
    for (int a = 0; a < 3; ++a) {
#pragma unroll
        for (int s = 16; s > 0; s >>= 1) {
            lo[a] = fminf(lo[a], __shfl_xor_sync(0xffffffffu, lo[a], s));
            hi[a] = fmaxf(hi[a], __shfl_xor_sync(0xffffffffu, hi[a], s));
        }
    }
    if (lane == 0) {
        Box b;
        b.lox = lo[0]; b.loy = lo[1]; b.loz = lo[2];
        b.hix = hi[0]; b.hiy = hi[1]; b.hiz = hi[2];
        b.pad0 = 0.f; b.pad1 = 0.f;
        boxes[leaf] = b;
    }
}

__global__ void __launch_bounds__(256) pyramid_kernel(const Box *child, uint32_t n_child,
                                                      Box *parent, uint32_t n_parent)
{
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_parent) return;
    Box a = child[2 * i];
    if (2 * i + 1 < n_child) {
        Box b = child[2 * i + 1];
        a.lox = fminf(a.lox, b.lox); a.loy = fminf(a.loy, b.loy); a.loz = fminf(a.loz, b.loz);
        a.hix = fmaxf(a.hix, b.hix); a.hiy = fmaxf(a.hiy, b.hiy); a.hiz = fmaxf(a.hiz, b.hiz);
    }
    parent[i] = a;
}

// ---- K2: sort ------------------------------------------------------------------------------
// Only key bits [first_bit, 63) are ordered: the grid tables need cells contiguous down to level
// 16 (48 key bits) and the 32-point leaves gain nothing from the order inside a cell that small.
static int sort_pairs(unsigned long long *&keys, unsigned long long *keys_alt, uint32_t *&vals,
                      uint32_t *vals_alt, uint32_t n, int first_bit, void *ws, cudaStream_t s)
{
    if (opt_sort() != 0) {   // hand-written LSD radix sort (pt_sort.cu), the default
        unsigned long long *ko = nullptr;
        uint32_t *vo = nullptr;
        int rc = radix_sort_pairs(keys, keys_alt, vals, vals_alt, n, first_bit, 63, ws, s, &ko, &vo);
        if (rc != PT_OK) return rc;
        keys = ko;
        vals = vo;
        return PT_OK;
    }
    // library radix sort (CCCL), kept as the reference point the hand-written sort is measured against
    cub::DoubleBuffer<unsigned long long> dk(keys, keys_alt);
    cub::DoubleBuffer<uint32_t> dv(vals, vals_alt);
    size_t tmp_bytes = 0;
    PT_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, dk, dv, (int)n, first_bit, 63, s));
    void *tmp = nullptr;
    PT_CUDA(cudaMalloc(&tmp, tmp_bytes ? tmp_bytes : 16));
    cudaError_t e = cub::DeviceRadixSort::SortPairs(tmp, tmp_bytes, dk, dv, (int)n, first_bit, 63, s);
    count_launch(9);
    cudaError_t e2 = cudaStreamSynchronize(s);
    cudaFree(tmp);
    if (e != cudaSuccess) return map_cuda_error(e);
    if (e2 != cudaSuccess) return map_cuda_error(e2);
    keys = dk.Current();
    vals = dv.Current();
    return PT_OK;
}

static inline unsigned int cdiv(uint64_t a, uint64_t b) { return (unsigned int)((a + b - 1) / b); }

// Build temporaries (sort keys / values / counters: ~24 bytes per point), the sorted points, the
// boxes, the cell tables and the per-launch hand-over lists come from a PRIVATE stream-ordered
// memory pool per device with an unlimited release threshold, so a rebuild reuses them instead
// of paying cudaMalloc / cudaFree (3-30 ms per GB, host-synchronous) every time -- and the host
// application's default pool keeps its own retention policy.
static std::mutex g_pool_mutex;
static cudaMemPool_t g_pools[64] = {};

static int device_pool(int dev, cudaMemPool_t *out)
{
    if (dev < 0 || dev >= 64) return PT_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> lock(g_pool_mutex);
    if (!g_pools[dev]) {
        cudaMemPoolProps props{};
        props.allocType = cudaMemAllocationTypePinned;
        props.handleTypes = cudaMemHandleTypeNone;
        props.location.type = cudaMemLocationTypeDevice;
        props.location.id = dev;
        cudaMemPool_t pool = nullptr;
        PT_CUDA(cudaMemPoolCreate(&pool, &props));
        unsigned long long keep = ~0ull;
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
        g_pools[dev] = pool;
    }
    *out = g_pools[dev];
    return PT_OK;
}

// Debug option "pool_guard": every device allocation of the library gets GUARD bytes of 0xA5 in
// front and behind, checked when it is released; get_option("pool_guard_hits") counts the
// allocations found damaged.  (The library's own bounds check: tools/sanitize.py,
// tests/test_gpu_parity.py::test_guard_words_stay_intact.)
constexpr size_t GUARD = 256;
static std::mutex g_guard_mutex;
static std::unordered_map<void *, size_t> g_guarded;   // user pointer -> user bytes
static std::atomic<int> g_guard_hits{0};
int guard_hits() { return g_guard_hits.load(); }

static int guard_arm(void *base, size_t bytes, cudaStream_t s, void **user)
{
    PT_CUDA(cudaMemsetAsync(base, 0xA5, GUARD, s));
    PT_CUDA(cudaMemsetAsync((char *)base + GUARD + bytes, 0xA5, GUARD, s));
    *user = (char *)base + GUARD;
    std::lock_guard<std::mutex> lock(g_guard_mutex);
    try { g_guarded[*user] = bytes; } catch (...) { return PT_ERR_OUT_OF_MEMORY; }
    return PT_OK;
}

// returns the pointer to hand to cudaFree / cudaFreeAsync
static void *guard_release(void *user, cudaStream_t s)
{
    size_t bytes = 0;
    {
        std::lock_guard<std::mutex> lock(g_guard_mutex);
        auto it = g_guarded.find(user);
        if (it == g_guarded.end()) return user;
        bytes = it->second;
        g_guarded.erase(it);
    }
    char *base = (char *)user - GUARD;
    unsigned char h[2 * GUARD];
    memset(h, 0, sizeof h);
    cudaMemcpyAsync(h, base, GUARD, cudaMemcpyDeviceToHost, s);
    cudaMemcpyAsync(h + GUARD, base + GUARD + bytes, GUARD, cudaMemcpyDeviceToHost, s);
    cudaStreamSynchronize(s);
    int bad = 0;
    for (size_t i = 0; i < 2 * GUARD; ++i) bad += h[i] != 0xA5;
    if (bad) {
        g_guard_hits.fetch_add(1);
        fprintf(stderr, "[points_transfer] guard words damaged: %d bytes around an allocation of %zu bytes\n", bad, bytes);
    }
    return base;
}

int pool_alloc(void **p, size_t bytes, cudaStream_t s)
{
    int dev = 0;
    PT_CUDA(cudaGetDevice(&dev));
    cudaMemPool_t pool;
    PT_TRY(device_pool(dev, &pool));
    if (!bytes) bytes = 16;
    if (!opt_pool_guard()) {
        PT_CUDA(cudaMallocFromPoolAsync(p, bytes, pool, s));
        return PT_OK;
    }
    void *base = nullptr;
    PT_CUDA(cudaMallocFromPoolAsync(&base, bytes + 2 * GUARD, pool, s));
    return guard_arm(base, bytes, s, p);
}

void pool_free(void *p, cudaStream_t s)
{
    if (p) cudaFreeAsync(guard_release(p, s), s);
}

// cudaMalloc / cudaFree for the long-lived buffers of an index, with the same guard words.
int dev_alloc(void **p, size_t bytes)
{
    if (!bytes) bytes = 16;
    if (!opt_pool_guard()) {
        PT_CUDA(cudaMalloc(p, bytes));
        return PT_OK;
    }
    void *base = nullptr;
    PT_CUDA(cudaMalloc(&base, bytes + 2 * GUARD));
    return guard_arm(base, bytes, nullptr, p);
}

void dev_free(void *p)
{
    if (p) cudaFree(guard_release(p, nullptr));
}

void pool_trim(int device, size_t keep_bytes)
{
    std::lock_guard<std::mutex> lock(g_pool_mutex);
    if (device >= 0 && device < 64 && g_pools[device]) cudaMemPoolTrimTo(g_pools[device], keep_bytes);
    cudaGetLastError();
}

static int temp_alloc(void **p, size_t bytes, cudaStream_t s) { return pool_alloc(p, bytes, s); }

template <typename In, typename Out>
static int build_impl(pt_index *ix, In in, uint32_t n)
{
    cudaStream_t s = ix->stream;
    PT_CUDA(cudaEventRecord(ix->ev[0], s));
    auto wall0 = std::chrono::steady_clock::now();
    auto lap = [&](const char *what) {   // PT_VERBOSE=1: host wall-clock per build phase
        if (!verbose()) return;
        cudaStreamSynchronize(s);
        auto now = std::chrono::steady_clock::now();
        fprintf(stderr, "[points_transfer] build %-18s %8.3f ms\n", what,
                std::chrono::duration<double, std::milli>(now - wall0).count());
        wall0 = now;
    };
    ix->n = n;
    ix->n_leaves = cdiv(n, LEAF);
    ix->coord_f64 = sizeof(Out) == 32;
    for (int a = 0; a < 3; ++a) { ix->bb_lo[a] = 0; ix->bb_hi[a] = 0; }
    ix->grid = GridParams{};
    ix->pyr = Pyramid{};
    ix->w_levels = 0;
    ix->t_levels = 0;
    if (n == 0) { ix->build_ms = 0; return PT_OK; }

    // K1: bbox
    BBoxAcc *acc = nullptr, h_acc;
    PT_TRY(temp_alloc((void **)&acc, sizeof(BBoxAcc), s));
    for (int a = 0; a < 3; ++a) { h_acc.lo[a] = ~0ull; h_acc.hi[a] = 0ull; }
    h_acc.non_finite = 0; h_acc.pad = 0;
    PT_CUDA(cudaMemcpyAsync(acc, &h_acc, sizeof h_acc, cudaMemcpyHostToDevice, s));
    {
        unsigned int blocks = cdiv(n, 256);
        if (blocks > (unsigned)ix->sm_count * 8u) blocks = (unsigned)ix->sm_count * 8u;
        bbox_kernel<In><<<blocks, 256, 0, s>>>(in, n, acc);
        count_launch();
    }
    PT_CUDA(cudaMemcpyAsync(&h_acc, acc, sizeof h_acc, cudaMemcpyDeviceToHost, s));
    PT_CUDA(cudaStreamSynchronize(s));
    pool_free(acc, s);
    if (h_acc.non_finite) return PT_ERR_NON_FINITE;
    KeyParams kp;
    double ext = 0;
    for (int a = 0; a < 3; ++a) {
        ix->bb_lo[a] = dec_f64(h_acc.lo[a]);
        ix->bb_hi[a] = dec_f64(h_acc.hi[a]);
        kp.lo[a] = ix->bb_lo[a];
        ext = fmax(ext, ix->bb_hi[a] - ix->bb_lo[a]);
    }
    kp.inv_cell = ext > 0 ? 2097152.0 / ext : 0.0;
    if (!std::isfinite(kp.inv_cell)) kp.inv_cell = 0.0;
    kp.order = opt_order();

    lap("bbox");
    // K1: keys, K2: sort
    unsigned long long *keys = nullptr, *keys_alt = nullptr;
    uint32_t *vals = nullptr, *vals_alt = nullptr;
    // one arena for all sort temporaries (cudaMalloc costs milliseconds per call)
    const size_t kbytes = (sizeof(unsigned long long) * (size_t)n + 255) & ~(size_t)255;
    const size_t vbytes = (sizeof(uint32_t) * (size_t)n + 255) & ~(size_t)255;
    char *arena = nullptr;
    PT_TRY(temp_alloc((void **)&arena, 2 * kbytes + 2 * vbytes + radix_sort_workspace_bytes(n), s));
    keys = (unsigned long long *)arena;
    keys_alt = (unsigned long long *)(arena + kbytes);
    vals = (uint32_t *)(arena + 2 * kbytes);
    vals_alt = (uint32_t *)(arena + 2 * kbytes + vbytes);
    void *sort_ws = arena + 2 * kbytes + 2 * vbytes;
    lap("alloc keys");
    morton_kernel<In><<<cdiv(n, 256), 256, 0, s>>>(in, n, kp, keys, vals);
    count_launch();
    lap("keys");
    struct ArenaGuard {    // the sort arena goes back to the pool on every exit path
        char *p; cudaStream_t s;
        ~ArenaGuard() { pool_free(p, s); }
    } arena_guard{arena, s};
    // "sort_bits" 0 (default) = auto: 40 bits order the cells down to level 13 -- finer cells hold
    // less than one point until a cloud has some 10^8 points (a surface fills <= 4^13 = 67 M of
    // them), so the sixth pass would only order points inside one cell; larger clouds get 48.
    int sort_bits = opt_sort_bits();
    if (sort_bits <= 0) sort_bits = n <= (1u << 27) ? 40 : 48;
    sort_bits = sort_bits < 8 ? 8 : (sort_bits > 63 ? 63 : sort_bits);
    const int passes = (sort_bits + 7) / 8;                      // 8-bit digits from the top of the key down
    const int first_bit = (kp.order == 2 || passes >= 8) ? 0 : 63 - 8 * passes;
    int rc = sort_pairs(keys, keys_alt, vals, vals_alt, n, first_bit, sort_ws, s);
    lap("sort");
    if (rc != PT_OK) return rc;

    // gather into leaves
    size_t n_pad = (size_t)ix->n_leaves * LEAF;
    Out *pts = nullptr;
    PT_TRY(temp_alloc((void **)&pts, sizeof(Out) * n_pad, s));   // pooled: a rebuild reuses the block
    // attributes in sorted order for knn_grid_span_kernel (float4 records with cell tables only):
    // the winners of a sample sit in a few adjacent cells, so their records share DRAM lines
    if (ix->attrs && sizeof(Out) == 16 && kp.order != 2 && opt_grid() != 0 && n >= 64)
        PT_TRY(temp_alloc((void **)&ix->attrs_curve, sizeof(pt_attr) * (size_t)n, s));
    gather_kernel<In, Out><<<cdiv(n_pad, 256), 256, 0, s>>>(in, vals, n, (uint32_t)n_pad, pts, ix->attrs,
                                                            ix->attrs_curve);
    count_launch();
    ix->pts = pts;
    lap("gather");
    if (kp.order == 2) PT_TRY(kd_refine<Out>(pts, (uint32_t)n_pad, s));
    lap("kd refine");
    // cell tables over the curve order (the kd refinement reorders inside blocks: no cell runs)
    if (kp.order != 2) PT_TRY(build_grid(ix, keys, first_bit, kp.lo, kp.inv_cell, ext));
    lap("grid tables");
    if (sizeof(Out) == 16) PT_TRY(build_blocks(ix));
    lap("block runs");

    // box pyramid
    uint64_t total = 0;
    uint32_t cnt = ix->n_leaves;
    int levels = 0;
    uint32_t counts[MAX_PYR_LEVELS];
    for (;;) {
        counts[levels++] = cnt;
        total += (cnt + 7u) & ~7u;   // every level starts 256-byte aligned: an 8-box group is 2 lines
        if (cnt == 1) break;
        cnt = (cnt + 1) / 2;
    }
    PT_TRY(temp_alloc((void **)&ix->boxes, sizeof(Box) * total, s));
    Box *lvl = ix->boxes;
    for (int j = 0; j < levels; ++j) {
        ix->pyr.level[j] = lvl;
        ix->pyr.count[j] = counts[j];
        lvl += (counts[j] + 7u) & ~7u;
    }
    ix->pyr.n_levels = levels;
    leaf_box_kernel<Out><<<cdiv((uint64_t)ix->n_leaves * 32, 256), 256, 0, s>>>(
        pts, n, ix->n_leaves, const_cast<Box *>(ix->pyr.level[0]));
    count_launch();
    for (int j = 1; j < levels; ++j) {
        pyramid_kernel<<<cdiv(counts[j], 256), 256, 0, s>>>(
            ix->pyr.level[j - 1], counts[j - 1], const_cast<Box *>(ix->pyr.level[j]), counts[j]);
        count_launch();
    }
    int t = 1;
    for (uint64_t cap = 32; cap < ix->n_leaves; cap *= 32) ++t;
    ix->w_levels = t;
    t = 1;
    for (uint64_t cap = 8; cap < ix->n_leaves; cap *= 8) ++t;
    ix->t_levels = t;

    PT_CUDA(cudaEventRecord(ix->ev[1], s));
    PT_CUDA(cudaStreamSynchronize(s));
    lap("boxes");
    PT_CUDA(cudaEventElapsedTime(&ix->build_ms, ix->ev[0], ix->ev[1]));
    pool_free(arena, s);
    arena_guard.p = nullptr;
    cudaStreamSynchronize(s);
    pool_trim(ix->device, opt_pool_keep_bytes());   // "pool_keep_mb" of it stays mapped for the next build
    ix->device_bytes = sizeof(Out) * n_pad + sizeof(Box) * total + ix->grid_bytes + ix->blk_bytes +
                       (ix->attrs ? sizeof(pt_attr) * (size_t)n : 0) +
                       (ix->attrs_curve ? sizeof(pt_attr) * (size_t)n : 0) +
                       (ix->ids ? sizeof(int32_t) * (size_t)n : 0);
    return PT_OK;
}

int build_index_f4(pt_index *ix, const float4 *pos, uint32_t n, bool out_f64)
{
    InF4 in{pos};
    return out_f64 ? build_impl<InF4, PointD>(ix, in, n) : build_impl<InF4, PointF>(ix, in, n);
}
int build_index_d4(pt_index *ix, const double *pos, uint32_t n, bool out_f64)
{
    InD4 in{pos};
    return out_f64 ? build_impl<InD4, PointD>(ix, in, n) : build_impl<InD4, PointF>(ix, in, n);
}
int build_index_d3(pt_index *ix, const double *pos, uint32_t n, bool out_f64)
{
    InD3 in{pos};
    return out_f64 ? build_impl<InD3, PointD>(ix, in, n) : build_impl<InD3, PointF>(ix, in, n);
}

// ---- ingest of the reference's 80-byte AoS `struct Point` (src/Point.h:1-6) ------------------
struct Raw80 {
    double ver[3];
    double normal[3];
    int    color[3];
    int    pad;
    double U, V;
};
static_assert(sizeof(Raw80) == PT_POINT_STRIDE, "Point must be 80 bytes");

__global__ void __launch_bounds__(256) unpack_points_kernel(const Raw80 *raw, uint32_t count,
                                                            double *xyz, pt_attr *attrs,
                                                            unsigned int *not_representable)
{
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    bool bad = false;
    if (i < count) {
        const Raw80 &r = raw[i];
        double x = r.ver[0], y = r.ver[1], z = r.ver[2];
        xyz[3 * (size_t)i] = x; xyz[3 * (size_t)i + 1] = y; xyz[3 * (size_t)i + 2] = z;
        bad = ((double)(float)x != x) || ((double)(float)y != y) || ((double)(float)z != z);
        pt_attr a;
        a.nx = (float)r.normal[0]; a.ny = (float)r.normal[1]; a.nz = (float)r.normal[2];
        a.r = (uint8_t)min(max(r.color[0], 0), 255);
        a.g = (uint8_t)min(max(r.color[1], 0), 255);
        a.b = (uint8_t)min(max(r.color[2], 0), 255);
        a.a = 255;
        attrs[i] = a;
    }
    if (__any_sync(0xffffffffu, bad) && (threadIdx.x & 31) == 0) atomicOr(not_representable, 1u);
}

__global__ void __launch_bounds__(256) unpack_queries_kernel(const Raw80 *raw, uint32_t m,
                                                             double *xyz)
{
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    xyz[3 * (size_t)i] = raw[i].ver[0];
    xyz[3 * (size_t)i + 1] = raw[i].ver[1];
    xyz[3 * (size_t)i + 2] = raw[i].ver[2];
}

int unpack_queries_aos(const void *raw80_dev, size_t m, double *xyz_dev, cudaStream_t s)
{
    if (m == 0) return PT_OK;
    unpack_queries_kernel<<<cdiv(m, 256), 256, 0, s>>>((const Raw80 *)raw80_dev, (uint32_t)m,
                                                       xyz_dev);
    count_launch();
    PT_CUDA(cudaGetLastError());
    return PT_OK;
}

int ingest_points_aos(pt_index *ix, const void *points, size_t n, int coord_mode,
                      double **xyz_out, bool *representable)
{
    (void)coord_mode;
    cudaStream_t s = ix->stream;
    *xyz_out = nullptr;
    *representable = true;
    if (n == 0) return PT_OK;
    // one exit path: whatever was acquired before a failure is released (ix->attrs belongs to the
    // handle and is released with it)
    double *xyz = nullptr;
    unsigned int *flag = nullptr;
    Raw80 *stage[2] = {nullptr, nullptr};
    cudaEvent_t done[2] = {nullptr, nullptr};
    unsigned int h_flag = 0;
    cudaError_t e = cudaSuccess;
    auto ok = [&](cudaError_t r) { if (e == cudaSuccess) e = r; return e == cudaSuccess; };
    auto got = [&](int st) {
        return ok(st == PT_OK ? cudaSuccess : st == PT_ERR_OUT_OF_MEMORY ? cudaErrorMemoryAllocation : cudaErrorUnknown);
    };
    // chunked upload through two device staging buffers
    const size_t chunk = (size_t)1 << 22;  // 4 Mi records = 320 MiB per buffer
    const size_t cap = n < chunk ? n : chunk;
    if (got(dev_alloc((void **)&xyz, sizeof(double) * 3 * n)) && got(pool_alloc((void **)&ix->attrs, sizeof(pt_attr) * n, s)) &&
        got(dev_alloc((void **)&flag, sizeof(unsigned int))) && ok(cudaMemsetAsync(flag, 0, sizeof(unsigned int), s)) &&
        got(dev_alloc((void **)&stage[0], sizeof(Raw80) * cap)) && got(dev_alloc((void **)&stage[1], sizeof(Raw80) * cap)) &&
        ok(cudaEventCreateWithFlags(&done[0], cudaEventDisableTiming)) &&
        ok(cudaEventCreateWithFlags(&done[1], cudaEventDisableTiming))) {
        int b = 0;
        for (size_t off = 0; off < n && e == cudaSuccess; off += cap, b ^= 1) {
            const size_t cnt = n - off < cap ? n - off : cap;
            if (!ok(cudaEventSynchronize(done[b]))) break;
            if (!ok(cudaMemcpyAsync(stage[b], (const char *)points + off * sizeof(Raw80), cnt * sizeof(Raw80),
                                    cudaMemcpyHostToDevice, s)))
                break;
            unpack_points_kernel<<<cdiv(cnt, 256), 256, 0, s>>>(stage[b], (uint32_t)cnt, xyz + 3 * off,
                                                                ix->attrs + off, flag);
            count_launch();
            ok(cudaEventRecord(done[b], s));
        }
        if (e == cudaSuccess) ok(cudaMemcpyAsync(&h_flag, flag, sizeof h_flag, cudaMemcpyDeviceToHost, s));
    }
    const cudaError_t es = cudaStreamSynchronize(s);      // nothing is still reading `points` after this
    if (e == cudaSuccess) e = es;
    dev_free(stage[0]); dev_free(stage[1]); dev_free(flag);
    if (done[0]) cudaEventDestroy(done[0]);
    if (done[1]) cudaEventDestroy(done[1]);
    if (e != cudaSuccess) {
        dev_free(xyz);
        cudaGetLastError();
        if (verbose()) fprintf(stderr, "[points_transfer] ingest: %s\n", cudaGetErrorString(e));
        return map_cuda_error(e);
    }
    *representable = h_flag == 0;
    *xyz_out = xyz;
    return PT_OK;
}

}  // namespace pt

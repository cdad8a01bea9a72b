// pt_knn_thread.cuh -- variant 2 ("thread"): one thread per sample, all per-sample state in
// shared-memory columns (element j of thread t at [j * T_THREADS + t]: conflict-free).
//
//   * traversal : best-first over the 8-wide pyramid levels.  The queue holds one entry per
//                 partially visited node -- (fp32 bound of its nearest unvisited child, node id,
//                 8-bit mask of unvisited children) -- so it stays tiny; a popped node is
//                 re-expanded (its 8 child boxes re-tested) to pick the next child.  After an
//                 expansion the nearest child is followed directly while it is still the best
//                 candidate ("dive"), which costs no queue traffic.
//   * leaf scan : 32 points, exact fp64 metric (src/Distance.h:6-11); candidates that beat the
//                 current k-th are parked in a small pending column and drained into the heap
//                 in a warp-converged loop, so heap updates do not serialise the scan.
//   * top-k     : bounded max-heap column keyed (d2, index); heap-sorted at the end.
// Samples whose queue overflows go to the warp kernel (exact fallback).
#pragma once

namespace pt {

#ifndef PT_T_THREADS
#define PT_T_THREADS 32      // one warp per block: finest scheduling granularity (sweep: 32 > 64 > 128)
#endif
#ifndef PT_T_CHUNK
#define PT_T_CHUNK 8          // leaf points scanned between two drains (= pending capacity)
#endif
constexpr int T_THREADS = PT_T_THREADS;
constexpr int TPD_CAP = PT_T_CHUNK;

// sift `(cd, ci)` down from `pos` in the max-heap column of size n (element j at [j * STRIDE])
template <int STRIDE>
__device__ __forceinline__ void heap_sift_s(double *hd, int *hi, int pos, int n, double cd, int ci)
{
    for (;;) {
        int c = 2 * pos + 1;
        if (c >= n) break;
        double xd = hd[c * STRIDE];
        int xi = hi[c * STRIDE];
        if (c + 1 < n) {
            double yd = hd[(c + 1) * STRIDE];
            int yi = hi[(c + 1) * STRIDE];
            if (key_less(xd, xi, yd, yi)) { xd = yd; xi = yi; ++c; }
        }
        if (!key_less(cd, ci, xd, xi)) break;
        hd[pos * STRIDE] = xd;
        hi[pos * STRIDE] = xi;
        pos = c;
    }
    hd[pos * STRIDE] = cd;
    hi[pos * STRIDE] = ci;
}

__device__ __forceinline__ void heap_sift(double *hd, int *hi, int pos, int n, double cd, int ci)
{
    heap_sift_s<T_THREADS>(hd, hi, pos, n, cd, ci);
}

__device__ __forceinline__ void heapify(double *hd, int *hi, int n)
{
    for (int s = n / 2 - 1; s >= 0; --s)
        heap_sift(hd, hi, s, n, hd[s * T_THREADS], hi[s * T_THREADS]);
}

// Sorts the hn candidates of a column ascending by (d2, index) and writes every output of the
// sample: neighbour ids, d2, candidate records, blended colour / normal (frozen definition).
#ifndef PT_EMIT_PREFETCH
#define PT_EMIT_PREFETCH 1
#endif
template <int STRIDE>
__device__ __forceinline__ void emit_sample(const QueryParams &P, uint32_t q, double *hd, int *hi,
                                            int hn)
{
    const int k = P.k;
#if PT_EMIT_PREFETCH
    // the winners' attribute records (and ids) are random 16 / 4-byte gathers: pull them into
    // L2 now, the sort below hides the DRAM latency
    if ((P.rgba_out || P.normal_out || P.cand_out) && P.attrs)
        for (int j = 0; j < hn; ++j)
            asm volatile("prefetch.global.L2 [%0];" ::"l"(P.attrs + hi[j * STRIDE]));
    if (P.ids)
        for (int j = 0; j < hn; ++j)
            asm volatile("prefetch.global.L2 [%0];" ::"l"(P.ids + hi[j * STRIDE]));
#endif
    for (int s = hn / 2 - 1; s >= 0; --s)
        heap_sift_s<STRIDE>(hd, hi, s, hn, hd[s * STRIDE], hi[s * STRIDE]);
    for (int n = hn - 1; n > 0; --n) {
        const double ld = hd[n * STRIDE];
        const int li = hi[n * STRIDE];
        hd[n * STRIDE] = hd[0];
        hi[n * STRIDE] = hi[0];
        heap_sift_s<STRIDE>(hd, hi, 0, n, ld, li);
    }
    const bool want_blend = P.rgba_out || P.normal_out;
    const bool need_attr = (want_blend || P.cand_out) && P.attrs;
    const size_t o = (size_t)q * k;
    const int mode = (hn > 0 && hd[0] == 0.0) ? 1 : 0;
    BlendAcc acc;
    acc.reset();
    for (int j = 0; j < k; ++j) {
        const bool has = j < hn;
        const double d = has ? hd[j * STRIDE] : INFINITY;
        const int li = has ? hi[j * STRIDE] : IDX_NONE;
        const int gid = has ? (P.ids ? __ldg(P.ids + li) : li) : -1;
        if (P.idx_out) P.idx_out[o + j] = gid;
        if (P.d2_out) P.d2_out[o + j] = d;
        AttrRaw at{0.f, 0.f, 0.f, 0u};
        if (has && need_attr) at = load_attr(P.attrs + li);
        if (P.cand_out) store_cand(P.cand_out + o + j, d, gid, at);
        if (has && want_blend) acc.add(blend_weight(mode, d, j), at.rgba, at.nx, at.ny, at.nz);
    }
    if (want_blend) {
        uint8_t *ro = P.rgba_out ? P.rgba_out + 4 * (size_t)q : nullptr;
        float *no = P.normal_out ? P.normal_out + 3 * (size_t)q : nullptr;
        if (hn == 0) { store_empty_blend(ro, no); return; }
        if (!acc.weight_ok()) {   // overflowed weights: nearest neighbour only
            acc.reset();
            AttrRaw at = load_attr(P.attrs + hi[0]);
            acc.add(1.0, at.rgba, at.nx, at.ny, at.nz);
        }
        acc.store(ro, no);
    }
}

#ifndef PT_T_MIN_BLOCKS
#define PT_T_MIN_BLOCKS 17      // = the shared-memory limit at k = 16: keeps the register count from capping occupancy
#endif
template <typename PT>
__global__ void __launch_bounds__(T_THREADS, PT_T_MIN_BLOCKS)
knn_thread_kernel(const QueryParams P, uint32_t *ovf_count, uint32_t *ovf_list)
{
    extern __shared__ __align__(16) unsigned char t_smem[];
    const int k = P.k;
    const unsigned tid = threadIdx.x;
    double *hd = reinterpret_cast<double *>(t_smem) + tid;                      // [k]
    double *pdd = hd + k * T_THREADS;                                             // [TPD_CAP]
    int *hi = reinterpret_cast<int *>(t_smem + sizeof(double) * (k + TPD_CAP) * T_THREADS) + tid;
    int *pdi = hi + k * T_THREADS;                                                // [TPD_CAP]
    uint32_t *pqk = reinterpret_cast<uint32_t *>(pdi + TPD_CAP * T_THREADS);     // [TPQ_CAP]
    uint32_t *pqw = pqk + TPQ_CAP * T_THREADS;                                    // [TPQ_CAP]

    // list mode (second stage behind the grid kernel, pt_knn_grid.cuh): sample qlist[i], i < *qcount,
    // blocks of T_THREADS list entries grid-stride (the grid is sized to the resident blocks,
    // launch_thread); the list is read after the kernel that wrote it has completed
    pdl_wait();
    uint32_t m_eff = P.qlist ? min(*P.qcount, P.m) : P.m;
    if (P.qlist && m_eff < P.qlist_min) m_eff = 0;       // short lists are the warp kernel's
#pragma unroll 1
    for (uint32_t b0 = blockIdx.x * T_THREADS; b0 < m_eff; b0 += gridDim.x * T_THREADS) {
        const uint32_t qi = b0 + tid;
        const bool live = qi < m_eff;
        const uint32_t q = live ? (P.qlist ? P.qlist[qi] : qi) : 0u;
        bool done = !live || P.t_levels == 0;
        bool overflow = false;

        double qx = 0, qy = 0, qz = 0, r2 = 0;
        if (live) {
            qx = __ldg(P.queries + 3 * (size_t)q);
            qy = __ldg(P.queries + 3 * (size_t)q + 1);
            qz = __ldg(P.queries + 3 * (size_t)q + 2);
            r2 = P.r2_per_query ? __ldg(P.r2_per_query + q) : P.r2;
        }
        float bound = __double2float_ru(r2);

#ifdef PT_STATS
        unsigned st_[16];
        for (int a = 0; a < 16; ++a) st_[a] = 0;
#endif
        int hn = 0;                 // candidates held; the column is a max-heap once hn == k
        double root_d = INFINITY;   // heap root (current k-th) -- meaningful once hn == k
        int root_i = IDX_NONE;
        Traverser<PT, T_THREADS> tr(P, pqk, pqw, qx, qy, qz, !done);
#ifdef PT_STATS
        tr.st_ = st_;
#endif

        for (;;) {
            const int leaf = tr.next_leaf(bound, hn < k, done);
            if (__all_sync(0xffffffffu, done)) break;

            // ---- leaf phase: every lane that holds a leaf scans it, 8 points per chunk -------------
            PT_STAT(1, leaf >= 0 ? 1 : 0);
            if (tid == 0) PT_STAT(7, 1);
            const uint32_t base = (uint32_t)(leaf < 0 ? 0 : leaf) * LEAF;
#pragma unroll 1
            for (int chunk = 0; chunk < LEAF / PT_T_CHUNK; ++chunk) {
                int pend = 0;
                if (leaf >= 0) {
#pragma unroll
                    for (int p = 0; p < PT_T_CHUNK; ++p) {
                        const uint32_t pi = base + chunk * PT_T_CHUNK + p;
                        double px, py, pz;
                        int pidx;
                        PointLoad<PT>::load(P.pts, pi, px, py, pz, pidx);
                        const double d = dist2_exact(qx, qy, qz, px, py, pz);
                        if (pi < P.n && d <= r2 && (hn < k || key_less(d, pidx, root_d, root_i))) {
                            pdd[pend * T_THREADS] = d;
                            pdi[pend * T_THREADS] = pidx;
                            ++pend;
                            PT_STAT(6, 1);
                        }
                    }
                }
                while (__any_sync(0xffffffffu, pend > 0)) {
                    if (tid == 0) PT_STAT(10, 1);
                    if (pend > 0) {
                        --pend;
                        const double d = pdd[pend * T_THREADS];
                        const int pidx = pdi[pend * T_THREADS];
                        if (hn < k || key_less(d, pidx, root_d, root_i)) PT_STAT(5, 1);
                        if (hn < k) {
                            hd[hn * T_THREADS] = d;
                            hi[hn * T_THREADS] = pidx;
                            if (++hn == k) {
                                heapify(hd, hi, k);
                                root_d = hd[0];
                                root_i = hi[0];
                            }
                        } else if (key_less(d, pidx, root_d, root_i)) {
                            heap_sift(hd, hi, 0, k, d, pidx);
                            root_d = hd[0];
                            root_i = hi[0];
                        }
                    }
                }
            }
            if (hn == k) bound = __double2float_ru(fmin(root_d, r2));
        }

        overflow = tr.proof_failed(bound);
#ifdef PT_STATS
        st_[8] = overflow ? 1 : 0;
        st_[9] = live ? 1 : 0;
        for (int a = 0; a < 12; ++a) {
            unsigned v = st_[a];
            for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
            if (tid == 0 && v) atomicAdd(&g_stats[a], (unsigned long long)v);
        }
#endif
        if (live && overflow) {
            uint32_t slot = atomicAdd(ovf_count, 1u);
            ovf_list[slot] = q;
        } else if (live) {
            emit_sample<T_THREADS>(P, q, hd, hi, hn);   // sort ascending (d2, index), outputs, blend
        }
    }
}

static inline size_t thread_kernel_smem(int k)
{
    return (size_t)T_THREADS * ((size_t)(k + TPD_CAP) * 12 + (size_t)TPQ_CAP * 8);
}

// As launch_scan: a list-mode launch gets the resident blocks; `pdl`: a programmatic dependent.
template <typename PT>
static int launch_thread(const QueryParams &qp, int sm_count, bool pdl, uint32_t *count, uint32_t *list,
                         cudaStream_t s)
{
    const size_t smem = thread_kernel_smem(qp.k) + (size_t)opt_smem_pad();
    if (smem > 48 * 1024)   // only the occupancy probe (smem_pad) ever exceeds the default limit
        PT_CUDA(cudaFuncSetAttribute(knn_thread_kernel<PT>,
                                     cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    unsigned blocks = (qp.m + T_THREADS - 1) / T_THREADS;
    if (qp.qlist) {
        // resident blocks per SM, asked once per shared-memory size (it depends on nothing else)
        static std::atomic<unsigned long long> cached{0};   // smem << 16 | blocks per SM
        unsigned long long c = cached.load();
        if (c >> 16 != smem) {
            int per_sm = 0;
            PT_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, knn_thread_kernel<PT>, T_THREADS, smem));
            c = (unsigned long long)smem << 16 | (unsigned long long)max(per_sm, 1);
            cached.store(c);
        }
        blocks = min(blocks, (unsigned)(c & 0xffffu) * (unsigned)sm_count);
    }
    PT_CUDA(launch_maybe_pdl(pdl, knn_thread_kernel<PT>, blocks, T_THREADS, smem, s, qp, count, list));
    count_launch();
    return PT_OK;
}

int debug_stats_n(unsigned long long *out, int n, int reset)
{
    if (n < 0) return PT_ERR_INVALID_ARG;
    for (int a = 0; a < n; ++a) out[a] = 0;
#ifdef PT_STATS
    PT_CUDA(cudaDeviceSynchronize());
    if (n > 0) PT_CUDA(cudaMemcpyFromSymbol(out, g_stats, sizeof(unsigned long long) * (size_t)min(n, PT_STATS_N)));
    if (reset) {
        unsigned long long z[PT_STATS_N] = {};
        PT_CUDA(cudaMemcpyToSymbol(g_stats, z, sizeof z));
    }
#else
    (void)reset;
#endif
    return PT_OK;
}

int debug_stats(unsigned long long *out16, int reset) { return debug_stats_n(out16, 16, reset); }

}  // namespace pt

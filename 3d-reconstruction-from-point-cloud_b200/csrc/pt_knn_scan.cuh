// pt_knn_scan.cuh -- variant 5 ("scan"): the thread kernel with the top-k kept as an UNSORTED
// set of slots and its maximum found by a short linear scan instead of a heap.
//
//   slot j:  key  = (fp32 bits of d2 rounded down, low 5 bits replaced by j)     4 bytes
//            pos  = position of the point in the sorted cloud                       4 bytes
//
// The keys of a sample sit in 128-bit shared-memory columns, so "which slot holds the k-th
// candidate" is k/4 conflict-free LDS.128 plus an integer max tree -- no dependent chain of
// shared-memory round trips like a sift-down, and about half its instructions.  Truncating a
// monotone key is still monotone: a strictly smaller truncated key is a strictly smaller d2, a
// strictly larger one is strictly larger.  EQUAL truncated keys (the key of a candidate against
// the maximum, or two slots sharing the maximum; 2^-18 relative, or true ties) are decided on
// the exact (d2, index) re-read from the cloud.  The winners' exact d2 / indices are re-read
// at the end and sorted by (d2, index), so every output is bit-identical to variant 2.
// State per sample at k = 16: 288 bytes (thread kernel: 384).
#pragma once

namespace pt {

constexpr int SCAN_SB = 5;                       // slot bits inside a key (k <= 32)
constexpr uint32_t SCAN_SM = (1u << SCAN_SB) - 1u;

#ifndef PT_SCAN_PREFETCH
#define PT_SCAN_PREFETCH 1
#endif
#ifndef PT_SCAN_MIN_BLOCKS
#define PT_SCAN_MIN_BLOCKS 20
#endif
template <typename PT>
__global__ void __launch_bounds__(T_THREADS, PT_SCAN_MIN_BLOCKS)
knn_scan_kernel(const QueryParams P, uint32_t *ovf_count, uint32_t *ovf_list)
{
    extern __shared__ __align__(16) unsigned char t_smem[];
    const int k = P.k;
    const unsigned tid = threadIdx.x;
    const int KG = (k + 3) >> 2, KP = KG * 4;                    // key groups of 4 slots
    uint32_t *pis = reinterpret_cast<uint32_t *>(t_smem) + tid;                                    // [KP] positions
    uint4 *kq = reinterpret_cast<uint4 *>(t_smem + 4 * T_THREADS * (size_t)KP) + tid;              // [KG] keys
    unsigned long long *pe = reinterpret_cast<unsigned long long *>(t_smem + 8 * T_THREADS * (size_t)KP) + tid;  // [TPD_CAP]
    uint32_t *pqk = reinterpret_cast<uint32_t *>(pe + TPD_CAP * T_THREADS - tid) + tid;            // [TPQ_CAP]
    uint32_t *pqw = pqk + TPQ_CAP * T_THREADS;                                                     // [TPQ_CAP]
    auto key_at = [&](int j) -> uint32_t & {
        return reinterpret_cast<uint32_t *>(&kq[(j >> 2) * T_THREADS])[j & 3];
    };

    // list mode (second stage behind the grid kernel): sample qlist[i], i < *qcount, blocks of
    // T_THREADS list entries grid-stride (the grid is sized to the resident blocks, launch_scan);
    // the list is read after the kernel that wrote it has completed (a programmatic dependent)
    pdl_wait();
    uint32_t m_eff = P.qlist ? min(*P.qcount, P.m) : P.m;
    if (P.qlist && m_eff < P.qlist_min) m_eff = 0;       // short lists are the warp kernel's
#pragma unroll 1
    for (uint32_t b0 = blockIdx.x * T_THREADS; b0 < m_eff; b0 += gridDim.x * T_THREADS) {
        for (int g = 0; g < KG; ++g) kq[g * T_THREADS] = make_uint4(0u, 0u, 0u, 0u);
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
        const float bound_r = __double2float_ru(r2);
        float bound = bound_r;

        int hn = 0;                      // slots in use
        uint32_t rtk = 0xffffffffu;      // truncated key (key >> 5) of the current k-th candidate ...
        int rslot = 0;                   // ... and its slot -- meaningful once hn == k
        Traverser<PT, T_THREADS> tr(P, pqk, pqw, qx, qy, qz, !done);

        // exact (d2, index) of an entry, re-read from the sorted cloud (rare: only on equal keys)
        auto exact_of = [&](uint32_t pos, double &d, int &idx) {
            double px, py, pz;
            PointLoad<PT>::load(P.pts, pos, px, py, pz, idx);
            d = dist2_exact(qx, qy, qz, px, py, pz);
        };
        // the slot of the current k-th candidate: maximum key; if a second slot shares its truncated
        // key (seen as a different winner when the slot bits are inverted) the tied slots are compared
        // on the exact (d2, index)
        auto find_root = [&]() {
            uint32_t M = 0, M2 = 0;
            for (int g = 0; g < KG; ++g) {
                const uint4 v = kq[g * T_THREADS];
                M = max(max(M, v.x), max(max(v.y, v.z), v.w));
                M2 = max(max(M2, v.x ^ SCAN_SM), max(max(v.y ^ SCAN_SM, v.z ^ SCAN_SM), v.w ^ SCAN_SM));
            }
            rslot = (int)(M & SCAN_SM);
            rtk = M >> SCAN_SB;
            if ((M2 ^ SCAN_SM) != M) {
                double bd;
                int bi;
                exact_of(pis[rslot * T_THREADS], bd, bi);
                for (int j = 0; j < k; ++j) {
                    if (j == (int)(M & SCAN_SM) || (key_at(j) >> SCAN_SB) != rtk) continue;
                    double cd;
                    int ci;
                    exact_of(pis[j * T_THREADS], cd, ci);
                    if (key_less(bd, bi, cd, ci)) { bd = cd; bi = ci; rslot = j; }
                }
            }
        };
        auto put = [&](int slot, unsigned long long e) {
            key_at(slot) = ((uint32_t)(e >> 32) & ~SCAN_SM) | (uint32_t)slot;
            pis[slot * T_THREADS] = (uint32_t)e;
        };

        for (;;) {
            const int leaf = tr.next_leaf(bound, hn < k, done);
            if (__all_sync(0xffffffffu, done)) break;

            // ---- leaf phase: every lane that holds a leaf scans it, 8 points per chunk -------------
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
                        const uint32_t cf = __float_as_uint(__double2float_rd(d));
                        if (pi < P.n && d <= r2 && (hn < k || (cf >> SCAN_SB) <= rtk)) {
                            pe[pend * T_THREADS] = ((unsigned long long)cf << 32) | pi;
                            ++pend;
                        }
                    }
                }
                while (__any_sync(0xffffffffu, pend > 0)) {
                    if (pend > 0) {
                        --pend;
                        const unsigned long long e = pe[pend * T_THREADS];
                        const uint32_t ctk = (uint32_t)(e >> 32) >> SCAN_SB;
                        if (hn < k) {
                            put(hn, e);
                            if (++hn == k) find_root();
                        } else if (ctk < rtk) {
                            put(rslot, e);
                            find_root();
                        } else if (ctk == rtk) {             // undecidable on truncated keys: exact compare
                            double cd, rd;
                            int ci, ri;
                            exact_of((uint32_t)e, cd, ci);
                            exact_of(pis[rslot * T_THREADS], rd, ri);
                            if (key_less(cd, ci, rd, ri)) {
                                put(rslot, e);
                                find_root();
                            }
                        }
                    }
                }
            }
            // smallest fp32 value that is certainly > the k-th exact d2 (its key is truncated)
            if (hn == k) {
                const bool first = bound == bound_r;
                bound = fminf(__uint_as_float((rtk + 1u) << SCAN_SB), bound_r);
                // the siblings queued during the first dive were pushed with an infinite bound:
                // most of them are dead now, which keeps a small queue sufficient
                if (first && bound < bound_r) tr.compact(bound);
            }
        }

        overflow = tr.proof_failed(bound);
#ifdef PT_STATS
        {
            unsigned v = (live && overflow) ? 1u : 0u, w = live ? 1u : 0u;
            for (int o = 16; o > 0; o >>= 1) { v += __shfl_xor_sync(0xffffffffu, v, o); w += __shfl_xor_sync(0xffffffffu, w, o); }
            if (tid == 0) { if (v) atomicAdd(&g_stats[8], (unsigned long long)v); atomicAdd(&g_stats[9], (unsigned long long)w); }
        }
#endif
        if (live && overflow) {
            uint32_t slot = atomicAdd(ovf_count, 1u);
            ovf_list[slot] = q;
        }
        // the lanes that emit; the others wait at the end of the block's turn, because the columns
        // below overlap their key and position columns
        const bool emit = live && !overflow;
        const unsigned emask = __ballot_sync(0xffffffffu, emit);
        if (emit) {
            // the winners' exact (d2, index) from the sorted cloud, then the common sort + output +
            // blend.  The 8-byte column hd[j] of a lane covers the 4-byte position columns 2j and 2j+1
            // of OTHER lanes (or the dead keys), so the whole warp converts slot j together, from the
            // last slot down: whatever a store overwrites was read in an earlier step, or -- slot 0 --
            // before the __syncwarp of this one.  The int column lives in the dead pending / queue
            // columns.
            double *hd = reinterpret_cast<double *>(t_smem) + tid;                                        // [k]
            int *hi = reinterpret_cast<int *>(t_smem + 8 * T_THREADS * (size_t)KP) + tid;                 // [k]
#if PT_SCAN_PREFETCH
            // the loop below waits for one point per step: start all the loads now
            for (int j = 0; j < hn; ++j)
                asm volatile("prefetch.global.L1 [%0];" ::"l"(reinterpret_cast<const PT *>(P.pts) + pis[j * T_THREADS]));
#endif
            for (int j = k - 1; j >= 0; --j) {
                double d = 0.0;
                int pidx = 0;
                if (j < hn) {
                    double px, py, pz;
                    PointLoad<PT>::load(P.pts, pis[j * T_THREADS], px, py, pz, pidx);
                    d = dist2_exact(qx, qy, qz, px, py, pz);
                }
                __syncwarp(emask);
                if (j < hn) {
                    hd[j * T_THREADS] = d;
                    hi[j * T_THREADS] = pidx;
                }
            }
            emit_sample<T_THREADS>(P, q, hd, hi, hn);
        }
        if (T_THREADS > 32) __syncthreads(); else __syncwarp();   // every column is free for the next turn
    }
}

static inline size_t scan_kernel_smem(int k)
{
    // positions + keys (8 B per padded slot) + pending [TPD_CAP] (8 B) + queue [TPQ_CAP] (8 B);
    // the epilogue's 8 B * k + 4 B * k columns fit (the ints go to the pending / queue columns)
    const size_t kp = (size_t)((k + 3) / 4) * 4;
    return (size_t)T_THREADS * (kp * 8 + (size_t)TPD_CAP * 8 + (size_t)TPQ_CAP * 8);
}

// A list-mode launch (qp.qlist) does not know the list's length on the host: its grid is the
// resident blocks, not one block per T_THREADS samples of qp.m; `pdl`: a programmatic dependent
// of the kernel that writes the list.
template <typename PT>
static int launch_scan(const QueryParams &qp, int sm_count, bool pdl, uint32_t *count, uint32_t *list,
                       cudaStream_t s)
{
    const size_t smem = scan_kernel_smem(qp.k) + (size_t)opt_smem_pad();
    if (smem > 48 * 1024)   // only the occupancy probe (smem_pad) ever exceeds the default limit
        PT_CUDA(cudaFuncSetAttribute(knn_scan_kernel<PT>,
                                     cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    unsigned blocks = (qp.m + T_THREADS - 1) / T_THREADS;
    if (qp.qlist) {
        // resident blocks per SM, asked once per shared-memory size (it depends on nothing else)
        static std::atomic<unsigned long long> cached{0};   // smem << 16 | blocks per SM
        unsigned long long c = cached.load();
        if (c >> 16 != smem) {
            int per_sm = 0;
            PT_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, knn_scan_kernel<PT>, T_THREADS, smem));
            c = (unsigned long long)smem << 16 | (unsigned long long)max(per_sm, 1);
            cached.store(c);
        }
        blocks = min(blocks, (unsigned)(c & 0xffffu) * (unsigned)sm_count);
    }
    PT_CUDA(launch_maybe_pdl(pdl, knn_scan_kernel<PT>, blocks, T_THREADS, smem, s, qp, count, list));
    count_launch();
    return PT_OK;
}

}  // namespace pt

// pt_knn_traverse.cuh -- the best-first traversal shared by the thread and the scan kernel
// (one thread per sample): a small priority queue in shared-memory columns plus the node being
// expanded in registers.
//
//   queue entry : key  = fp32 lower bound of the nearest UNVISITED child of a partially visited
//                        node, low 4 mantissa bits replaced by the node's 8-wide level (still a
//                        valid, slightly smaller bound);
//                 word = 8-bit mask of the unvisited children << 23 | node id.
//   expansion   : the 8 child boxes are fetched up front (16 independent 16-byte loads), tested
//                 with bounds rounded toward the safe side (src/Distance.h:27-57), the nearest
//                 child is followed directly while it is still the best candidate (no queue
//                 traffic) and the siblings are re-queued as ONE entry.
//   full queue  : first the entries beyond the bound are dropped (it only shrinks, so they are
//                 dead); if every entry is live the least promising one (largest key; in a
//                 min-heap it is among the leaves) is given up and the smallest key ever given up
//                 is remembered.  Nothing inside a dropped subtree is closer than its key, so the
//                 result is exact iff the final bound stays below that key (proof_failed());
//                 otherwise the sample is re-run by the warp kernel.  tests: test_tiny_queue_*.
#pragma once

namespace pt {

// -DPT_STATS: per-launch work counters (diagnosis builds only; pt_debug_stats reads them)
constexpr int PT_STATS_N = 32;   // counter words (pt_debug_stats reads the first 16, pt_debug_stats_n up to all)
#ifdef PT_STATS
__device__ unsigned long long g_stats[PT_STATS_N];
#define PT_STAT(slot, v) (st_[slot] += (v))
#else
#define PT_STAT(slot, v) ((void)0)
#endif
// slots: 0 expansions, 1 leaves, 2 pushes, 3 pops, 4 compactions, 5 heap inserts, 6 candidates
// parked, 7 warp rounds, 8 overflowed samples, 9 samples, 10 drain iterations (warp), 11 expand
// iterations (warp); 12-15 grid kernels (pt_knn_grid.cuh); 16-24 knn_grid_span_kernel: 16 parent
// look-ups, 17 bulk copies, 18 copies that continue another copy of the same half in the sorted
// cloud (what merging spans across parents would save), 19 warps, 20 / 21 sum / maximum of a
// warp's busy time (ns), 22 ~earliest warp start, 23 latest warp finish (%globaltimer), 24 halves
// redone by the whole warp

constexpr int T_LOG = 3;      // 8-wide levels of the box pyramid: binary levels 0, 3, 6, ...
#ifndef PT_TPQ_CAP
// queue entries per sample: 8 already works (a few fallbacks per million samples), 12 had none on
// any workload shape, and every 8 entries less is one more resident warp per SM
#define PT_TPQ_CAP 12
#endif
constexpr int TPQ_CAP = PT_TPQ_CAP;
#ifndef PT_T_PREFETCH
#define PT_T_PREFETCH 1       // L2-prefetch the chosen leaf while other lanes still traverse
#endif

template <typename PT, int STRIDE>
struct Traverser {
    const QueryParams &P;
    uint32_t *pqk, *pqw;          // queue columns of this sample (element e at [e * STRIDE])
    float qdn[3], qup[3];         // the query bracketed in fp32 (round down / round up)
    int pq_n = 0, qcap;
    uint32_t lost = 0xffffffffu;  // smallest key of an entry that had to be given up
    bool cur_valid;               // the node being expanded (not in the queue)
    int cur_tl;
    uint32_t cur_id = 0, cur_mask = 0xffu;
#ifdef PT_STATS
    unsigned *st_;
#endif

    __device__ __forceinline__ Traverser(const QueryParams &p, uint32_t *keys, uint32_t *words,
                                         double qx, double qy, double qz, bool valid)
        : P(p), pqk(keys), pqw(words), cur_valid(valid), cur_tl(p.t_levels)
    {
        qdn[0] = __double2float_rd(qx); qdn[1] = __double2float_rd(qy); qdn[2] = __double2float_rd(qz);
        qup[0] = __double2float_ru(qx); qup[1] = __double2float_ru(qy); qup[2] = __double2float_ru(qz);
        qcap = min(max(p.pq_cap, 2), TPQ_CAP);     // runtime cap <= layout (tests shrink it)
    }

    __device__ __forceinline__ void sift_up(int i, uint32_t key, uint32_t word)
    {
        while (i > 0) {
            const int p = (i - 1) >> 1;
            const uint32_t pk = pqk[p * STRIDE];
            if (pk <= key) break;
            pqk[i * STRIDE] = pk;
            pqw[i * STRIDE] = pqw[p * STRIDE];
            i = p;
        }
        pqk[i * STRIDE] = key;
        pqw[i * STRIDE] = word;
    }

    // drop the entries that lie beyond the bound and rebuild the heap in place
    __device__ __forceinline__ void compact(float bound)
    {
        int live = 0;
#pragma unroll 1
        for (int e = 0; e < pq_n; ++e) {
            const uint32_t ek = pqk[e * STRIDE], ew = pqw[e * STRIDE];
            if (__uint_as_float(ek & ~0xfu) <= bound) sift_up(live++, ek, ew);
        }
        pq_n = live;
    }

    __device__ __forceinline__ void push(uint32_t key, uint32_t word, float bound)
    {
        PT_STAT(2, 1);
        if (pq_n == qcap) {
            PT_STAT(4, 1);
            compact(bound);
            if (pq_n == qcap) {            // all live: give up the largest key (see the header)
                int mi = qcap / 2;
                uint32_t mk = pqk[mi * STRIDE];
#pragma unroll 1
                for (int e = qcap / 2 + 1; e < qcap; ++e) {
                    const uint32_t ek = pqk[e * STRIDE];
                    if (ek > mk) { mk = ek; mi = e; }
                }
                if (key >= mk) { lost = min(lost, key); return; }
                lost = min(lost, mk);
                sift_up(mi, key, word);
                return;
            }
        }
        sift_up(pq_n++, key, word);
    }

    __device__ __forceinline__ void pop(uint32_t &key, uint32_t &word)
    {
        key = pqk[0];
        word = pqw[0];
        const int n = --pq_n;
        if (n == 0) return;
        const uint32_t lk = pqk[n * STRIDE], lw = pqw[n * STRIDE];
        int i = 0;
        for (;;) {
            int c = 2 * i + 1;
            if (c >= n) break;
            uint32_t ck = pqk[c * STRIDE];
            if (c + 1 < n) {
                const uint32_t ck2 = pqk[(c + 1) * STRIDE];
                if (ck2 < ck) { ck = ck2; ++c; }
            }
            if (ck >= lk) break;
            pqk[i * STRIDE] = ck;
            pqw[i * STRIDE] = pqw[c * STRIDE];
            i = c;
        }
        pqk[i * STRIDE] = lk;
        pqw[i * STRIDE] = lw;
    }

    // Advances the search to the next leaf worth scanning under `bound` and returns it, or
    // returns -1 with done = true when nothing closer than the bound is left.  `filling`: the
    // sample holds fewer than k candidates (plain dive: every leaf helps).
    __device__ __forceinline__ int next_leaf(float bound, bool filling, bool &done)
    {
        int leaf = -1;
        while (!done && leaf < 0) {
            if (!cur_valid) {
                if (pq_n == 0) { done = true; break; }
                uint32_t key, word;
                pop(key, word);
                PT_STAT(3, 1);
                if (__uint_as_float(key & ~0xfu) > bound) { done = true; break; }   // rest is farther
                cur_tl = (int)(key & 0xfu);
                cur_id = word & 0x7fffffu;
                cur_mask = word >> 23;
            }
            cur_valid = false;
            PT_STAT(0, 1);
            if (threadIdx.x % 32 == (unsigned)(__ffs(__activemask()) - 1)) PT_STAT(11, 1);
            // expand: test the unvisited children (8-wide level cur_tl - 1)
            const int pl = (cur_tl - 1) * T_LOG;
            const uint32_t cnt = P.pyr.count[pl];
            const Box *boxes = P.pyr.level[pl];
            float best = INFINITY, second = INFINITY;
            int best_c = -1;
            uint32_t rem = 0;
            Box cb[8];   // children past the end of the level are clamped and masked out below
#pragma unroll
            for (int c = 0; c < 8; ++c) cb[c] = load_box(boxes + min(cur_id * 8 + c, cnt - 1));
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                if (((cur_mask >> c) & 1u) && cur_id * 8 + c < cnt) {
                    const float lb = box_lower_bound(qdn, qup, cb[c]);
                    if (lb <= bound) {
                        rem |= 1u << c;
                        if (lb < best) { second = best; best = lb; best_c = c; }
                        else second = fminf(second, lb);
                    }
                }
            }
            if (best_c < 0) continue;
            rem &= ~(1u << best_c);
            if (rem) push((__float_as_uint(second) & ~0xfu) | (uint32_t)cur_tl, (rem << 23) | cur_id, bound);
            const uint32_t child = cur_id * 8 + (uint32_t)best_c;
            if (cur_tl == 1) {
                leaf = (int)child;
#if PT_T_PREFETCH
                const char *lp = reinterpret_cast<const char *>(P.pts) + (size_t)child * LEAF * sizeof(PT);
#pragma unroll
                for (int l = 0; l < (int)(LEAF * sizeof(PT) / 128); ++l)
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(lp + 128 * l));
#endif
            } else {
                const bool dive = filling || pq_n == 0 || best <= __uint_as_float(pqk[0] & ~0xfu);
                if (dive) { cur_valid = true; cur_tl -= 1; cur_id = child; cur_mask = 0xffu; }
                else push((__float_as_uint(best) & ~0xfu) | (uint32_t)(cur_tl - 1), (0xffu << 23) | child, bound);
            }
        }
        return leaf;
    }

    // a dropped queue entry matters only if its subtree could still reach inside the final bound
    __device__ __forceinline__ bool proof_failed(float bound) const
    {
        return lost != 0xffffffffu && __uint_as_float(lost & ~0xfu) <= bound;
    }
};

}  // namespace pt

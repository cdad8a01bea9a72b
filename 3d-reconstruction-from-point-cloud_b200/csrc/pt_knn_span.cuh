// pt_knn_span.cuh -- knn_grid_span_kernel: the two-samples-per-warp grid kernel of
// pt_knn_grid.cuh (knn_grid_pair_kernel) with fewer and larger memory requests per sample.
//
//   * one look-up per PARENT cell: the 3^3 block around a sample's cell touches exactly 2 parents
//     per axis, so sub-lanes 0-7 of each half probe one of the 8 parent buckets each (one round);
//     from the bucket's octant -> curve-rank map the lane finds which children lie in the block
//     and cuts the parent's run into <= 4 spans of consecutive curve ranks (a rank with no points
//     never breaks a span);
//   * one cp.async.bulk per span instead of one per cell;
//   * the winners' attributes are read from the curve-ordered copy (pt_index::attrs_curve): the
//     winners sit in a few adjacent cells, so their 16-byte records share DRAM lines, where the
//     original order scatters them over 16 unrelated lines.  A per-half table of span heads in
//     shared memory turns a winner's slot into its sorted position without a global access.
//
// The staged candidate SET is the pair kernel's (only the slot order differs), and the selection
// never depends on slot order (a tie of truncated keys goes to the exact (d2, index) selection),
// so `total`, the go / redo decisions and every output are those of knn_grid_pair_kernel.
#pragma once

namespace pt {

constexpr int SPAN_MAX = 32;          // spans per half: 8 parents x <= 4
// 7 blocks x 4 warps per SM at 72 registers (measured at cfg2: 6 blocks at 80 registers 0.357 ms,
// 7 blocks 0.342 ms, 8 blocks at 64 registers 0.351 ms; DESIGN.md section 4)
#ifndef PT_SPAN_MIN_BLOCKS
#define PT_SPAN_MIN_BLOCKS 7
#endif

// Bucket of parent cell (px, py, pz), probed like grid_lookup.  false: the parent holds no points.
__device__ __forceinline__ bool grid_parent_lookup(const GridBucket *buckets, uint32_t cap, uint32_t px,
                                                   uint32_t py, uint32_t pz, uint32_t &start, uint32_t &perm,
                                                   uint4 &cum)
{
    const unsigned long long pkey = (unsigned long long)px | ((unsigned long long)py << 21) |
                                    ((unsigned long long)pz << 42);
    const uint32_t ngroups = cap >> 1;
    uint32_t g = __umulhi(grid_hash_q(pkey), ngroups);
    for (;;) {
        const unsigned long long *p = reinterpret_cast<const unsigned long long *>(buckets + 2 * (size_t)g);
        const unsigned long long k0 = __ldg(p), k1 = __ldg(p + 4);
        if (k0 == pkey || k1 == pkey) {
            const unsigned long long *b = k0 == pkey ? p : p + 4;
            const uint2 a = __ldg(reinterpret_cast<const uint2 *>(b + 1));     // start, perm
            start = a.x;
            perm = a.y;
            cum = __ldg(reinterpret_cast<const uint4 *>(b + 2));
            return true;
        }
        if (k0 == ~0ull || k1 == ~0ull) return false;
        if (++g == ngroups) g = 0;
    }
}

// Points of the parent's children of curve rank < r (r = 0..8), from the bucket's cum[] fields.
__device__ __forceinline__ uint32_t span_cum_at(const uint4 &c, unsigned r)
{
    const uint32_t w = r < 4 ? (r < 2 ? c.x : c.y) : (r < 6 ? c.z : c.w);
    const uint32_t v = (w >> (16u * (r & 1u))) & 0xffffu;
    return r == 0 ? 0u : (r == 8 ? (c.x & 0xffffu) : v);
}

// Calls f(first, count) for every span of the parent's run, in curve order: maximal groups of
// the ranks in `inr` (the children inside the block) not separated by a rank of `brk` (children
// outside the block that hold points).  first is relative to the parent's start.
template <typename F>
__device__ __forceinline__ void for_each_span(uint32_t inr, uint32_t brk, const uint4 &cum, F f)
{
    while (inr) {
        const unsigned r0 = __ffs(inr) - 1;
        const uint32_t b = brk & (0xffu << r0);
        const unsigned r1 = b ? __ffs(b) - 1 : 8u;
        const uint32_t beg = span_cum_at(cum, r0);
        f(beg, span_cum_at(cum, r1) - beg);
        inr &= ~((1u << r1) - 1u);
    }
}

// Look-ups of the 3^3 block around cell c: sub-lane j < 8 of each half takes parent j of the
// block's 2 x 2 x 2 parents.  Along an axis the block's cells c - 1 .. c + 1 lie in parents
// ((c + 1) >> 1) - 1 and (c + 1) >> 1; child bit b of parent q is cell 2q + b, inside the block iff
// it is one of c - 1 .. c + 1 and below ncell (the unsigned compare also rejects "negative"
// cells).  Gives the lane's parent start, the curve ranks of its children inside the block (inr)
// and of its occupied children outside it (brk), its cum[] fields, and dense when the parent has
// too many points for them.
__device__ __forceinline__ void span_parent(const GridTable &T, const uint32_t c[3], uint32_t ncell, unsigned sl,
                                            bool look, uint32_t &pstart, uint32_t &inr, uint32_t &brk, uint4 &cum,
                                            bool &dense)
{
    pstart = 0;
    inr = 0;
    brk = 0;
    cum = make_uint4(0u, 0u, 0u, 0u);
    dense = false;
    if (look && sl < 8u) {
        uint32_t pq[3], oct = 0xffu;
#pragma unroll
        for (int ax = 0; ax < 3; ++ax) {
            pq[ax] = ((c[ax] + 1u) >> 1) - 1u + ((sl >> ax) & 1u);
            const uint32_t x0 = 2u * pq[ax], x1 = x0 + 1u;
            const bool b0 = x0 - c[ax] + 1u < 3u && x0 < ncell, b1 = x1 - c[ax] + 1u < 3u && x1 < ncell;
            // octants o with bit `ax` of o = 0 (b0) or 1 (b1)
            const uint32_t m1 = ax == 0 ? 0xaau : (ax == 1 ? 0xccu : 0xf0u);
            oct &= (b0 ? (~m1 & 0xffu) : 0u) | (b1 ? m1 : 0u);
        }
        uint32_t perm = 0;
#ifdef PT_STATS
        if (oct) atomicAdd(&g_stats[16], 1ull);
#endif
        if (oct && grid_parent_lookup(T.buckets, T.cap, pq[0], pq[1], pq[2], pstart, perm, cum)) {
            const uint32_t occ = perm >> 24, om = oct & occ;
            if (om && (cum.x & 0xffffu) == 0xffffu) dense = true;
            else if (om) {
#pragma unroll
                for (int o = 0; o < 8; ++o) {
                    const uint32_t rb = 1u << ((perm >> (3 * o)) & 7u);
                    if ((om >> o) & 1u) inr |= rb;
                    else if ((occ >> o) & 1u) brk |= rb;
                }
            }
        }
    }
}

// Spans << 24 | points of this lane's parent (mine_v), its inclusive sum over the half's parents
// (incl); returns the half's sum.  Every lane of the warp calls it.
__device__ __forceinline__ uint32_t span_scan(uint32_t inr, uint32_t brk, const uint4 &cum, unsigned sl,
                                              unsigned hbase, uint32_t &mine_v, uint32_t &incl)
{
    mine_v = 0;
    for_each_span(inr, brk, cum, [&](uint32_t, uint32_t n) { mine_v += (1u << 24) + n; });
    incl = mine_v;
#pragma unroll
    for (int o = 1; o < 8; o <<= 1) {
        const uint32_t y = __shfl_up_sync(0xffffffffu, incl, o);
        if (sl >= (unsigned)o) incl += y;
    }
    return __shfl_sync(0xffffffffu, incl, (int)(hbase | 7u));
}

// ---- block runs (pt_index::blk_mem, built by build_blocks) ---------------------------------------
// For every occupied cell c of one table level, one run holds the records the span kernel stages
// for a sample in c, in its slot order, followed by its span heads (padded to an even count).
// The table slot gives the run's place and size, so one probe and two bulk copies stage a sample.
__device__ __forceinline__ unsigned long long block_key(const uint32_t c[3])
{
    return (unsigned long long)c[0] | ((unsigned long long)c[1] << 21) | ((unsigned long long)c[2] << 42);
}
__device__ __forceinline__ uint32_t block_heads_pad(uint32_t nspan) { return (nspan + 1u) & ~1u; }

// The slot of cell `key`: its meta (BLOCK_MISS when the cell is empty) and, for a stageable
// run, the run's offset in 16-byte units.  Four slots are probed at a time (one aligned 64-byte
// group = one DRAM fetch); a group is filled in slot order, so an empty slot ends the search.
__device__ __forceinline__ uint32_t block_lookup(const BlockSlot *tab, uint32_t cap, unsigned long long key,
                                                 uint32_t &off)
{
    const uint32_t ngroups = cap >> 2;
    uint32_t g = __umulhi(grid_hash_q(key), ngroups);
    for (;;) {
        const uint4 *p = reinterpret_cast<const uint4 *>(tab + 4 * (size_t)g);
        uint4 v[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) v[i] = __ldg(p + i);
        bool open = false, found = false;
        uint32_t hit_off = 0, hit_meta = BLOCK_MISS;
#pragma unroll
        for (int i = 0; i < 4; ++i) {              // selects, not an indexed (local-memory) array
            const unsigned long long ki = (unsigned long long)v[i].x | ((unsigned long long)v[i].y << 32);
            const bool m = ki == key;
            hit_off = m ? v[i].z : hit_off;
            hit_meta = m ? v[i].w : hit_meta;
            found |= m;
            open |= ki == ~0ull;
        }
        if (found) { off = hit_off; return hit_meta; }
        if (open) return BLOCK_MISS;
        if (++g == ngroups) g = 0;
    }
}

// One pass of build_blocks over the buckets of table T: a half-warp per bucket, its children in
// octant order, each through the span kernel's own look-ups and span order.  COUNT: the run
// units (16 bytes) of the bucket's children into units[bucket].  Otherwise: each child's run at
// runs + off[bucket] + (units of the bucket's earlier children), and its slot in tab.
template <bool COUNT>
__global__ void __launch_bounds__(256)
block_run_kernel(const GridTable T, unsigned long long *units, const unsigned long long *off, const PointF *pts,
                 uint4 *runs, BlockSlot *tab, uint32_t tab_cap)
{
    __shared__ uint2 s_heads[256 / 16][SPAN_MAX];
    const unsigned lane = threadIdx.x & 31u, sl = lane & 15u, hbase = lane & 16u;
    uint2 *heads = s_heads[threadIdx.x >> 4];
    const uint32_t b = (blockIdx.x * blockDim.x + threadIdx.x) >> 4;
    unsigned long long key = ~0ull;
    uint32_t perm = 0;
    if (b < T.cap) {
        key = T.buckets[b].key;
        perm = T.buckets[b].perm;
    }
    const uint32_t occ = key != ~0ull ? perm >> 24 : 0u;
    const uint32_t ncell = 1u << T.level;
    const uint32_t par[3] = {(uint32_t)(key & 0x1fffffu), (uint32_t)((key >> 21) & 0x1fffffu),
                             (uint32_t)((key >> 42) & 0x1fffffu)};
    unsigned long long u_sum = 0;
    for (int o = 0; o < 8; ++o) {                // all lanes: the look-ups end in warp shuffles
        const bool look = (occ >> o) & 1u;
        const uint32_t c[3] = {2u * par[0] + (o & 1u), 2u * par[1] + ((o >> 1) & 1u), 2u * par[2] + ((o >> 2) & 1u)};
        uint32_t pstart, inr, brk, mine_v, incl;
        uint4 cum;
        bool dense;
        span_parent(T, c, ncell, sl, look, pstart, inr, brk, cum, dense);
        const uint32_t hsum = span_scan(inr, brk, cum, sl, hbase, mine_v, incl);
        const uint32_t total = hsum & 0xffffffu, nspan = hsum >> 24;
        const bool dense_h = ((__ballot_sync(0xffffffffu, dense) >> hbase) & 0xffffu) != 0u;
        // the span kernel stages such a block only when it holds <= PAIR_CAP records and no dense parent
        const bool ok = look && !dense_h && total <= (uint32_t)PAIR_CAP;
        const uint32_t u = ok ? total + block_heads_pad(nspan) / 2u : 0u;
        if (!COUNT && look) {
            uint4 *run = runs + off[b] + u_sum;
            if (ok) {
                uint32_t slot = (incl - mine_v) & 0xffffffu, e = (incl - mine_v) >> 24;
                for_each_span(inr, brk, cum, [&](uint32_t first, uint32_t n) {
                    heads[e] = make_uint2(slot, pstart + first);
                    slot += n;
                    ++e;
                });
            }
            __syncwarp(0xffffu << hbase);
            if (ok) {
                for (uint32_t j = sl; j < total; j += 16u) {     // last head with first slot <= j
                    uint32_t lo = 0, n = nspan;
                    while (n > 1u) {
                        const uint32_t h = n >> 1;
                        if (heads[lo + h].x <= j) lo += h;
                        n -= h;
                    }
                    run[j] = __ldg(reinterpret_cast<const uint4 *>(pts + heads[lo].y + (j - heads[lo].x)));
                }
                uint2 *hout = reinterpret_cast<uint2 *>(run + total);
                for (uint32_t e = sl; e < block_heads_pad(nspan); e += 16u)
                    hout[e] = e < nspan ? heads[e] : make_uint2(0u, 0u);
            }
            if (sl == 0u) {
                const unsigned long long ck = block_key(c);
                uint32_t s = 4u * __umulhi(grid_hash_q(ck), tab_cap >> 2);
                for (;;) {                           // the order block_lookup probes in
                    BlockSlot *S = tab + s;
                    if (atomicCAS(&S->key, ~0ull, ck) == ~0ull) {
                        S->off = ok ? (uint32_t)(off[b] + u_sum) : 0u;
                        S->meta = ok ? total | (nspan << 16) : BLOCK_MISS;
                        break;
                    }
                    if (++s == tab_cap) s = 0;
                }
            }
            __syncwarp(0xffffu << hbase);            // the heads are free for the next child
        }
        u_sum += u;
    }
    if (COUNT && sl == 0u && b < T.cap) units[b] = u_sum;
}

// Outputs of both halves: pair_emit (pt_knn_grid.cuh) with the winner's attribute record passed
// in.  Same arithmetic, in the same order (frozen blend, DESIGN.md section 5).
__device__ __forceinline__ void span_emit(const QueryParams &P, uint32_t s, bool em, uint32_t mine, double d,
                                          int li, const AttrRaw &at, unsigned lane, PointF *wcand)
{
    const unsigned sl = lane & 15u, hbase = lane & 16u;
    const int k = P.k;
    const bool has = em && mine != GKEY_NONE;
    const int gid = has ? (P.ids ? __ldg(P.ids + li) : li) : -1;
    const bool want_blend = P.rgba_out || P.normal_out;
    if (em && sl < (unsigned)k) {
        const size_t o = (size_t)s * k + sl;
        if (P.idx_out) P.idx_out[o] = gid;
        if (P.d2_out) P.d2_out[o] = d;
        if (P.cand_out) store_cand(P.cand_out + o, d, gid, at);
    }
    if (!want_blend) return;
    uint8_t *ro = P.rgba_out ? P.rgba_out + 4 * (size_t)s : nullptr;
    float *no = P.normal_out ? P.normal_out + 3 * (size_t)s : nullptr;
    const int cnt = __popc((__ballot_sync(0xffffffffu, has) >> hbase) & 0xffffu);
    if (em && cnt == 0 && sl == 0u) store_empty_blend(ro, no);
    const bool bl = em && cnt > 0;
    if (!__any_sync(0xffffffffu, bl)) return;
    const int mode = __shfl_sync(0xffffffffu, d, (int)hbase) == 0.0 ? 1 : 0;
    const double w = has ? (mode ? (d == 0.0 ? 1.0 : 0.0) : __ddiv_rn(1.0, d)) : 0.0;
    double *tile = reinterpret_cast<double *>(wcand);
    __syncwarp();                               // every lane has read its winner's record
    tile[0 * 32 + lane] = w;
    tile[1 * 32 + lane] = __dmul_rn(w, (double)(at.rgba & 0xffu));
    tile[2 * 32 + lane] = __dmul_rn(w, (double)((at.rgba >> 8) & 0xffu));
    tile[3 * 32 + lane] = __dmul_rn(w, (double)((at.rgba >> 16) & 0xffu));
    tile[4 * 32 + lane] = __dmul_rn(w, (double)at.nx);
    tile[5 * 32 + lane] = __dmul_rn(w, (double)at.ny);
    tile[6 * 32 + lane] = __dmul_rn(w, (double)at.nz);
    __syncwarp();
    double acc = 0.0;
    if (bl && sl < 7u) {
        const double *row = tile + sl * 32u + hbase;
        int j = 0;
#pragma unroll 1
        for (; j + 4 <= cnt; j += 4) {
            acc = __dadd_rn(acc, row[j]);
            acc = __dadd_rn(acc, row[j + 1]);
            acc = __dadd_rn(acc, row[j + 2]);
            acc = __dadd_rn(acc, row[j + 3]);
        }
#pragma unroll 1
        for (; j < cnt; ++j) acc = __dadd_rn(acc, row[j]);
    }
    double s0 = __shfl_sync(0xffffffffu, acc, (int)hbase);
    const uint32_t c0 = __shfl_sync(0xffffffffu, at.rgba, (int)hbase);
    const float n0x = __shfl_sync(0xffffffffu, at.nx, (int)hbase), n0y = __shfl_sync(0xffffffffu, at.ny, (int)hbase),
                n0z = __shfl_sync(0xffffffffu, at.nz, (int)hbase);
    if (bl && !(s0 > 0.0 && s0 < INFINITY)) {   // overflowed weights: nearest neighbour only
        const double v[7] = {1.0, (double)(c0 & 0xffu), (double)((c0 >> 8) & 0xffu), (double)((c0 >> 16) & 0xffu),
                             (double)n0x, (double)n0y, (double)n0z};
        acc = 0.0;
#pragma unroll
        for (int a = 0; a < 7; ++a) if (sl == (unsigned)a) acc = v[a];
        s0 = 1.0;
    }
    const double s4 = __shfl_sync(0xffffffffu, acc, (int)hbase + 4), s5 = __shfl_sync(0xffffffffu, acc, (int)hbase + 5),
                 s6 = __shfl_sync(0xffffffffu, acc, (int)hbase + 6);
    const double len = __dsqrt_rn(__dadd_rn(__dadd_rn(__dmul_rn(s4, s4), __dmul_rn(s5, s5)), __dmul_rn(s6, s6)));
    const double den = sl < 4u ? s0 : len;
    const double quo = __ddiv_rn(acc, den);
    const int ci = min(max(__double2int_rz(quo), 0), 255);
    const int cr = __shfl_sync(0xffffffffu, ci, (int)hbase + 1), cg = __shfl_sync(0xffffffffu, ci, (int)hbase + 2),
              cb = __shfl_sync(0xffffffffu, ci, (int)hbase + 3);
    if (bl && sl == 0u && ro) *reinterpret_cast<uchar4 *>(ro) = make_uchar4((unsigned char)cr, (unsigned char)cg, (unsigned char)cb, 255);
    if (bl && sl >= 4u && sl < 7u && no)
        no[sl - 4u] = (len > 0.0 && len < INFINITY) ? __double2float_rn(quo) : 0.0f;
}

// claim (not null): after its first pair a warp claims its next pair with one atomicAdd (pairs
// n_warps.. in claiming order) instead of taking every n_warps-th pair, so that the persistent
// launch ends with the last pair rather than with the warp whose pairs happened to be slowest.
// Which warp answers a pair never changes the pair's answer.
// BLOCK: a sample stages the block run of its cell (P.grid.blk) instead of the eight parents' spans;
// the staged records and heads are the same, so is everything from the selection on.
template <bool BLOCK>
__device__ __forceinline__ void span_body(const QueryParams &P, uint32_t *ovf_count, uint32_t *ovf_list,
                                          uint32_t *claim)
{
    extern __shared__ __align__(128) unsigned char g_smem[];
    const unsigned lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const unsigned sl = lane & 15u, hbase = lane & 16u;
    PointF *wcand = reinterpret_cast<PointF *>(g_smem) + (size_t)wib * (2 * PAIR_CAP);
    PointF *cand = wcand + (hbase ? PAIR_CAP : 0);
    // span heads of this half, in slot order: (first slot, sorted position of that slot)
    uint2 *heads = reinterpret_cast<uint2 *>(g_smem + sizeof(PointF) * 2 * PAIR_CAP * GRID_WARPS) +
                   (size_t)wib * (2 * SPAN_MAX) + (hbase ? SPAN_MAX : 0);
    unsigned long long *bars = reinterpret_cast<unsigned long long *>(
        g_smem + sizeof(PointF) * 2 * PAIR_CAP * GRID_WARPS + sizeof(uint2) * 2 * SPAN_MAX * GRID_WARPS);
    const uint32_t bar = smem_u32(bars + wib);
    // every block is resident from the start (launch_grid_span): the hand-over kernels behind this
    // one may launch now, they only take the space that finished blocks give up and wait for the
    // whole grid before they read the list
    pdl_launch_dependents();
    if (lane == 0) mbar_init(bar, 1);
    __syncwarp();
    uint32_t phase = 0;
    const int k = P.k;
    const GridParams &G = P.grid;
    const uint32_t n_warps = gridDim.x * GRID_WARPS, n_pairs = (P.m + 1u) >> 1;
    const PointF *pts = reinterpret_cast<const PointF *>(P.pts);
    uint32_t p = blockIdx.x * GRID_WARPS + wib;
    if (p >= n_pairs) return;
#ifdef PT_STATS
    unsigned long long t_start;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_start));
#endif
    while (p < n_pairs) {
        // the warp's next pair, claimed now so that the atomic's latency hides behind this pair
        uint32_t nxt = p + n_warps;
        if (claim && lane == 0) nxt = n_warps + atomicAdd(claim, 1u);
        // a pair whose second sample does not exist answers the first one twice and emits it once
        const bool valid = 2u * p + (lane >> 4) < P.m;
        const uint32_t s = min(2u * p + (lane >> 4), P.m - 1u);
        const double qx = __ldg(P.queries + 3 * (size_t)s), qy = __ldg(P.queries + 3 * (size_t)s + 1),
                     qz = __ldg(P.queries + 3 * (size_t)s + 2);
        if (!claim && lane == 0 && nxt < n_pairs)    // the next pair's coordinates: towards L2 meanwhile
            asm volatile("prefetch.global.L2 [%0];" ::"l"(P.queries + 6 * (size_t)nxt));
        const double r2 = P.r2_per_query ? __ldg(P.r2_per_query + s) : P.r2;
        const bool dead = valid && !(r2 >= 0.0);
        const bool look = valid && !dead;
        // ---- the sample's cell and its distance to the faces of the 3^3 block (as the pair kernel) --
        const GridTable &T = G.tab[G.att_tab[0]];
        const int sh = 21 - T.level;
        const uint32_t ncell = 1u << T.level;
        const float S = (float)(1u << sh), above = 2.0f * S;
        const double qv[3] = {qx, qy, qz};
        uint32_t c[3];
        float gl = INFINITY;
#pragma unroll
        for (int ax = 0; ax < 3; ++ax) {
            const double t = (qv[ax] - G.lo[ax]) * G.inv_cell21;
            const uint32_t c21 = min(__double2uint_rz(t), 2097151u);
            c[ax] = c21 >> sh;
            const double f = t - (double)(c[ax] << sh);
            const float dl = __fadd_rd(__double2float_rd(f), S);
            const float du = __fsub_rd(above, __double2float_ru(f));
            gl = fminf(gl, c[ax] > 1u ? dl : INFINITY);
            gl = fminf(gl, c[ax] + 2u < ncell ? du : INFINITY);
        }
        const double slack = G.slack + 1.8e-15 * (fabs(qx) + fabs(qy) + fabs(qz));
        const double g = (double)gl * G.cell21 - slack;
        const double g2 = g > 0.0 ? __dmul_rd(g, g) : 0.0;
        uint32_t total, nspan;
        bool dense_h;
        // block runs: the slot of the sample's cell (sub-lane 0); an empty cell is a miss like a
        // block that cannot be staged, and goes to the whole-warp redo
        uint32_t boff = 0, bmeta = BLOCK_MISS;
        // span staging: sub-lane j < 8 takes parent j of the block's 2 x 2 x 2 parents
        uint32_t pstart, inr, brk, mine_v, incl;
        uint4 cum;
        if constexpr (BLOCK) {
            if (look && sl == 0u) bmeta = block_lookup(G.blk, G.blk_cap, block_key(c), boff);
            bmeta = __shfl_sync(0xffffffffu, bmeta, (int)hbase);
            boff = __shfl_sync(0xffffffffu, boff, (int)hbase);
            total = bmeta & 0xffffu;
            nspan = (bmeta >> 16) & 0xffu;
            dense_h = (bmeta & BLOCK_MISS) != 0u;
        } else {
            bool dense;
            span_parent(T, c, ncell, sl, look, pstart, inr, brk, cum, dense);
            const uint32_t hsum = span_scan(inr, brk, cum, sl, hbase, mine_v, incl);
            total = hsum & 0xffffffu;
            nspan = hsum >> 24;
            dense_h = ((__ballot_sync(0xffffffffu, dense) >> hbase) & 0xffffu) != 0u;
        }
        const bool go = look && !dense_h && total <= (uint32_t)PAIR_CAP && (total >= (uint32_t)k || r2 <= g2);
        const uint32_t tot = go ? total : 0u;
        const uint32_t tA = __shfl_sync(0xffffffffu, tot, 0), tB = __shfl_sync(0xffffffffu, tot, 16);
#ifdef PT_STATS
        if (sl == 0 && valid) { atomicAdd(&g_stats[12], 1ull); atomicAdd(&g_stats[13], (unsigned long long)tot); }
#endif
        // ---- stage both halves' spans; one mbarrier ----------------------------------------------
        if (tA + tB > 0u) {
            fence_proxy_async();
            __syncwarp();
            if constexpr (BLOCK) {
                // records and heads of the run: 16 bytes per record, 8 per (padded) head
                const uint32_t hb = go ? block_heads_pad(nspan) * (uint32_t)sizeof(uint2) : 0u;
                const uint32_t hbA = __shfl_sync(0xffffffffu, hb, 0), hbB = __shfl_sync(0xffffffffu, hb, 16);
                if (lane == 0) mbar_arrive_expect(bar, (tA + tB) * (uint32_t)sizeof(PointF) + hbA + hbB);
                __syncwarp();
                if (go && sl == 0u) {
                    const uint4 *run = G.blk_runs + boff;
                    bulk_g2s(smem_u32(cand), run, total * (uint32_t)sizeof(PointF), bar);
                    bulk_g2s(smem_u32(heads), run + total, hb, bar);
                }
            } else {
                if (lane == 0) mbar_arrive_expect(bar, (tA + tB) * (uint32_t)sizeof(PointF));
                __syncwarp();
                if (go) {
                    uint32_t slot = (incl - mine_v) & 0xffffffu, e = (incl - mine_v) >> 24;
                    for_each_span(inr, brk, cum, [&](uint32_t first, uint32_t n) {
                        bulk_g2s(smem_u32(cand + slot), pts + pstart + first, n * (uint32_t)sizeof(PointF), bar);
                        heads[e] = make_uint2(slot, pstart + first);
                        slot += n;
                        ++e;
                    });
                }
            }
            __syncwarp();                           // the span heads are visible to the whole half
#ifdef PT_STATS
            if (!BLOCK && go) {   // spans whose sorted start is the sorted end of another span of the half
                uint32_t hits = 0;
                for (uint32_t a = sl; a < nspan; a += 16u)
                    for (uint32_t b = 0; b < nspan; ++b) {
                        const uint32_t nb = (b + 1u < nspan ? heads[b + 1u].x : tot) - heads[b].x;
                        hits += heads[b].y + nb == heads[a].y ? 1u : 0u;
                    }
                if (hits) atomicAdd(&g_stats[18], (unsigned long long)hits);
                if (sl == 0) atomicAdd(&g_stats[17], (unsigned long long)nspan);
            }
#endif
            mbar_wait(bar, phase);
            phase ^= 1u;
        }
        // ---- select (the pair kernel's selection, unchanged) ---------------------------------------
        uint32_t mine = GKEY_NONE;
        bool amb = false;
        const uint32_t tmax = max(tA, tB);
        if (tmax == 0u) { /* nothing staged (unused rows, empty blocks): no key to select */ }
        else if (tmax <= 32u) pair_select<2>(cand, tot, qx, qy, qz, r2, k, sl, hbase != 0u, mine, amb);
        else if (tmax <= 64u) pair_select<4>(cand, tot, qx, qy, qz, r2, k, sl, hbase != 0u, mine, amb);
#if PT_PAIR_CAP > 128
        else if (tmax <= 128u) pair_select<8>(cand, tot, qx, qy, qz, r2, k, sl, hbase != 0u, mine, amb);
        else pair_select<12>(cand, tot, qx, qy, qz, r2, k, sl, hbase != 0u, mine, amb);
#else
        else pair_select<8>(cand, tot, qx, qy, qz, r2, k, sl, hbase != 0u, mine, amb);
#endif
        const uint32_t amb_all = __ballot_sync(0xffffffffu, amb);
        if (amb_all) {
            const bool act = ((amb_all >> hbase) & 0xffffu) != 0u;
#ifdef PT_STATS
            if (sl == 0 && act) atomicAdd(&g_stats[14], 1ull);
#endif
            pair_select_exact(cand, act, tot, qx, qy, qz, r2, k, lane, mine);
        }
        double d = INFINITY;
        int li = IDX_NONE;
        if (mine != GKEY_NONE) {
            double px, py, pz;
            GridRec<PointF>::load(cand, mine & 0xffu, px, py, pz, li);
            d = dist2_exact(qx, qy, qz, px, py, pz);
        }
        const double kth = __shfl_sync(0xffffffffu, d, (int)hbase + k - 1);   // +inf while the list is short
        const bool done = dead || (go && fmin(kth, r2) <= g2);
        // ---- the winner's attributes: slot -> sorted position through the span heads -----------------
        AttrRaw at{0.f, 0.f, 0.f, 0u};
        if (done && mine != GKEY_NONE && (P.rgba_out || P.normal_out || P.cand_out) && P.attrs_curve) {
            const uint32_t j = mine & 0xffu;
            uint32_t lo = 0, n = nspan;              // last head with first slot <= j (heads[0] is slot 0)
            while (n > 1u) {
                const uint32_t h = n >> 1;
                if (heads[lo + h].x <= j) lo += h;
                n -= h;
            }
            const uint2 hd = heads[lo];
            at = load_attr(P.attrs_curve + hd.y + (j - hd.x));
        }
        span_emit(P, s, done, mine, d, li, at, lane, wcand);
        // ---- halves this attempt could not finish: the whole warp, the whole schedule ----------------
        const uint32_t redo = __ballot_sync(0xffffffffu, valid && !done);
#ifdef PT_STATS
        if (lane == 0 && redo) atomicAdd(&g_stats[24], (unsigned long long)__popc(redo & 0x10001u));
#endif
        if (redo & 1u) {
            const double fx = __shfl_sync(0xffffffffu, qx, 0), fy = __shfl_sync(0xffffffffu, qy, 0),
                         fz = __shfl_sync(0xffffffffu, qz, 0);
            grid_sample<PointF, true>(P, 2u * p, fx, fy, fz, lane, wcand, bar, phase, ovf_count, ovf_list);
        }
        if (redo & 0x10000u) {
            const double fx = __shfl_sync(0xffffffffu, qx, 16), fy = __shfl_sync(0xffffffffu, qy, 16),
                         fz = __shfl_sync(0xffffffffu, qz, 16);
            grid_sample<PointF, true>(P, 2u * p + 1u, fx, fy, fz, lane, wcand, bar, phase, ovf_count, ovf_list);
        }
        if (claim && lane == 0 && nxt < n_pairs)
            asm volatile("prefetch.global.L2 [%0];" ::"l"(P.queries + 6 * (size_t)nxt));
        p = __shfl_sync(0xffffffffu, nxt, 0);
    }
#ifdef PT_STATS
    unsigned long long t_end;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_end));
    if (lane == 0) {
        atomicAdd(&g_stats[19], 1ull);
        atomicAdd(&g_stats[20], t_end - t_start);
        atomicMax(&g_stats[21], t_end - t_start);
        atomicMax(&g_stats[22], ~t_start);
        atomicMax(&g_stats[23], t_end);
    }
#endif
}

__global__ void __launch_bounds__(GRID_WARPS * 32, PT_SPAN_MIN_BLOCKS)
knn_grid_span_kernel(const QueryParams P, uint32_t *ovf_count, uint32_t *ovf_list, uint32_t *claim)
{
    span_body<false>(P, ovf_count, ovf_list, claim);
}

__global__ void __launch_bounds__(GRID_WARPS * 32, PT_SPAN_MIN_BLOCKS)
knn_grid_block_kernel(const QueryParams P, uint32_t *ovf_count, uint32_t *ovf_list, uint32_t *claim)
{
    span_body<true>(P, ovf_count, ovf_list, claim);
}

// The pair kernel's conditions (launch_grid) plus the curve-ordered attributes wherever the
// launch reads attributes.
template <typename PT>
static bool grid_span_applies(const QueryParams &qp)
{
    const bool want_attr = qp.rgba_out || qp.normal_out || qp.cand_out;
    return std::is_same<PT, PointF>::value && opt_grid_tma() != 0 && opt_grid_span() != 0 && opt_grid_pair() != 0 &&
           qp.k <= 16 && qp.grid.n_attempts > 0 && qp.grid.att_rc[0] == 1 &&
           (opt_grid_pair() == 2 || qp.grid.expect_cand <= 0.74f * (float)PAIR_CAP) &&
           (qp.attrs_curve != nullptr || qp.attrs == nullptr || !want_attr);
}

// Under grid_span_applies: whether the launch stages block runs -- the index has them for the level
// of the launch's first attempt.
static bool grid_block_applies(const QueryParams &qp)
{
    return opt_grid_block() != 0 && qp.grid.blk != nullptr && qp.grid.tab[qp.grid.att_tab[0]].level == qp.grid.blk_level;
}

static int launch_grid_span(const QueryParams &qp, bool block, int sm_count, uint32_t *count, uint32_t *list,
                            uint32_t *claim, cudaStream_t s)
{
    const auto kernel = block ? knn_grid_block_kernel : knn_grid_span_kernel;
    const size_t smem = (sizeof(PointF) * 2 * PAIR_CAP + sizeof(uint2) * 2 * SPAN_MAX + 8) * GRID_WARPS;
    if (smem > 48 * 1024)
        PT_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 0;
    PT_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, GRID_WARPS * 32, smem));
    if (per_sm < 1) per_sm = 1;
    const unsigned want = ((qp.m + 1u) / 2u + GRID_WARPS - 1) / GRID_WARPS;
    const unsigned resident = (unsigned)(sm_count * per_sm);
    const unsigned blocks = want < resident ? want : resident;
    // pairs claimed once a warp has more than two of them (cfg2: 24, cfg5: 120; measured at cfg2
    // 0.342 -> 0.311 ms, cfg5 7.00 -> 6.49 ms); at cfg1 (1.2 pairs per warp) the static stride is
    // 1 us faster (DESIGN.md section 4)
    const bool use_claim = opt_grid_claim() != 0 && (qp.m + 1u) / 2u > 2u * blocks * GRID_WARPS;
    kernel<<<blocks, GRID_WARPS * 32, smem, s>>>(qp, count, list, use_claim ? claim : nullptr);
    count_launch();
    PT_CUDA(cudaGetLastError());
    return PT_OK;
}

}  // namespace pt

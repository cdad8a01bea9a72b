/*
 * pt_orient_oracle.c -- CPU statement of the normal orientation (DESIGN.md section 8, "Normal
 * orientation"), which csrc/pt_orient.cu must equal bit for bit.
 *
 * TEST INFRASTRUCTURE ONLY.  Built with -ffp-contract=off (no FMA), fp64 throughout, every operation
 * rounded on its own.  It works in the plainest way: every edge of the graph, qsort by (w, lo, hi),
 * Kruskal with union-find, then a breadth-first walk of each tree from its root.  The neighbour lists
 * come from the caller (oracle.pto_normals.neighbours: ascending (d2, id), padded with -1).
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

typedef struct { double x, y, z; } d3;
typedef struct { double w; int32_t lo, hi; int neg; } edge;

static double dot3(d3 a, d3 b) { return (a.x * b.x + a.y * b.y) + a.z * b.z; }
static int usable3(d3 a) { return isfinite(a.x) && isfinite(a.y) && isfinite(a.z) && dot3(a, a) > 0.0; }

static int edge_cmp(const void *pa, const void *pb)
{
    const edge *a = pa, *b = pb;
    if (a->w != b->w) return a->w < b->w ? -1 : 1;
    if (a->lo != b->lo) return a->lo < b->lo ? -1 : 1;
    return (a->hi > b->hi) - (a->hi < b->hi);
}

static int64_t find(int64_t *uf, int64_t x)
{
    while (uf[x] != x) {
        uf[x] = uf[uf[x]];
        x = uf[x];
    }
    return x;
}

/* the list of i, cut at its first -1 */
static int list_len(const int32_t *idx, int64_t n, int k, int64_t i)
{
    int c = 0;
    while (c < k && idx[i * k + c] >= 0 && idx[i * k + c] < n) ++c;
    return c;
}

/* xyz: n x 3 stored positions, nrm: n x 3 stored fp32 normals, idx: n x k lists, view: 3 doubles or
 * NULL.  Outputs: normal_out n x 3, root_out n, parent_out n (the forest: parent point id, -1 at roots
 * and at points that do not take part; may be NULL), counts (oriented, flipped, components, edges).
 * Returns 0, -1 on bad arguments or when memory runs out. */
int pto_orient_normals(const double *xyz, const float *nrm, int64_t n, const int32_t *idx, int k, const double *view,
                       float *normal_out, int32_t *root_out, int32_t *parent_out, int64_t *counts)
{
    if (n < 0 || (n && (!xyz || !nrm || !idx)) || !normal_out || !root_out || !counts || k < 1) return -1;
    d3 *nh = malloc(sizeof(d3) * (size_t)(n ? n : 1));
    char *part = malloc((size_t)(n ? n : 1));
    edge *e = malloc(sizeof(edge) * (size_t)(n * k > 0 ? n * k : 1));
    int64_t *uf = malloc(sizeof(int64_t) * (size_t)(n ? n : 1));
    int64_t *deg = calloc((size_t)n + 1, sizeof(int64_t));
    int32_t *adj = malloc(sizeof(int32_t) * (size_t)(2 * n + 1));
    char *adj_neg = malloc((size_t)(2 * n + 1));
    int32_t *top = malloc(sizeof(int32_t) * (size_t)(n ? n : 1));
    int32_t *queue = malloc(sizeof(int32_t) * (size_t)(n ? n : 1));
    signed char *sigma = malloc((size_t)(n ? n : 1));
    int32_t *par = malloc(sizeof(int32_t) * (size_t)(n ? n : 1));
    edge *fe = malloc(sizeof(edge) * (size_t)(n ? n : 1));
    int rc = -1;
    if (!nh || !part || !e || !uf || !deg || !adj || !adj_neg || !top || !queue || !sigma || !par || !fe) goto out;
    memset(counts, 0, 4 * sizeof(int64_t));

    for (int64_t i = 0; i < n; ++i) {
        const d3 m = {(double)nrm[3 * i], (double)nrm[3 * i + 1], (double)nrm[3 * i + 2]};
        part[i] = (char)usable3(m);
        if (part[i]) {
            const double l = sqrt(dot3(m, m));
            nh[i] = (d3){m.x / l, m.y / l, m.z / l};
            ++counts[0];
        }
        uf[i] = i;
        sigma[i] = 0;
        par[i] = -1;
    }
    /* the union of the lists, each pair once */
    int64_t ne = 0;
    for (int64_t i = 0; i < n; ++i) {
        if (!part[i]) continue;
        const int li = list_len(idx, n, k, i);
        for (int s = 0; s < li; ++s) {
            const int32_t j = idx[i * k + s];
            if (j == i || !part[j]) continue;
            int keep = i < j;
            if (!keep) {
                const int lj = list_len(idx, n, k, j);
                keep = 1;
                for (int t = 0; t < lj; ++t)
                    if (idx[(int64_t)j * k + t] == i) keep = 0;
            }
            if (!keep) continue;
            const double d = dot3(nh[i], nh[j]);
            double w = 1.0 - fabs(d);
            if (w < 0.0) w = 0.0;
            e[ne++] = (edge){w, (int32_t)(i < j ? i : j), (int32_t)(i < j ? j : i), d < 0.0};
        }
    }
    counts[3] = ne;
    qsort(e, (size_t)ne, sizeof(edge), edge_cmp);
    /* Kruskal */
    int64_t nf = 0;
    for (int64_t a = 0; a < ne; ++a) {
        const int64_t ru = find(uf, e[a].lo), rv = find(uf, e[a].hi);
        if (ru == rv) continue;
        uf[ru] = rv;
        fe[nf++] = e[a];
        ++deg[e[a].lo];
        ++deg[e[a].hi];
    }
    /* the forest as adjacency lists */
    int64_t *first = deg;
    int64_t acc = 0;
    for (int64_t i = 0; i <= n; ++i) {
        const int64_t c = first[i];
        first[i] = acc;
        acc += c;
    }
    for (int64_t a = 0; a < nf; ++a) {
        adj[first[fe[a].lo]] = fe[a].hi; adj_neg[first[fe[a].lo]++] = (char)fe[a].neg;
        adj[first[fe[a].hi]] = fe[a].lo; adj_neg[first[fe[a].hi]++] = (char)fe[a].neg;
    }
    for (int64_t i = n; i > 0; --i) first[i] = first[i - 1];
    first[0] = 0;
    /* roots: the largest z of each component, the lowest id on ties */
    for (int64_t i = 0; i < n; ++i) top[i] = -1;
    for (int64_t i = 0; i < n; ++i) {
        if (!part[i]) continue;
        const int64_t c = find(uf, i);
        if (top[c] < 0 || xyz[3 * i + 2] > xyz[3 * (int64_t)top[c] + 2]) top[c] = (int32_t)i;
    }
    for (int64_t i = 0; i < n; ++i) root_out[i] = part[i] ? top[find(uf, i)] : -1;
    /* the root's sign, then breadth first along the forest */
    for (int64_t r = 0; r < n; ++r) {
        if (!part[r] || root_out[r] != r) continue;
        ++counts[2];
        const d3 nr = nh[r];
        int neg;
        if (view) {
            const d3 w = {view[0] - xyz[3 * r], view[1] - xyz[3 * r + 1], view[2] - xyz[3 * r + 2]};
            neg = dot3(nr, w) < 0.0;
        } else if (nr.z != 0.0) {
            neg = nr.z < 0.0;
        } else {
            const double ax = fabs(nr.x), ay = fabs(nr.y), az = fabs(nr.z);
            neg = (ax >= ay && ax >= az) ? nr.x < 0.0 : (ay >= az ? nr.y < 0.0 : nr.z < 0.0);
        }
        sigma[r] = neg ? -1 : 1;
        int64_t head = 0, tail = 0;
        queue[tail++] = (int32_t)r;
        while (head < tail) {
            const int32_t p = queue[head++];
            for (int64_t a = first[p]; a < first[p + 1]; ++a) {
                const int32_t c = adj[a];
                if (sigma[c] != 0) continue;
                sigma[c] = adj_neg[a] ? (signed char)-sigma[p] : sigma[p];
                par[c] = p;
                queue[tail++] = c;
            }
        }
    }
    for (int64_t i = 0; i < n; ++i) {
        float x = nrm[3 * i], y = nrm[3 * i + 1], z = nrm[3 * i + 2];
        if (part[i] && sigma[i] < 0) {
            x = -x; y = -y; z = -z;
            ++counts[1];
        }
        normal_out[3 * i] = x;
        normal_out[3 * i + 1] = y;
        normal_out[3 * i + 2] = z;
        if (parent_out) parent_out[i] = par[i];
    }
    rc = 0;
out:
    free(nh); free(part); free(e); free(uf); free(deg); free(adj); free(adj_neg);
    free(top); free(queue); free(sigma); free(par); free(fe);
    return rc;
}

// pt_bake.cuh -- the per-texel bake (pt_texture.cu) in the pieces that pt_texture_bake_height and
// the sharded bake (pt_sharded.cu) both run, on the internal side of the C ABI.
//
//   bake_prepare   upload, texel raster, sample positions and owner faces, vertex frames
//   answer         one index: bake_answer_rows over every sample; a sharded cloud:
//                  bake_partition routes the samples to their slabs, each slab answers its rows
//                  with bake_answer_rows on its own device, and the results are scattered back
//   bake_finish    composition, tangent maps, height range + encoding, padding, copies out
#pragma once

#include <vector>

#include "pt_index.cuh"

namespace pt {

// Samples per launch of the query + height kernel when the neighbour lists (heights) or the
// distances (ghost-zone check) are kept: 4 k and 8 k bytes per sample.
constexpr uint32_t HEIGHT_CHUNK = 1u << 22;
// slabs a sample can be routed to (pt_sharded_opts.n_devices)
constexpr int BAKE_MAX_SLABS = 64;

struct BakeMesh {
    const double  *v;          // n_vertices rows of `stride` doubles: x, y, z, u, v, ...
    int            stride;
    uint32_t       n_vertices;
    const int32_t *faces;
    uint32_t       n_faces;
    int            res;
};
constexpr int BAKE_ROW = 8;    // mesh and frame rows of the bake: 8 doubles

// Everything one bake keeps on its home device between the pieces.  Samples are in ascending
// texel order: d_texels, d_q (xyz), d_sface (owner face), d_rgba, d_normal.
struct BakeJob {
    cudaStream_t s = nullptr;
    int res = 0;
    size_t n_vertices = 0, count = 0;
    bool heights = false;
    BakeMesh M{};
    void *d_raw = nullptr;
    double *d_rows = nullptr, *d_q = nullptr, *d_frames = nullptr, *d_range = nullptr;
    int32_t *d_faces = nullptr, *d_sface = nullptr;
    uint32_t *d_texels = nullptr;
    uint8_t *d_rgba = nullptr, *d_bgra = nullptr, *d_nbgra = nullptr, *d_tbgra = nullptr;
    float *d_normal = nullptr, *d_nf = nullptr, *d_tnf = nullptr, *d_vt = nullptr, *d_height = nullptr;
    uint16_t *d_h16 = nullptr;
    unsigned long long *d_empty = nullptr;
    cudaEvent_t ev[4]{};
    std::vector<cudaEvent_t> marks;   // around each query chunk of a single-index bake with heights
};

// The argument rules of pt_texture_bake_height that do not concern the index: PT_OK or its error.
int bake_check_args(const void *vertices, size_t n_vertices, const int32_t *faces, size_t n_faces, int k,
                    int resolution, const pt_bake_outputs &o, const pt_bake_height *height);
// On the current device, asynchronous on s apart from the texel count: everything before the search.
int bake_prepare(BakeJob &J, cudaStream_t s, const void *vertices, size_t n_vertices, const int32_t *faces,
                 size_t n_faces, int resolution, const pt_bake_outputs &o, const pt_bake_height *hb);

// Ghost-zone check of a slab's answers (launch_ghost_check): device boxes and flag.
struct BakeGhost {
    const double *boxes;
    int n_ranks, self;
    double halo;
    uint32_t *flag;
};
// k-NN + blend of m sample rows (xyz, texel, owner face) on index ix, on ix's device, in chunks of
// HEIGHT_CHUNK when heights or the ghost check are on.  Neighbour ids are the index's own (qp.ids
// is not used), so a slab index's records give the heights.  M and frames live on ix's device.
// height (may be null): by_sample ? m floats in row order : the res x res image (by texel).
// marks (may be null): events around each query chunk.
int bake_answer_rows(pt_index *ix, const BakeMesh &M, const double *frames, const double *xyz,
                     const uint32_t *texels, const int32_t *sample_faces, size_t m, int k, double radius,
                     const BakeGhost *ghost, uint8_t *rgba, float *normal, float *height, bool by_sample,
                     std::vector<cudaEvent_t> *marks, cudaStream_t s);
// Stable partition of the samples by slab (the number of the n_slabs - 1 ascending host `cuts`
// c with !(x < c)); a sample with a NaN component goes nowhere.  Row j of the output is sample
// sel[j]; slab r has rows starts[r] .. starts[r + 1] - 1 (host, n_slabs + 1 entries), in ascending
// sample order.  faces / pface may be null.  Synchronises s.
int bake_partition(const double *xyz, const uint32_t *texels, const int32_t *faces, size_t count,
                   const double *cuts, int n_slabs, int32_t *sel, double *pxyz, uint32_t *ptex, int32_t *pface,
                   size_t *starts, cudaStream_t s);
// Composition, tangent maps, heights' range and codes, padding, copies to the host; synchronises.
int bake_finish(BakeJob &J, int pad, const pt_bake_outputs &o, pt_bake_height *hb, pt_bake_stats *st);
void bake_release(BakeJob &J);

}  // namespace pt

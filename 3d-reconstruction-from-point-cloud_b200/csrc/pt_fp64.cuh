// pt_fp64.cuh -- device helpers of the fp64 definitions that are stated operation by operation
// (the bakes in pt_texture.cu, normal estimation in pt_normals.cu): every operation rounded on its
// own (no contraction, no rsqrt), so the CPU oracles built with -ffp-contract=off equal them bit for
// bit.  a.b = (a.x b.x + a.y b.y) + a.z b.z; "usable" = all components finite and a.a > 0;
// normalising divides each component by sqrt(a.a).
#pragma once

#include "pt_common.cuh"

namespace pt {

struct D3 { double x, y, z; };

__device__ __forceinline__ D3 d3_add(D3 a, D3 b) { return {__dadd_rn(a.x, b.x), __dadd_rn(a.y, b.y), __dadd_rn(a.z, b.z)}; }
__device__ __forceinline__ D3 d3_sub(D3 a, D3 b) { return {__dsub_rn(a.x, b.x), __dsub_rn(a.y, b.y), __dsub_rn(a.z, b.z)}; }
__device__ __forceinline__ D3 d3_scale(double s, D3 a) { return {__dmul_rn(s, a.x), __dmul_rn(s, a.y), __dmul_rn(s, a.z)}; }
__device__ __forceinline__ double d3_dot(D3 a, D3 b)
{
    return __dadd_rn(__dadd_rn(__dmul_rn(a.x, b.x), __dmul_rn(a.y, b.y)), __dmul_rn(a.z, b.z));
}
__device__ __forceinline__ D3 d3_cross(D3 a, D3 b)
{
    return {__dsub_rn(__dmul_rn(a.y, b.z), __dmul_rn(a.z, b.y)), __dsub_rn(__dmul_rn(a.z, b.x), __dmul_rn(a.x, b.z)),
            __dsub_rn(__dmul_rn(a.x, b.y), __dmul_rn(a.y, b.x))};
}
__device__ __forceinline__ bool d3_finite(D3 a) { return isfinite(a.x) && isfinite(a.y) && isfinite(a.z); }
__device__ __forceinline__ bool d3_usable(D3 a) { return d3_finite(a) && d3_dot(a, a) > 0.0; }
__device__ __forceinline__ D3 d3_normalise(D3 a)
{
    const double l = __dsqrt_rn(d3_dot(a, a));
    return {__ddiv_rn(a.x, l), __ddiv_rn(a.y, l), __ddiv_rn(a.z, l)};
}
__device__ __forceinline__ D3 d3_load(const double *p) { return {p[0], p[1], p[2]}; }

__device__ __forceinline__ double shfl_d(double v, int src) { return __shfl_sync(0xffffffffu, v, src); }

// where the position of cloud point `id` (original index) comes from
template <typename PT> struct PosSorted {      // an index: sorted records + inverse permutation
    const PT *pts;
    const uint32_t *inv;
    __device__ __forceinline__ void get(int id, double x[3]) const
    {
        const PT rec = pts[inv[id]];
        x[0] = (double)rec.x; x[1] = (double)rec.y; x[2] = (double)rec.z;
    }
};

}  // namespace pt

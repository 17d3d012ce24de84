// vec3.cuh -- the reference's 3-D point helpers (point.py:25-45) in IEEE fp64 with its operation order: correctly
// rounded sqrt and division, explicit _rn intrinsics so that nothing is contracted into FMAs.  Shared by the 3-D
// FABRIK kernels (fabrik_generic_ikine_kernel in fabrik.cu, fabrik_chain_kernel in fabrik_chain.cu).
#pragma once
#include <cuda_runtime.h>

struct Vec3 {
    double x, y, z;
};

// get_distance_between(a, b) = sqrt((a.x - b.x)^2 + (a.y - b.y)^2 + (a.z - b.z)^2), summed left to right
__device__ __forceinline__ double dist3(const Vec3 &a, const Vec3 &b)
{
    const double dx = __dsub_rn(a.x, b.x), dy = __dsub_rn(a.y, b.y), dz = __dsub_rn(a.z, b.z);
    return __dsqrt_rn(__dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz)));
}

// get_point_between(s, e, L) = s + (L / |s - e|) * (e - s); NaN when the distance is 0
__device__ __forceinline__ Vec3 point_between3(const Vec3 &s, const Vec3 &e, double L)
{
    const double t = __ddiv_rn(L, dist3(s, e));
    Vec3 o;
    o.x = __dadd_rn(s.x, __dmul_rn(t, __dsub_rn(e.x, s.x)));
    o.y = __dadd_rn(s.y, __dmul_rn(t, __dsub_rn(e.y, s.y)));
    o.z = __dadd_rn(s.z, __dmul_rn(t, __dsub_rn(e.z, s.z)));
    return o;
}

// fk_device.cuh -- the DH forward-kinematics position (reference forward.py:62-94) as inline device code.
// Used by the batched FK kernel (fk.cu, K3) and by the solvers' fused error epilogues (fabrik.cu, mlp*.cu), so
// that ||FK(angles) - target|| costs no second pass over HBM (SURVEY 8 a6).
#pragma once
#include "ikb_common.cuh"

// The angle guard of forward.py:23-25 rejects |theta| > 2 pi, compared in fp64.  (float)(2 pi) = 6.2831855f lies ABOVE
// 2 pi, so comparing a float angle with it would accept float32(2 pi), which the reference (and fk_transforms_kernel,
// which widens to double) rejects.  The float guard compares with the largest float below 2 pi instead: for a float
// theta, |theta| > 6.2831850f  <=>  |(double)theta| > 2 pi.
#define IKB_TWO_PI_F32 6.28318500518798828125f
template <typename Real>
__device__ __forceinline__ Real ikb_two_pi();
template <>
__device__ __forceinline__ float ikb_two_pi<float>() { return IKB_TWO_PI_F32; }
template <>
__device__ __forceinline__ double ikb_two_pi<double>() { return 6.283185307179586; }

// sin/cos for |x| <= 2 pi (larger angles are rejected by the guard of forward.py:23-25 anyway):
// two-term Cody-Waite reduction by pi/2 (|k| <= 4, exact products) + the cephes single-precision
// kernels on [-pi/4, pi/4]; max error ~1.2e-7.  libdevice's sincosf carries a Payne-Hanek slow path whose
// integer instructions made the fp32 FK kernel instruction-bound instead of HBM-bound.
__device__ __forceinline__ void ikb_sincos(float x, float *s, float *c)
{
    // k = rint(x 2/pi) through the 1.5 * 2^23 trick: the sum's low mantissa bits ARE k (two's complement), so neither
    // a round nor a float-to-int conversion (both quarter-rate XU instructions) is needed; |x| <= 2 pi keeps |k| <= 4
    const float t = fmaf(x, 0.63661977236758134f, 12582912.0f);
    const int q = __float_as_int(t);
    const float k = t - 12582912.0f;
    float r = fmaf(k, -1.57079625129699707031f, x);
    r = fmaf(k, -7.54978941586159635335e-8f, r);
    const float r2 = r * r;
    float sp = fmaf(r2, -1.9515295891e-4f, 8.3321608736e-3f);
    sp = fmaf(sp, r2, -1.6666654611e-1f);
    sp = fmaf(sp * r2, r, r);
    float cp = fmaf(r2, 2.443315711809948e-5f, -1.388731625493765e-3f);
    cp = fmaf(cp, r2, 4.166664568298827e-2f);
    cp = fmaf(cp * r2, r2, fmaf(r2, -0.5f, 1.0f));
    const float ss = (q & 1) ? cp : sp, cc = (q & 1) ? sp : cp;
    *s = (q & 2) ? -ss : ss;
    *c = ((q + 1) & 2) ? -cc : cc;
}
__device__ __forceinline__ void ikb_sincos(double x, double *s, double *c) { sincos(x, s, c); }

// ---- two angles at a time on the packed fp32 pipe (sm_100: FFMA2 / FMUL2 / FADD2 = fma.rn.f32x2 ...) -----------------
// Same operations in the same order as ikb_sincos(float), every one correctly rounded, so the results are bit-identical
// to two scalar calls; what changes is the instruction count (15 packed + 12 select instructions for two angles instead
// of 2 x 23), which is what bounds K3 (fk.cu) once the loads are vectorised.
typedef unsigned long long ikb_f32x2;
__device__ __forceinline__ ikb_f32x2 ikb_pack2(float lo, float hi)
{
    ikb_f32x2 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void ikb_unpack2(ikb_f32x2 v, float &lo, float &hi)
{
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ ikb_f32x2 ikb_dup2(float x) { return ikb_pack2(x, x); }
__device__ __forceinline__ ikb_f32x2 ikb_fma2(ikb_f32x2 a, ikb_f32x2 b, ikb_f32x2 c)
{
    ikb_f32x2 r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
    return r;
}
__device__ __forceinline__ ikb_f32x2 ikb_mul2(ikb_f32x2 a, ikb_f32x2 b)
{
    ikb_f32x2 r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ ikb_f32x2 ikb_add2(ikb_f32x2 a, ikb_f32x2 b)
{
    ikb_f32x2 r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}

__device__ __forceinline__ void ikb_sincos2(float x0, float x1, float &s0, float &c0, float &s1, float &c1)
{
    const ikb_f32x2 X = ikb_pack2(x0, x1);
    const ikb_f32x2 T = ikb_fma2(X, ikb_dup2(0.63661977236758134f), ikb_dup2(12582912.0f));
    float t0, t1;
    ikb_unpack2(T, t0, t1);
    const int q0 = __float_as_int(t0), q1 = __float_as_int(t1);
    const ikb_f32x2 K = ikb_add2(T, ikb_dup2(-12582912.0f));
    ikb_f32x2 R = ikb_fma2(K, ikb_dup2(-1.57079625129699707031f), X);
    R = ikb_fma2(K, ikb_dup2(-7.54978941586159635335e-8f), R);
    const ikb_f32x2 R2 = ikb_mul2(R, R);
    ikb_f32x2 SP = ikb_fma2(R2, ikb_dup2(-1.9515295891e-4f), ikb_dup2(8.3321608736e-3f));
    SP = ikb_fma2(SP, R2, ikb_dup2(-1.6666654611e-1f));
    SP = ikb_fma2(ikb_mul2(SP, R2), R, R);
    ikb_f32x2 CP = ikb_fma2(R2, ikb_dup2(2.443315711809948e-5f), ikb_dup2(-1.388731625493765e-3f));
    CP = ikb_fma2(CP, R2, ikb_dup2(4.166664568298827e-2f));
    CP = ikb_fma2(ikb_mul2(CP, R2), R2, ikb_fma2(R2, ikb_dup2(-0.5f), ikb_dup2(1.0f)));
    float sp0, sp1, cp0, cp1;
    ikb_unpack2(SP, sp0, sp1);
    ikb_unpack2(CP, cp0, cp1);
    // quadrant: odd k swaps sine and cosine, bit 1 of k (k + 1 for the cosine) flips the sign -- the flip as an XOR of
    // the sign bit (bit 1 shifted to bit 31), which is what `(q & 2) ? -v : v` means for every v including 0 and NaN
    const float ss0 = (q0 & 1) ? cp0 : sp0, cc0 = (q0 & 1) ? sp0 : cp0;
    const float ss1 = (q1 & 1) ? cp1 : sp1, cc1 = (q1 & 1) ? sp1 : cp1;
    s0 = __int_as_float(__float_as_int(ss0) ^ ((q0 << 30) & 0x80000000));
    c0 = __int_as_float(__float_as_int(cc0) ^ (((q0 + 1) << 30) & 0x80000000));
    s1 = __int_as_float(__float_as_int(ss1) ^ ((q1 << 30) & 0x80000000));
    c1 = __int_as_float(__float_as_int(cc1) ^ (((q1 + 1) << 30) & 0x80000000));
}

// Closed form for arms whose joints 2..4 have alpha == 0 (see fk_position): the constants are passed as scalars so
// that the solvers' out-of-line epilogue helpers can call it without the robot block.
template <typename Real>
__device__ __forceinline__ void fk_planar_tail_position(const Real s[4], const Real c[4], Real a0, Real a1, Real a2,
                                                        Real a3, Real eps0, Real w, Real ca, Real sa, Real &px, Real &py,
                                                        Real &pz)
{
    Real cs = c[1], sn = s[1];
    Real u = a1 * cs, v = a1 * sn;
    {
        const Real cn = cs * c[2] - sn * s[2];
        sn = sn * c[2] + cs * s[2];
        cs = cn;
        u += a2 * cs;
        v += a2 * sn;
    }
    {
        const Real cn = cs * c[3] - sn * s[3];
        sn = sn * c[3] + cs * s[3];
        cs = cn;
        u += a3 * cs;
        v += a3 * sn;
    }
    const Real lx = a0 + u, ly = v * ca - w * sa, lz = eps0 + v * sa + w * ca;
    px = c[0] * lx - s[0] * ly;
    py = s[0] * lx + c[0] * ly;
    pz = lz;
}

// ||FK(th) - target|| through the closed form, callable with plain scalars (no robot block): NaN when an angle is
// outside [-2 pi, 2 pi] (forward.py:23-25), exactly as ikb_fk_error / K3 report such rows.
template <typename Real>
__device__ __forceinline__ Real ikb_fk_error_planar_tail(const Real th[4], Real tx, Real ty, Real tz, Real a0, Real a1,
                                                         Real a2, Real a3, Real eps0, Real w, Real ca, Real sa)
{
    const Real TWO_PI = ikb_two_pi<Real>();
    bool ok = true;
    Real s[4], c[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        ok &= !(fabs(th[i]) > TWO_PI);
        ikb_sincos(th[i], &s[i], &c[i]);
    }
    Real px, py, pz;
    fk_planar_tail_position<Real>(s, c, a0, a1, a2, a3, eps0, w, ca, sa, px, py, pz);
    const Real dx = px - tx, dy = py - ty, dz = pz - tz;
    const Real err = sqrt(dx * dx + dy * dy + dz * dz);
    return ok ? err : (Real)__int_as_float(0x7fc00000);
}

template <typename Real>
__device__ __forceinline__ const Real *fk_constants(const IkbRobot &rc);
template <>
__device__ __forceinline__ const double *fk_constants<double>(const IkbRobot &rc) { return rc.fkc; }
template <>
__device__ __forceinline__ const float *fk_constants<float>(const IkbRobot &rc) { return rc.fkc_f; }

// Position-only DH chain.  General form: p += R [a c, a s, eps]; R = R Rz(theta) Rx(alpha).
// When joints 2..4 have alpha == 0 (rc.fk_planar_tail: every arm of the reference's family, robot.py:40) the
// tail is planar in joint 1's frame and the product collapses to
//   local = (sum a_i cos(phi_i), sum a_i sin(phi_i), sum eps_i),  phi_i = theta_2 + .. + theta_i
//   p     = Rz(theta_1) ([a_1, 0, eps_1] + Rx(alpha_1) local)
// with the cumulative angles formed by the addition theorems -- ~1/3 of the general path's instructions,
// which is what lets the fp32 kernel run at HBM speed.
template <typename Real>
__device__ __forceinline__ bool fk_position(const IkbRobot &rc, const Real th[4], Real &px, Real &py,
                                            Real &pz)
{
    const Real TWO_PI = ikb_two_pi<Real>();
    bool ok = true;
    Real s[4], c[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        ok &= !(fabs(th[i]) > TWO_PI);  // forward.py:23-25 (NaN passes, as upstream)
        ikb_sincos(th[i], &s[i], &c[i]);
    }
    if (rc.fk_planar_tail) {
        const Real *k = fk_constants<Real>(rc);
        fk_planar_tail_position<Real>(s, c, k[0], k[1], k[2], k[3], k[4], k[5], k[6], k[7], px, py, pz);
        return ok;
    }
    Real R[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
    px = py = pz = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const Real a = (Real)rc.a[i], e = (Real)rc.eps[i];
        const Real vx = a * c[i], vy = a * s[i];
        px += R[0] * vx + R[1] * vy + R[2] * e;
        py += R[3] * vx + R[4] * vy + R[5] * e;
        pz += R[6] * vx + R[7] * vy + R[8] * e;
        if (i < 3) {
            const Real ca = (Real)rc.cos_alpha[i], sa = (Real)rc.sin_alpha[i];
            // M = Rz(t) Rx(alpha) = [[c, -s ca, s sa], [s, c ca, -c sa], [0, sa, ca]]
            const Real m01 = -s[i] * ca, m02 = s[i] * sa, m11 = c[i] * ca, m12 = -c[i] * sa;
#pragma unroll
            for (int r = 0; r < 3; ++r) {
                const Real r0 = R[3 * r], r1 = R[3 * r + 1], r2 = R[3 * r + 2];
                R[3 * r] = r0 * c[i] + r1 * s[i];
                R[3 * r + 1] = r0 * m01 + r1 * m11 + r2 * sa;
                R[3 * r + 2] = r0 * m02 + r1 * m12 + r2 * ca;
            }
        }
    }
    return ok;
}

// ||FK(th) - target|| for the solvers' epilogues: same arithmetic as K3 on the same (already rounded) angles.
// Out-of-range angles (forward.py:23-25) give NaN, as K3 stores for such rows.
template <typename Real>
__device__ __forceinline__ Real ikb_fk_error(const IkbRobot &rc, const Real th[4], Real tx, Real ty, Real tz)
{
    Real px, py, pz;
    bool ok = fk_position<Real>(rc, th, px, py, pz);
#pragma unroll
    for (int j = 0; j < 4; ++j)
        ok &= !(rc.alpha[j] < -6.283185307179586) & !(rc.alpha[j] > 6.283185307179586);
    const Real dx = px - tx, dy = py - ty, dz = pz - tz;
    const Real err = sqrt(dx * dx + dy * dy + dz * dz);
    return ok ? err : (Real)__int_as_float(0x7fc00000);
}

// fabrik.cu -- K1: batched FABRIK inverse kinematics + fp64 angle extraction (sm_100a).
//
// Replaces, per target, reference FabrikInverseKinematics.ikine (inverse.py:115-139):
//   check_limits (inverse.py:26-35) -> Fabrik.calculate (fabrik.py:44-67, built from
//   get_point_between / get_distance_between, point.py:25-45) -> __get_angles (inverse.py:54-112).
//
// Design (see DESIGN.md "K1"):
//  * One chain per lane, chain state in registers.  The seed chain and the target lie in one
//    vertical plane through the z axis, so the iteration runs in 2-D (r, z) coordinates.
//  * P0 is pinned to the start joint and P3 is only needed at the end, so one iteration is
//    4 point-at-distance updates + 5 reciprocal square roots; the two convergence errors are
//    | |S - b1| - d0 | and | |T - f2| - d3 | (algebraically the reference's |b0 - S|, |f3 - T|).
//  * ONE scan of the input: persistent warps pull chunks of IKB_FABRIK_CHUNK consecutive targets from a global
//    counter, classify every target when it is staged (workspace limits, in-plane radius, theta_1 of its plane,
//    reachable / out of reach) and queue it in shared memory; the rows of the next staging step are loaded before
//    the pass loop and consumed after it.
//  * Iteration counts are bimodal (3..8 inside the workspace, exactly max_iter outside).  Reachable targets run with
//    LANE REFILL: a lane that converges parks its chain (with everything the angle extraction needs about its
//    target) in a per-warp ring and takes the next staged target in the same step, so the pass loop stays at full
//    width.  Out-of-reach targets run in LOCKSTEP batches of 64, two chains per lane, exactly max_iter passes with
//    no verdict, vote or parking, while the warp's reachable chains wait in registers.
//  * The angle extraction runs on 32 parked chains at once; its cosines and their 8-decimal rounding are fp64,
//    the trigonometric tail follows the precision of the caller's angle buffer (fp32 pipe for float32 buffers).
//  * Row i of the output always belongs to row i of the input, whatever order lanes finish in.
#include <cstdlib>

#include "fk_device.cuh"
#include "vec3.cuh"

// -DIKB_FABRIK_CHECK: trap when a shared-memory queue would be indexed outside its capacity (the pool's
// compute-sanitizer is closed, so the debug variant of tools/build_variant.sh carries its own bounds checks)
#ifdef IKB_FABRIK_CHECK
#include <cstdio>
#define IKB_CHECK(cond)                                                                    \
    do {                                                                                   \
        if (!(cond)) {                                                                     \
            printf("IKB_CHECK failed: %s (line %d, block %d thread %d)\n", #cond, __LINE__, \
                   (int)blockIdx.x, (int)threadIdx.x);                                     \
            __trap();                                                                      \
        }                                                                                  \
    } while (0)
#else
#define IKB_CHECK(cond) do {} while (0)
#endif

#define IKB_FABRIK_CHUNK 256
#define IKB_FABRIK_WARPS 8
#define IKB_Q 64  // per-warp input queue capacity (ring), power of two
#ifndef IKB_FABRIK_MIN_CTAS
#define IKB_FABRIK_MIN_CTAS 3
#endif

namespace {

struct FabrikArgs {
    const void *xyz;
    int xyz_f64;
    long long n;
    long long index_base;  // global row of xyz[0] (host pipeline chunks)
    void *angles;
    int angles_f64;
    int *iters;  // nullable
    void *fk_err;  // nullable: ||FK(angles) - target|| per row in the angles' dtype (fused K3, SURVEY 8 a6)
    int fk_stats;  // accumulate sum_fk_error / n_fk_error even without the per-row array
    IkbDeviceStats *stats;
    unsigned long long *work_counter;
    double far_thr2;  // > 0: targets with |T - S|^2 above it run in lockstep batches (see is_far)
    IkbRobot rc;
};

template <typename Real>
struct PlanarChain {
    Real r1, z1, r2, z2;  // joints 1 and 2; joint 0 is pinned, joint 3 is derived
};

// Convergence band of one end of the chain: |sqrt(n2) - d| > tol  <=>  n2 outside [lo2, hi2] with
// lo2 = max(d - tol, 0)^2, hi2 = (d + tol)^2.  Testing the squared length saves the square root; the two
// forms differ only when n2 sits within an ulp of a band edge (probability ~1e-13 per test in fp64).
template <typename Real>
struct Band {
    Real lo2, hi2;  // precomputed on the host (IkbRobot::band_*): kernel-parameter constants
    __device__ __forceinline__ bool outside(Real n2) const { return (n2 < lo2) | (n2 > hi2); }
};

template <typename Real>
__device__ __forceinline__ Band<Real> make_band(const IkbRobot &rc, int which);
template <>
__device__ __forceinline__ Band<double> make_band<double>(const IkbRobot &rc, int which)
{
    return Band<double>{rc.band_lo2[which], rc.band_hi2[which]};
}
template <>
__device__ __forceinline__ Band<float> make_band<float>(const IkbRobot &rc, int which)
{
    return Band<float>{rc.band_lo2_f[which], rc.band_hi2_f[which]};
}

// One forward-and-backward-reaching pass (reference fabrik.py:60-63) in the (r, z) plane.
// Returns true when the reference's loop condition (start_error > tol or goal_error > tol) holds.
// start_error = |b0 - S| = | |S - b1| - d0 | and goal_error = |f3 - T| = | |T - f2| - d3 |, because b0 and
// f3 are the points at distance d0 / d3 from b1 / f2 towards S / T.
// d / sqrt(n2): fp64 folds the link length into the correction step (ikb_rsqrt_times), fp32 is seed times d
template <typename Real>
struct LinkScale;
template <>
struct LinkScale<double> {
    const IkbScaledRsqrt &k;  // in the kernel's parameter block: the DFMAs take the constants as c[][] operands
    __device__ __forceinline__ explicit LinkScale(const IkbScaledRsqrt &kk) : k(kk) {}
    __device__ __forceinline__ double over_sqrt(double n2) const { return ikb_rsqrt_times(n2, k); }
};
template <>
struct LinkScale<float> {
    float d;
    __device__ __forceinline__ explicit LinkScale(const IkbScaledRsqrt &kk) : d((float)kk.d) {}
    __device__ __forceinline__ float over_sqrt(float n2) const { return d * ikb_rsqrt(n2); }
};

template <typename Real>
__device__ __forceinline__ bool fabrik_pass(PlanarChain<Real> &c, Real Tr, Real Tz, Real R0, Real Z0,
                                            const LinkScale<Real> &d1, const LinkScale<Real> &d2,
                                            const Band<Real> &start_band, const Band<Real> &goal_band)
{
    // backward (fabrik.py:19-29): b3 = T, b2 = PB(b3, P2, d2), b1 = PB(b2, P1, d1), b0 = PB(b1, P0, d0)
    // (this file is compiled with --fmad=false: every fused multiply-add is written out, so that a row's result does
    //  not depend on which kernel, or which inlined copy of this function, happens to process it)
    Real dr = c.r2 - Tr, dz = c.z2 - Tz;
    Real s = d2.over_sqrt(fma(dz, dz, dr * dr));
    const Real b2r = fma(s, dr, Tr), b2z = fma(s, dz, Tz);
    dr = c.r1 - b2r; dz = c.z1 - b2z;
    s = d1.over_sqrt(fma(dz, dz, dr * dr));
    const Real b1r = fma(s, dr, b2r), b1z = fma(s, dz, b2z);
    dr = R0 - b1r; dz = Z0 - b1z;
    Real n2 = fma(dz, dz, dr * dr);
    const bool start_off = start_band.outside(n2);                       // fabrik.py:61
    // forward (fabrik.py:32-42): f0 = S, f1 = PB(f0, b1, d1), f2 = PB(f1, b2, d2), f3 = PB(f2, b3, d3)
    s = d1.over_sqrt(n2);
    c.r1 = fma(-s, dr, R0); c.z1 = fma(-s, dz, Z0);  // (b1 - S) = -(dr, dz)
    dr = b2r - c.r1; dz = b2z - c.z1;
    s = d2.over_sqrt(fma(dz, dz, dr * dr));
    c.r2 = fma(s, dr, c.r1); c.z2 = fma(s, dz, c.z1);
    dr = Tr - c.r2; dz = Tz - c.z2;
    n2 = fma(dz, dz, dr * dr);                // f3 itself is only needed after the last pass
    return start_off | goal_band.outside(n2);                            // fabrik.py:63
}

#ifndef IKB_FABRIK_LOW_WATER
#define IKB_FABRIK_LOW_WATER 8  // staged targets below which the warp leaves its pass loop to stage more (while input is left)
#endif

// theta_1 of a target's plane is evaluated when the target is staged and travels with the chain in the precision of
// the output buffer
template <bool OUT32>
struct TailType {
    using type = double;
};
template <>
struct TailType<true> {
    using type = float;
};

// sqrt(x) for x >= 0 through the reciprocal square root (2 ulp); exact 0 for x == 0
__device__ __forceinline__ double fast_sqrt(double x)
{
    const double s = x * ikb_rsqrt(x);
    return x == 0.0 ? 0.0 : s;
}

__device__ __forceinline__ double dist2d_sq(double ar, double az, double br, double bz)
{
    const double dr = ar - br, dz = az - bz;
    return fma(dz, dz, dr * dr);
}

// round(x, 8) of reference inverse.py:81,92,100: q = rint(x * 1e8) is an integer, q / 1e8 is formed as
// q * 1e-8 plus one exact-residual correction (1e8 is exactly representable), which reproduces the
// correctly rounded quotient np.round / Python's round give, in particular exactly +-1.0 at q = +-1e8.
__device__ __forceinline__ double round8(double x)
{
    const double q = rint(x * 1e8);
    const double r = q * 1e-8;
    return fma(fma(-r, 1e8, q), 1e-8, r);
}

// asin(s) for 0 <= s <= 0.5 given t = s^2: s + s t P(t), P fitted by tools/fit_asin_poly.py
// (degree 9, max abs error 1.2e-15).  Shared core of the acos / atan2 replacements below: the CUDA
// library versions cost ~4x more instructions and the epilogue is the second largest consumer of
// issue slots in this kernel.
__constant__ double c_asin_poly[10] = {
    0.16666666666025234, 0.07500000093993356, 0.04464280537685713, 0.03038341968562146,
    0.022347394121891163, 0.017613143412093663, 0.012211296489012176, 0.01903265892950786,
    -0.009325464322296697, 0.03306665466887422};

__device__ __forceinline__ double asin_core(double s, double t)
{
    double p = c_asin_poly[9];  // constant-bank operands: no immediates to materialise
#pragma unroll
    for (int i = 8; i >= 0; --i)
        p = fma(p, t, c_asin_poly[i]);
    return fma(s * t, p, s);
}

// acos(c), |c| <= 1 (NaN outside, like math.acos raising ValueError upstream); abs error < 3e-15.
// |c| <= 1/2: pi/2 - asin(c);  otherwise 2 asin(sqrt((1 - |c|) / 2)), reflected for c < 0.
__device__ __forceinline__ double acos_fast(double c)
{
    const double PI = 3.141592653589793;
    const double a = fabs(c);
    const bool small = a <= 0.5;
    const double t = small ? c * c : fma(-0.5, a, 0.5);
    const double s = small ? a : fast_sqrt(t);
    const double r = asin_core(s, t);
    const double big = c > 0.0 ? 2.0 * r : PI - 2.0 * r;
    return small ? PI / 2 - copysign(r, c) : big;
}

// atan2(uy, ux) for a UNIT vector (ux, uy); abs error < 3e-15.  The angle to the x axis comes from
// asin(|uy|) when |uy| <= 1/2, from pi/2 - asin(|ux|) when |ux| <= 1/2, else from the half-angle form.
__device__ __forceinline__ double atan2_unit(double uy, double ux)
{
    const double PI = 3.141592653589793;
    const double ay = fabs(uy), ax = fabs(ux);
    const bool m0 = ay <= 0.5, m1 = ax <= 0.5;
    const double t = m0 ? ay * ay : (m1 ? ax * ax : fma(-0.5, ax, 0.5));
    const double s = m0 ? ay : (m1 ? ax : fast_sqrt(t));
    const double r = asin_core(s, t);
    double phi = m0 ? r : (m1 ? PI / 2 - r : 2.0 * r);
    phi = ux < 0.0 ? PI - phi : phi;
    return copysign(phi, uy);
}

// ---- the same two functions on the fp32 pipe, for float32 OUTPUT buffers ------------------------------------------
// K1 is bound by the fp64 pipe while the fp32 pipe idles (ncu: 5 % active).  When the caller's angle buffer is float32
// the result is rounded to 24 bits anyway, so everything after the last step that needs fp64 -- the cosine with its
// 8-decimal rounding (inverse.py:81,92,100: the 1e-8 quantum must not flip) -- runs in fp32: t = (1 - |c|) / 2 is
// still formed in fp64 (no cancellation near |c| = 1, where the reference itself quantises), then sqrt, a degree-4
// polynomial (tools/fit_asin_poly.py 4: 1.6e-9 abs) and the final combination with pi in fp32.  Measured against the
// fp64 tail: <= 4e-7 rad (1.7 ulp of pi in fp32), 250x inside the 1e-4 rad bar.  float64 buffers (the list API, the
// reference's own tests) keep the fp64 tail above (2e-15).
#ifndef IKB_FABRIK_TAIL32
#define IKB_FABRIK_TAIL32 1
#endif
#define IKB_PI_F 3.14159274101257324f

__device__ __forceinline__ float asin_core_f(float s, float t)
{
    float p = 0.0437449409671523f;
    p = fmaf(p, t, 0.023150225160843828f);
    p = fmaf(p, t, 0.045707160478796506f);
    p = fmaf(p, t, 0.07493066952010845f);
    p = fmaf(p, t, 0.1666682263762875f);
    return fmaf(s * t, p, s);
}

__device__ __forceinline__ float sqrt_approx_f(float x)
{
    float y;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// acos of an fp64 cosine (NaN outside [-1, 1], like acos_fast)
__device__ __forceinline__ float acos_f32(double c)
{
    const double a = fabs(c);
    const bool small = a <= 0.5;
    const float v = (float)(small ? a : fma(-0.5, a, 0.5));  // |c|, or t = (1 - |c|) / 2 formed in fp64
    const float t = small ? v * v : v;
    const float s = small ? v : sqrt_approx_f(v);
    const float r = asin_core_f(s, t);
    const float big = c > 0.0 ? 2.0f * r : IKB_PI_F - 2.0f * r;
    return small ? 0.5f * IKB_PI_F - (c < 0.0 ? -r : r) : big;
}

// atan2(uy, ux) of a unit vector given in fp64, evaluated in fp32
__device__ __forceinline__ float atan2_unit_f32(double uy64, double ux64)
{
    const float uy = (float)uy64, ux = (float)ux64;
    const float ay = fabsf(uy), ax = fabsf(ux);
    const bool m0 = ay <= 0.5f, m1 = ax <= 0.5f;
    const float h = fmaf(-0.5f, ax, 0.5f);                   // exact: ax >= 1/2 on this branch
    const float t = m0 ? ay * ay : (m1 ? ax * ax : h);
    const float s = m0 ? ay : (m1 ? ax : sqrt_approx_f(h));
    const float r = asin_core_f(s, t);
    float phi = m0 ? r : (m1 ? 0.5f * IKB_PI_F - r : 2.0f * r);
    phi = ux < 0.0f ? IKB_PI_F - phi : phi;
    return copysignf(phi, uy);
}

// In-plane radius of a target and the unit direction of its vertical plane.  Targets on the z axis
// have no direction (the reference's theta_1 is rounding noise there, SURVEY 7.3-7): +x is used.
__device__ __forceinline__ double planar_radius(double x, double y, double &ux, double &uy)
{
    const double n2 = fma(y, y, x * x);
    const double rs = ikb_rsqrt(n2);
    const bool on_axis = (n2 == 0.0);
    ux = on_axis ? 1.0 : x * rs;
    uy = on_axis ? 0.0 : y * rs;
    return on_axis ? 0.0 : n2 * rs;
}

// Out-of-reach split.  With |T - S| > d1 + d2 + d3 + tol the goal error |f3 - T| = ||T - f2| - d3| can never get
// below tol (f2 stays within d1 + d2 of S), so the reference runs exactly max_iter passes on such a target and its
// last verdict is "not converged".  Those targets -- 38 % of a uniform workspace sample, 87 % of its passes -- go to
// fabrik_far_kernel, which runs the passes in lockstep without the per-pass verdict, parking and refill; the
// lane-refill kernel skips them when it stages its input.  Both kernels evaluate this predicate on the raw target,
// with explicitly rounded operations, so that every row is claimed by exactly one of them.
__device__ __forceinline__ bool is_far(double x, double y, double z, double R0, double Z0, double thr2)
{
    const double q = __fma_rn(x, x, __dmul_rn(y, y)), dz = __dadd_rn(z, -Z0);
    double d2;
    if (R0 == 0.0) {  // base on the z axis (every arm of the reference's family): no square root needed
        d2 = __fma_rn(dz, dz, q);
    } else {
        const double dr = __dadd_rn(__dsqrt_rn(q), -R0);
        d2 = __fma_rn(dr, dr, __dmul_rn(dz, dz));
    }
    return (d2 > thr2) & (d2 < 1.0e300);  // false for NaN and for infinite targets (those stop after one pass)
}

// Finish one solved chain: derive the effector, lift to 3-D, extract the four angles in fp64 as
// reference inverse.py:54-112 does, write outputs, raise the per-row flags.
// Out of line on purpose: the fp32 FK needs ~40 registers of its own, and inlined into the epilogue it pushed the
// register allocation of the whole kernel (the solve got 10 % slower even with the error switched off).  Scalars
// only, so nothing of the kernel's parameter block has to be spilled for the call.
__device__ __noinline__ float fused_fk_error_f32(float t0, float t1, float t2, float t3, float tx, float ty, float tz,
                                                 float a0, float a1, float a2, float a3, float eps0, float w, float ca,
                                                 float sa)
{
    const float th[4] = {t0, t1, t2, t3};
    return ikb_fk_error_planar_tail<float>(th, tx, ty, tz, a0, a1, a2, a3, eps0, w, ca, sa);
}
__device__ __noinline__ double fused_fk_error_f64(double t0, double t1, double t2, double t3, double tx, double ty,
                                                  double tz, double a0, double a1, double a2, double a3, double eps0,
                                                  double w, double ca, double sa)
{
    const double th[4] = {t0, t1, t2, t3};
    return ikb_fk_error_planar_tail<double>(th, tx, ty, tz, a0, a1, a2, a3, eps0, w, ca, sa);
}

// Bits riding in a chain's iteration counter (the count itself is below 2^28).
#define IKB_K_MASK 0x0fffffff
#define IKB_CAPPED_BIT 0x40000000  // the chain stopped on max_iter, not on the tolerance

// Finish one solved chain: derive the effector, extract the four angles as reference inverse.py:54-112 does, write
// the outputs, raise the per-row flags.  Everything it needs about the target travels with the parked chain (Tr, Tz,
// theta_1 of the target's plane): no second read of the input (round 1 re-read the row here).
// CONST_LINKS: the chain was iterated in fp64, so its segments have their link lengths to the last place (see below);
// an fp32-iterated chain is only good to 1e-7 there and takes the general form with computed lengths.
// ZERO_ITER: the reference's loop never runs (tol >= 1 or max_iter <= 0) and every chain is the seed chain -- a separate
// instantiation, so that the common one carries none of its code (the seed constants alone were 18 instructions per
// extraction when this was a run-time branch).
template <bool FUSE_FK, bool OUT32, bool CONST_LINKS, bool ZERO_ITER, typename Th1>
__device__ __forceinline__ void fabrik_epilogue(const FabrikArgs &a, int idx, int k_raw, double r1, double z1, double r2,
                                                double z2, double Tr, double Tz, Th1 th1, double &fk_sum, unsigned &fk_cnt)
{
    const IkbRobot &rc = a.rc;
    const double PI = 3.141592653589793;
    const int k = k_raw & IKB_K_MASK;
    const long long row = a.index_base + idx;
    const double R0 = rc.seed_r[0], Z0 = rc.seed_z[0];
    double r3, z3, c2, c3, c4, n_bd, n_ce;
    bool odd;  // anything that needs the slow classification below: a cosine outside [-1, 1], NaN, a zero length
    double n2 = 1.0;
    if (!ZERO_ITER) {  // f3 = PB(f2, T, d3) (fabrik.py:40)
        const double dr = Tr - r2, dz = Tz - z2;
        n2 = fma(dz, dz, dr * dr);
        const double s = ikb_rsqrt_times(n2, rc.link_k[3]);
        r3 = fma(s, dr, r2); z3 = fma(s, dz, z2);
    } else {  // the reference's loop never ran (tol >= 1 or max_iter <= 0): the chain is the seed chain
        r1 = rc.seed_r[1]; z1 = rc.seed_z[1]; r2 = rc.seed_r[2]; z2 = rc.seed_z[2];
        r3 = rc.seed_r[3]; z3 = rc.seed_z[3];
    }
    if (CONST_LINKS && !ZERO_ITER) {
        // The three cosines of inverse.py:77-100 on squared lengths.  After at least one pass B = S and C, D, E are
        // points at distance d1, d2, d3 from their predecessor (f1 = PB(S, b1, d1) etc.), so |BC|, |CD|, |DE| ARE the
        // link lengths up to the last-place rounding the reference's own sqrt / division carry -- the same order as
        // replacing a squared rounded root by the squared length, which this epilogue does throughout.  That leaves
        // three computed squared lengths (|AC|, |BD|, |CE|) and makes every denominator a constant of the arm:
        //   cos = (l1^2 + l2^2 - opposite^2) / (2 l1 l2)  ->  (sum_k - opposite^2) * inv_k   (host constants)
        const double n_ac = fma(z1, z1, r1 * r1);
        n_bd = dist2d_sq(R0, Z0, r2, z2);
        n_ce = dist2d_sq(r1, z1, r3, z3);
        c2 = round8((rc.cos_sum[0] - n_ac) * rc.cos_inv[0]);   // inverse.py:77-81
        c3 = round8((rc.cos_sum[1] - n_bd) * rc.cos_inv[1]);   // :90-92
        c4 = round8((rc.cos_sum[2] - n_ce) * rc.cos_inv[2]);   // :98-100
        // |c| <= 1 is false for NaN as well: a chain that went NaN / inf through 0 * inf inside a pass ends up here
        odd = !((fabs(c2) <= 1.0) & (fabs(c3) <= 1.0) & (fabs(c4) <= 1.0)) | (n2 == 0.0) | (n_ce == 0.0);
    } else {
        // the general form with computed segment lengths: the seed chain (its segments are whatever the DH table
        // says) and fp32-iterated chains
        const double n_bc = dist2d_sq(R0, Z0, r1, z1), n_cd = dist2d_sq(r1, z1, r2, z2), n_de = dist2d_sq(r2, z2, r3, z3);
        const double n_ac = fma(z1, z1, r1 * r1);
        n_bd = dist2d_sq(R0, Z0, r2, z2);
        n_ce = dist2d_sq(r1, z1, r3, z3);
        const double den3 = n_bc * n_cd, den4 = n_cd * n_de;
        c2 = round8(((rc.seed_ab2 + n_bc) - n_ac) * ikb_rsqrt(n_bc) * rc.half_inv_ab);
        c3 = round8(((n_bc + n_cd) - n_bd) * ikb_rsqrt(den3) * 0.5);
        c4 = round8(((n_cd + n_de) - n_ce) * ikb_rsqrt(den4) * 0.5);
        odd = !((fabs(c2) <= 1.0) & (fabs(c3) <= 1.0) & (fabs(c4) <= 1.0)) | (den3 == 0.0) | (den4 == 0.0) | (n_ce == 0.0) |
              (n2 == 0.0);
    }
    const bool flip = r3 < 0.0;  // theta_1 = atan2(E.y, E.x) with E = r3 (ux, uy) (inverse.py:60): only the sign of r3 matters
    // t4_point_bt = PB(C, E, |CE| / 2) (inverse.py:102): (|CE|/2)/|CE| is exactly 0.5
    const double mr = fma(0.5, r3 - r1, r1), mz = fma(0.5, z3 - z1, z1);
    // C.x * D.x < 0 (:82) with C.x = r1 ux, D.x = r2 ux: the sign of r1 r2.  On the plane x = 0 the reference's product
    // is seed noise (DESIGN 1); the in-plane sign is the limit x -> 0+ of its own rule
    const bool elbow_neg = r1 * r2 < 0;
    const bool wrist_neg = n_bd > dist2d_sq(R0, Z0, mr, mz);                // :103
    // Rare rows, classified out of line (a branch that is almost never taken):
    //  * a zero-length segment (ZeroDivisionError upstream, point.py:40) -- a length of 0, or a chain that is no longer
    //    finite although its target is (a NaN target gives NaN angles without an exception upstream);
    //  * a cosine outside [-1, 1] after the rounding (ValueError from acos upstream).
    bool zero_div = false;
    if (odd) {
        const bool finite_t = isfinite(Tr + Tz);
        const bool finite_c = isfinite(c2 + c3 + c4);
        zero_div = finite_t & (!finite_c | (n_ce == 0.0) | (rc.seed_ab == 0.0) | !isfinite(r3 + z3));
        if (zero_div)
            atomicMin(&a.stats->first_zero_division, row);
        else if (finite_c)
            atomicMin(&a.stats->first_domain_error, row);
    }
    if (a.iters)
        a.iters[idx] = k;
    double x = 0, y = 0, z = 0;
    if (FUSE_FK)  // small batches only (one launch instead of two): the error needs the target itself
        ikb_load_xyz(a.xyz, a.xyz_f64, idx, x, y, z);
    if (OUT32 && IKB_FABRIK_TAIL32) {
        // float32 buffer: the trigonometric tail on the fp32 pipe (see acos_f32).  theta_1 of the target's plane was
        // evaluated when the target was staged; an effector on the far side of the z axis turns it by pi.
        float t0 = (float)th1;
        t0 = flip ? t0 - copysignf(IKB_PI_F, t0) : t0;
        t0 = r3 == 0.0 ? 0.0f : (r3 != r3 ? __int_as_float(0x7fc00000) : t0);
        const float acos2 = acos_f32(c2), acos3 = acos_f32(c3), acos4 = acos_f32(c4);
        float t1 = elbow_neg ? 1.5f * IKB_PI_F - acos2 : -(0.5f * IKB_PI_F - acos2);     // :82-85
        float t2 = -(IKB_PI_F - acos3);                                                  // :93
        float t3 = wrist_neg ? -(IKB_PI_F - acos4) : (IKB_PI_F - acos4);                 // :103-108
        if (zero_div)
            t0 = t1 = t2 = t3 = __int_as_float(0x7fc00000);
        reinterpret_cast<float4 *>(a.angles)[idx] = make_float4(t0, t1, t2, t3);
        if (FUSE_FK) {  // fused K3: FK of the angles as stored
            const float e = fused_fk_error_f32(t0, t1, t2, t3, (float)x, (float)y, (float)z, rc.fkc_f[0], rc.fkc_f[1],
                                               rc.fkc_f[2], rc.fkc_f[3], rc.fkc_f[4], rc.fkc_f[5], rc.fkc_f[6], rc.fkc_f[7]);
            if (a.fk_err)
                reinterpret_cast<float *>(a.fk_err)[idx] = e;
            if (isfinite(e)) {
                fk_sum += (double)e;
                ++fk_cnt;
            }
        }
        return;
    }
    double th[4];
    th[0] = (double)th1;
    th[0] = flip ? th[0] - copysign(PI, th[0]) : th[0];
    th[0] = r3 == 0.0 ? 0.0 : (r3 != r3 ? r3 : th[0]);
    const double acos2 = acos_fast(c2);
    th[1] = elbow_neg ? (3 * PI / 2) - acos2 : -(PI / 2 - acos2);  // :82-85
    th[2] = -(PI - acos_fast(c3));                                                        // :93
    const double acos4 = acos_fast(c4);
    th[3] = wrist_neg ? -(PI - acos4) : (PI - acos4);   // :103-108
    if (zero_div)
        th[0] = th[1] = th[2] = th[3] = __longlong_as_double(0x7ff8000000000000LL);
    ikb_store_angles(a.angles, OUT32 ? 0 : 1, idx, th);
    if (FUSE_FK) {  // fused K3: FK of the angles as stored, in the stored precision
        double err;
        if (!OUT32) {
            err = fused_fk_error_f64(th[0], th[1], th[2], th[3], x, y, z, rc.fkc[0], rc.fkc[1], rc.fkc[2], rc.fkc[3],
                                     rc.fkc[4], rc.fkc[5], rc.fkc[6], rc.fkc[7]);
            if (a.fk_err)
                reinterpret_cast<double *>(a.fk_err)[idx] = err;
        } else {
            const float e = fused_fk_error_f32((float)th[0], (float)th[1], (float)th[2], (float)th[3], (float)x, (float)y,
                                               (float)z, rc.fkc_f[0], rc.fkc_f[1], rc.fkc_f[2], rc.fkc_f[3], rc.fkc_f[4],
                                               rc.fkc_f[5], rc.fkc_f[6], rc.fkc_f[7]);
            if (a.fk_err)
                reinterpret_cast<float *>(a.fk_err)[idx] = e;
            err = (double)e;
        }
        if (isfinite(err)) {
            fk_sum += err;
            ++fk_cnt;
        }
    }
}

// Per-warp queues in shared memory (one struct per warp: every access is "warp base + constant + slot").
//   in_*  : staged reachable targets waiting for a free lane (ring)
//   out_* : parked solved chains waiting for a full-width angle extraction (ring): < 32 wait when a pass starts and a
//           pass parks at most 32
//   far_* : staged out-of-reach targets waiting for a lockstep batch of 64 (always at the front of the arrays)
#define IKB_OUT_Q 64
#define IKB_FAR_BATCH 64
#define IKB_FAR_Q (IKB_FAR_BATCH + 32)
// Records are kept as pairs (16-byte shared-memory accesses for fp64): the lane-refill loop is bound by instruction
// issue on short-iteration data, and a park-and-refill step moves 13 values per finished chain.
template <typename Real>
struct Pair;
template <>
struct Pair<double> {
    using type = double2;
};
template <>
struct Pair<float> {
    using type = float2;
};
template <typename Real, typename Th1>
struct WarpQueues {
    using Real2 = typename Pair<Real>::type;
    Real2 in_t[IKB_Q];                                           // (Tr, Tz)
    Real2 out_j1[IKB_OUT_Q], out_j2[IKB_OUT_Q], out_t[IKB_OUT_Q];  // (r1, z1), (r2, z2), (Tr, Tz)
    Real2 far_t[IKB_FAR_Q];
    int2 in_ik[IKB_Q], out_ik[IKB_OUT_Q], far_ik[IKB_FAR_Q];     // (row, iteration count + flags)
    Th1 in_th1[IKB_Q], out_th1[IKB_OUT_Q], far_th1[IKB_FAR_Q];
};

// One warp's whole job: ONE scan of the input through a global chunk counter; every staged target is classified
// (is_far) and queued for one of two pass loops that the warp alternates between:
//   * reachable targets -> LANE REFILL: one chain per lane; a lane that converges parks its chain and takes the next
//     staged target in the same step, so the pass loop runs at full width until 32 parked chains are ready for the
//     angle extraction or the staged targets run low;
//   * out-of-reach targets -> LOCKSTEP: batches of 64 (two chains per lane for instruction-level parallelism) run
//     exactly max_iter passes without verdict, vote or parking, while the warp's reachable chains wait in registers.
// The input rows of the NEXT staging step are loaded before the pass loop and consumed after it (their latency is
// hidden behind the passes).
template <typename Real, bool FUSE_FK, bool OUT32, bool ZERO_ITER>
__device__ __forceinline__ void fabrik_warp_loop(const FabrikArgs &a, WarpQueues<Real, typename TailType<OUT32>::type> *s_queues)
{
    using Th1 = typename TailType<OUT32>::type;
    using Real2 = typename Pair<Real>::type;
    const int lane = threadIdx.x & 31;
    WarpQueues<Real, Th1> &q = s_queues[threadIdx.x >> 5];
    const unsigned lt = ikb_lanemask_lt();
    const IkbRobot &rc = a.rc;
    const Real R0 = (Real)rc.seed_r[0], Z0 = (Real)rc.seed_z[0];
    const LinkScale<Real> d1(rc.link_k[1]), d2(rc.link_k[2]);
    const Band<Real> start_band = make_band<Real>(rc, 0), goal_band = make_band<Real>(rc, 1);
    const int max_iter = rc.max_iter;
    constexpr bool zero_iter = ZERO_ITER;

    // lane-refill state: one chain per lane
    bool active = false;
    unsigned active_mask = 0;  // warp-uniform copy of `active`
    int idx = 0, k = 0;
    Real Tr = 0, Tz = 0;
    Th1 th1 = 0;
    PlanarChain<Real> c{0, 0, 0, 0};
    int in_head = 0, in_cnt = 0, out_head = 0, out_cnt = 0, far_cnt = 0;
    // input scan
    long long cur = 0, cur_end = 0;
    bool exhausted = false;
    double px = 0, py = 0, pz = 0;  // prefetched rows cur - pf_m .. cur - 1 (lane l holds row pf_row)
    long long pf_row = 0;
    int pf_m = 0;                   // 0: no more input
    unsigned long long iters_local = 0;
    unsigned solved_local = 0, capped_local = 0;
    double fk_sum = 0.0;
    unsigned fk_cnt = 0;

    auto prefetch = [&]() {
        if (cur == cur_end && !exhausted) {
            unsigned long long base = 0;
            if (lane == 0)
                base = atomicAdd(a.work_counter, (unsigned long long)IKB_FABRIK_CHUNK);
            base = __shfl_sync(IKB_FULL_MASK, base, 0);
            if ((long long)base >= a.n) {
                exhausted = true;
            } else {
                cur = (long long)base;
                cur_end = min(cur + IKB_FABRIK_CHUNK, a.n);
            }
        }
        pf_m = exhausted ? 0 : (int)min((long long)32, cur_end - cur);
        pf_row = cur + lane;
        if (lane < pf_m)
            ikb_load_xyz(a.xyz, a.xyz_f64, pf_row, px, py, pz);
        cur += pf_m;
    };

    // classify the prefetched rows and queue them (full warp width): workspace limits (inverse.py:26-35), the
    // in-plane radius, theta_1 of the target's plane, reachable / out of reach
    auto stage = [&]() {
        const bool valid = lane < pf_m;
        if (valid && ikb_out_of_limits(rc, px, py, pz))
            atomicMin(&a.stats->first_out_of_limits, a.index_base + pf_row);
        double ux, uy;
        const Real tr = (Real)planar_radius(px, py, ux, uy);
        Th1 t1;
        if (OUT32 && IKB_FABRIK_TAIL32)
            t1 = (Th1)atan2_unit_f32(uy, ux);
        else
            t1 = (Th1)atan2_unit(uy, ux);
        const bool far = valid && a.far_thr2 > 0.0 && is_far(px, py, pz, rc.seed_r[0], rc.seed_z[0], a.far_thr2);
        const bool near = valid && !far;
        const unsigned keep_n = __ballot_sync(IKB_FULL_MASK, near), keep_f = __ballot_sync(IKB_FULL_MASK, far);
        if (near) {
            const int slot = (in_head + in_cnt + __popc(keep_n & lt)) & (IKB_Q - 1);
            q.in_ik[slot] = make_int2((int)pf_row, 0);
            q.in_t[slot] = Real2{tr, (Real)pz};
            q.in_th1[slot] = t1;
        }
        if (far) {
            const int slot = far_cnt + __popc(keep_f & lt);
            q.far_ik[slot] = make_int2((int)pf_row, 0);
            q.far_t[slot] = Real2{tr, (Real)pz};
            q.far_th1[slot] = t1;
        }
        in_cnt += __popc(keep_n);
        far_cnt += __popc(keep_f);
        IKB_CHECK(in_cnt <= IKB_Q && far_cnt <= IKB_FAR_Q && in_cnt >= 0 && far_cnt >= 0);
        __syncwarp();
    };

    // angle extraction on a full warp of parked chains (or on the remainder once everything else is done)
    auto drain = [&](bool final) {
        while (out_cnt >= 32 || (final && out_cnt > 0)) {
            const int n_take = min(32, out_cnt);
            IKB_CHECK(out_cnt > 0 && out_cnt <= IKB_OUT_Q);
            if (lane < n_take) {
                const int slot = (out_head + lane) & (IKB_OUT_Q - 1);
                const int2 ik = q.out_ik[slot];
                const int k_raw = ik.y;
                const Real2 j1 = q.out_j1[slot], j2 = q.out_j2[slot], tt = q.out_t[slot];
                fabrik_epilogue<FUSE_FK, OUT32, sizeof(Real) == 8, ZERO_ITER, Th1>(a, ik.x, k_raw, (double)j1.x, (double)j1.y,
                                                                        (double)j2.x, (double)j2.y, (double)tt.x,
                                                                        (double)tt.y, q.out_th1[slot], fk_sum, fk_cnt);
                iters_local += (unsigned)(k_raw & IKB_K_MASK);
                ++solved_local;
                capped_local += (k_raw & IKB_CAPPED_BIT) ? 1u : 0u;
            }
            out_head = (out_head + n_take) & (IKB_OUT_Q - 1);
            out_cnt -= n_take;
            __syncwarp();
        }
    };

    // one lockstep batch of up to 64 out-of-reach targets: chain slot u of lane l takes entry u * 32 + l; empty
    // slots run on a harmless dummy target
    auto far_batch = [&]() {
        const int nb = min(far_cnt, IKB_FAR_BATCH);
        IKB_CHECK(nb > 0 && out_cnt < 32);
        PlanarChain<Real> fc[2];
        Real fTr[2], fTz[2];
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            const int e = u * 32 + lane;
            const Real2 ft = q.far_t[e < nb ? e : 0];
            fTr[u] = e < nb ? ft.x : (Real)100;
            fTz[u] = e < nb ? ft.y : (Real)100;
            fc[u].r1 = (Real)rc.seed_r[1]; fc[u].z1 = (Real)rc.seed_z[1];
            fc[u].r2 = (Real)rc.seed_r[2]; fc[u].z2 = (Real)rc.seed_z[2];
        }
#pragma unroll 1
        for (int it = 0; it < max_iter; ++it) {
#pragma unroll
            for (int u = 0; u < 2; ++u)
                (void)fabrik_pass(fc[u], fTr[u], fTz[u], R0, Z0, d1, d2, start_band, goal_band);
        }
        // park 32 chains at a time behind whatever the lane-refill loop has parked, extract angles at full width
        // (unrolled: a rolled loop keeps both chain sets live across the angle extraction and pushes spills into
        //  the lane-refill pass loop)
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            const int cnt_u = max(0, min(32, nb - 32 * u));
            if (lane < cnt_u) {
                const int e = u * 32 + lane;
                const int slot = (out_head + out_cnt + lane) & (IKB_OUT_Q - 1);
                const int2 fik = q.far_ik[e];
                q.out_ik[slot] = make_int2(fik.x, max_iter | IKB_CAPPED_BIT);
                q.out_j1[slot] = Real2{fc[u].r1, fc[u].z1};
                q.out_j2[slot] = Real2{fc[u].r2, fc[u].z2};
                q.out_t[slot] = Real2{fTr[u], fTz[u]};
                q.out_th1[slot] = q.far_th1[e];
            }
            out_cnt += cnt_u;
            IKB_CHECK(out_cnt <= IKB_OUT_Q);
            __syncwarp();
            drain(false);
        }
        // move the rest (< 32 entries) to the front
        const int rest = far_cnt - nb;
        int2 m_ik = make_int2(0, 0);
        Real2 m_t{0, 0};
        Th1 m_th1 = 0;
        if (lane < rest) {
            m_ik = q.far_ik[nb + lane]; m_t = q.far_t[nb + lane]; m_th1 = q.far_th1[nb + lane];
        }
        __syncwarp();
        if (lane < rest) {
            q.far_ik[lane] = m_ik; q.far_t[lane] = m_t; q.far_th1[lane] = m_th1;
        }
        __syncwarp();
        far_cnt = rest;
    };

    auto take_target = [&](int slot) {
        const int2 ik = q.in_ik[slot];
        const Real2 t = q.in_t[slot];
        idx = ik.x;
        k = ik.y;
        Tr = t.x;
        Tz = t.y;
        th1 = q.in_th1[slot];
        c.r1 = (Real)rc.seed_r[1]; c.z1 = (Real)rc.seed_z[1];
        c.r2 = (Real)rc.seed_r[2]; c.z2 = (Real)rc.seed_z[2];
    };

    prefetch();
    for (;;) {
        // 1. stage input until the reachable queue is more than half full (or the input ends); a lockstep batch runs
        //    whenever 64 out-of-reach targets are waiting, and once more for the remainder at the end of the input
        for (;;) {
            if (far_cnt >= IKB_FAR_BATCH || (pf_m == 0 && far_cnt > 0))
                far_batch();
            if (pf_m == 0 || in_cnt > IKB_Q - 32)
                break;
            stage();
            prefetch();
        }
        // 2. idle lanes take staged targets (start-up, and after the queue ran dry)
        if (active_mask != IKB_FULL_MASK && in_cnt > 0) {
            const unsigned need = ~active_mask;
            const int rank = __popc(need & lt);
            if (!active && rank < in_cnt) {
                take_target((in_head + rank) & (IKB_Q - 1));
                active = true;
            }
            const int take = min(__popc(need), in_cnt);
            in_head = (in_head + take) & (IKB_Q - 1);
            in_cnt -= take;
            active_mask = __ballot_sync(IKB_FULL_MASK, active);
        }
        // 3. FABRIK passes (reference fabrik.py:57-65).  Every lane executes the pass -- lanes without a live chain
        //    compute on stale registers and are ignored -- so the loop body is branch-free; a chain that finishes is
        //    parked and its lane takes the next staged target at once.  The warp leaves the loop when a full warp of
        //    parked chains is ready, when the staged targets run low while there is input left, or when no lane is live.
        if (active_mask != 0) {
            bool leave = false;
            const bool more_input = pf_m > 0;
            do {
                bool more = false;
                if (!zero_iter) {
                    more = fabrik_pass(c, Tr, Tz, R0, Z0, d1, d2, start_band, goal_band);
                    ++k;
                }
                const bool fin = active & (!more | ((k & IKB_K_MASK) >= max_iter));
                const unsigned m = __ballot_sync(IKB_FULL_MASK, fin);
                if (m != 0) {
                    const int rank = __popc(m & lt), nf = __popc(m);
                    if (fin) {
                        const int slot = (out_head + out_cnt + rank) & (IKB_OUT_Q - 1);
                        q.out_ik[slot] = make_int2(idx, more ? (k | IKB_CAPPED_BIT) : k);
                        q.out_j1[slot] = Real2{c.r1, c.z1};
                        q.out_j2[slot] = Real2{c.r2, c.z2};
                        q.out_t[slot] = Real2{Tr, Tz};
                        q.out_th1[slot] = th1;
                        if (rank < in_cnt)
                            take_target((in_head + rank) & (IKB_Q - 1));
                        else
                            active = false;
                    }
                    out_cnt += nf;
                    IKB_CHECK(out_cnt <= IKB_OUT_Q && in_cnt >= 0);
                    if (nf <= in_cnt) {  // every finished lane found a staged target: the loop stays at full width
                        in_head = (in_head + nf) & (IKB_Q - 1);
                        in_cnt -= nf;
                        leave = (out_cnt >= 32) | (more_input & (in_cnt < IKB_FABRIK_LOW_WATER));
                    } else {             // the queue ran dry: leave, restage (or carry on with fewer lanes in the tail)
                        in_head = (in_head + in_cnt) & (IKB_Q - 1);
                        in_cnt = 0;
                        active_mask = __ballot_sync(IKB_FULL_MASK, active);
                        leave = true;
                    }
                }
            } while (!leave);
            __syncwarp();
        }
        // 4. angle extraction at full width.  Same instruction sequence for every row of a launch, so results do not
        //    depend on where in the batch a target sits.
        const bool final = pf_m == 0 && in_cnt == 0 && far_cnt == 0 && active_mask == 0;
        drain(final);
        if (final)
            break;
    }
    // statistics: one atomic per warp and counter
    const unsigned long long it = ikb_warp_sum(iters_local);
    const unsigned sv = ikb_warp_sum(solved_local), cp = ikb_warp_sum(capped_local);
    if (lane == 0 && sv != 0) {
        atomicAdd(&a.stats->sum_iterations, it);
        atomicAdd(&a.stats->n_solved, (unsigned long long)sv);
        if (cp)
            atomicAdd(&a.stats->n_iter_capped, (unsigned long long)cp);
    }
    if (FUSE_FK) {
        const double es = ikb_warp_sum(fk_sum);
        const unsigned ec = ikb_warp_sum(fk_cnt);
        if (lane == 0 && ec != 0) {
            atomicAdd(&a.stats->sum_fk_error, es);
            atomicAdd(&a.stats->n_fk_error, (unsigned long long)ec);
        }
    }
}

template <typename Real, bool FUSE_FK, bool OUT32, bool ZERO_ITER>
__global__ void __launch_bounds__(IKB_FABRIK_WARPS * 32, IKB_FABRIK_MIN_CTAS) fabrik_planar_kernel(const FabrikArgs a)
{
    extern __shared__ __align__(16) unsigned char s_raw[];
    fabrik_warp_loop<Real, FUSE_FK, OUT32, ZERO_ITER>(a, reinterpret_cast<WarpQueues<Real, typename TailType<OUT32>::type> *>(s_raw));
}

// ---- generic ikine: robots whose seed chain leaves the vertical plane (general DH tables) ----------------------
// One target per thread, IEEE fp64 in 3-D with the reference's operation order: seed chain = the theta_1 = 0
// chain rotated about z by atan2(y, x) (inverse.py:123-130), Fabrik.calculate (fabrik.py:44-67), __get_angles
// (inverse.py:54-112).  Slower than the planar kernel (warp-vote exit, no lane refill) -- the reference's own
// robot never takes this path.
struct FabrikGenericIkineArgs {
    const void *xyz;
    int xyz_f64;
    long long n;
    long long index_base;
    void *angles;
    int angles_f64;
    int *iters;
    IkbDeviceStats *stats;
    IkbRobot rc;
};

__global__ void __launch_bounds__(128) fabrik_generic_ikine_kernel(const FabrikGenericIkineArgs a)
{
    const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const bool valid = tid < a.n;                 // lanes past the end redo the last row and write nothing,
    const long long i = valid ? tid : a.n - 1;    // so the warp-wide reductions below see full warps
    const IkbRobot &rc = a.rc;
    const double PI = 3.141592653589793;
    double x, y, z;
    ikb_load_xyz(a.xyz, a.xyz_f64, i, x, y, z);
    const long long row = a.index_base + i;
    if (valid && ikb_out_of_limits(rc, x, y, z))
        atomicMin(&a.stats->first_out_of_limits, row);
    double s1, c1;
    sincos(atan2(y, x), &s1, &c1);
    Vec3 P[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const double sx = rc.seed_xyz[3 * j], sy = rc.seed_xyz[3 * j + 1];
        P[j] = Vec3{sx * c1 - sy * s1, sx * s1 + sy * c1, rc.seed_xyz[3 * j + 2]};
    }
    const Vec3 S = P[0], T{x, y, z};
    const double *d = rc.links;
    double se = 1.0, ge = 1.0;
    int step = 0;
    while ((se > rc.tol || ge > rc.tol) && rc.max_iter > step) {
        const Vec3 b2 = point_between3(T, P[2], d[2]);
        const Vec3 b1 = point_between3(b2, P[1], d[1]);
        const Vec3 b0 = point_between3(b1, P[0], d[0]);
        se = dist3(b0, S);
        P[0] = S;
        P[1] = point_between3(P[0], b1, d[1]);
        P[2] = point_between3(P[1], b2, d[2]);
        P[3] = point_between3(P[2], T, d[3]);
        ge = dist3(P[3], T);
        ++step;
    }
    const Vec3 A{0.0, 0.0, 0.0};
    const Vec3 &B = P[0], &C = P[1], &D = P[2], &E = P[3];
    double th[4];
    th[0] = atan2(E.y, E.x);
    const double ab = dist3(A, B), bc = dist3(B, C), cd = dist3(C, D), de = dist3(D, E);
    const double ac = dist3(A, C), bd = dist3(B, D), ce = dist3(C, E);
    bool zero_div = false;
    double den = 2 * ab * bc;
    zero_div |= (den == 0.0);
    const double c2 = round8((ab * ab + bc * bc - ac * ac) / den);
    const double acos2 = acos(c2);
    th[1] = (C.x * D.x < 0) ? (3 * PI / 2) - acos2 : -(PI / 2 - acos2);
    den = 2 * bc * cd;
    zero_div |= (den == 0.0);
    const double c3 = round8((bc * bc + cd * cd - bd * bd) / den);
    th[2] = -(PI - acos(c3));
    den = 2 * cd * de;
    zero_div |= (den == 0.0) | (ce == 0.0);
    const double c4 = round8((cd * cd + de * de - ce * ce) / den);
    const double acos4 = acos(c4);
    const Vec3 mid = point_between3(C, E, ce / 2);
    th[3] = (bd > dist3(B, mid)) ? -(PI - acos4) : (PI - acos4);
    const bool finite_in = isfinite(x) & isfinite(y) & isfinite(z);
    bool chain_nan = false;
#pragma unroll
    for (int j = 0; j < 4; ++j)
        chain_nan |= !(isfinite(P[j].x) & isfinite(P[j].y) & isfinite(P[j].z));
    zero_div = (zero_div | chain_nan) & finite_in;
    const bool domain = !zero_div & (fabs(c2) > 1.0 | fabs(c3) > 1.0 | fabs(c4) > 1.0);
    if (zero_div) {
        th[0] = th[1] = th[2] = th[3] = __longlong_as_double(0x7ff8000000000000LL);
        if (valid)
            atomicMin(&a.stats->first_zero_division, row);
    }
    if (domain && valid)
        atomicMin(&a.stats->first_domain_error, row);
    if (valid) {
        ikb_store_angles(a.angles, a.angles_f64, i, th);
        if (a.iters)
            a.iters[i] = step;
    }
    const bool more = (se > rc.tol) | (ge > rc.tol);
    const unsigned long long it = ikb_warp_sum(valid ? (unsigned long long)step : 0ULL);
    const unsigned sv = ikb_warp_sum(valid ? 1u : 0u), cp = ikb_warp_sum((valid && more && step > 0) ? 1u : 0u);
    if ((threadIdx.x & 31) == 0 && sv != 0) {
        atomicAdd(&a.stats->sum_iterations, it);
        atomicAdd(&a.stats->n_solved, (unsigned long long)sv);
        if (cp)
            atomicAdd(&a.stats->n_iter_capped, (unsigned long long)cp);
    }
}

}  // namespace

// ---- launchers (called from capi.cu) --------------------------------------------------------------
namespace {
template <typename Real, bool FUSE_FK, bool OUT32, bool ZERO_ITER>
cudaError_t launch_planar_z(const FabrikArgs &a, unsigned grid, cudaStream_t stream)
{
    constexpr size_t smem = sizeof(WarpQueues<Real, typename TailType<OUT32>::type>) * IKB_FABRIK_WARPS;
    static const cudaError_t attr = cudaFuncSetAttribute(fabrik_planar_kernel<Real, FUSE_FK, OUT32, ZERO_ITER>,
                                                         cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (attr != cudaSuccess)
        return attr;
    // three CTAs per SM need ~200 KB of shared memory: ask for the largest carve-out
    static const cudaError_t carve = cudaFuncSetAttribute(fabrik_planar_kernel<Real, FUSE_FK, OUT32, ZERO_ITER>,
                                                          cudaFuncAttributePreferredSharedMemoryCarveout,
                                                          (int)cudaSharedmemCarveoutMaxShared);
    if (carve != cudaSuccess)
        return carve;
    fabrik_planar_kernel<Real, FUSE_FK, OUT32, ZERO_ITER><<<grid, IKB_FABRIK_WARPS * 32, smem, stream>>>(a);
    return cudaGetLastError();
}
template <typename Real, bool FUSE_FK, bool OUT32>
cudaError_t launch_planar(const FabrikArgs &a, unsigned grid, cudaStream_t stream)
{
    return a.rc.zero_iter ? launch_planar_z<Real, FUSE_FK, OUT32, true>(a, grid, stream)
                          : launch_planar_z<Real, FUSE_FK, OUT32, false>(a, grid, stream);
}
}  // namespace

// work_counter: the chunk counter of this launch (reset here).
cudaError_t ikb_launch_fabrik_planar(const void *xyz, int xyz_f64, long long n, long long index_base,
                                     void *angles, int angles_f64, int *iters, void *fk_err, int fk_stats,
                                     int precision, IkbDeviceStats *stats, unsigned long long *work_counter,
                                     const IkbRobot &rc, int num_sms, cudaStream_t stream)
{
    if (n <= 0)
        return cudaSuccess;
    FabrikArgs a;
    a.xyz = xyz; a.xyz_f64 = xyz_f64; a.n = n; a.index_base = index_base;
    a.angles = angles; a.angles_f64 = angles_f64; a.iters = iters;
    a.fk_err = fk_err; a.fk_stats = fk_stats;
    a.stats = stats; a.work_counter = work_counter; a.rc = rc;
    cudaError_t err = cudaMemsetAsync(work_counter, 0, sizeof(unsigned long long), stream);
    if (err != cudaSuccess)
        return err;
    const bool fuse = fk_err != nullptr || fk_stats != 0;  // the caller checked rc.fk_planar_tail
    // out-of-reach targets run in lockstep batches (see is_far); IKB_FABRIK_SPLIT=0 sends every target through the
    // lane-refill loop instead (same arithmetic, value-identical results: tests/test_gpu_fabrik.py)
    static const bool split_enabled = [] { const char *v = std::getenv("IKB_FABRIK_SPLIT"); return !v || v[0] != '0'; }();
    a.far_thr2 = -1.0;
    if (split_enabled && !rc.zero_iter && rc.max_iter >= 8) {
        const double reach = rc.links[1] + rc.links[2] + rc.links[3];
        const double thr = reach + rc.tol + 1e-6 * (1.0 + reach);  // margin >> the rounding of |f2 - S| <= d1 + d2
        a.far_thr2 = thr * thr;
    }
    // persistent grid: resident CTAs per SM x SM count, trimmed for small batches
    const int per_cta = IKB_FABRIK_WARPS * 32;
    long long grid = (long long)num_sms * IKB_FABRIK_MIN_CTAS;
    const long long want = (n + per_cta - 1) / per_cta;
    if (want < grid)
        grid = want;
    // kernel variant = (iterate precision, fused FK error, output precision); the trigonometric tail of the angle
    // extraction follows the output buffer's precision (see acos_f32)
#define IKB_PICK(REAL)                                                                           \
    (fuse ? (angles_f64 ? launch_planar<REAL, true, false>(a, (unsigned)grid, stream)            \
                        : launch_planar<REAL, true, true>(a, (unsigned)grid, stream))            \
          : (angles_f64 ? launch_planar<REAL, false, false>(a, (unsigned)grid, stream)           \
                        : launch_planar<REAL, false, true>(a, (unsigned)grid, stream)))
    return precision == IKB_FABRIK_F32 ? IKB_PICK(float) : IKB_PICK(double);
#undef IKB_PICK
}

cudaError_t ikb_launch_fabrik_generic_ikine(const void *xyz, int xyz_f64, long long n, long long index_base,
                                            void *angles, int angles_f64, int *iters, IkbDeviceStats *stats,
                                            const IkbRobot &rc, cudaStream_t stream)
{
    if (n <= 0)
        return cudaSuccess;
    FabrikGenericIkineArgs a;
    a.xyz = xyz; a.xyz_f64 = xyz_f64; a.n = n; a.index_base = index_base; a.angles = angles;
    a.angles_f64 = angles_f64; a.iters = iters; a.stats = stats; a.rc = rc;
    fabrik_generic_ikine_kernel<<<(unsigned)((n + 127) / 128), 128, 0, stream>>>(a);
    return cudaGetLastError();
}

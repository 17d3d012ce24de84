// fk.cu -- K0 (workspace-limit check), K3 (batched DH forward kinematics / position error) and the
// FMA-pipe microbenchmark (sm_100a).
//
// K3 replaces reference ForwardKinematics.fkine (forward.py:73-94) for batches:
//   T = prod_i Rz(theta_i) Tz(eps_i) Tx(a_i) Rx(alpha_i)                      (forward.py:62-70)
// Only what callers read is produced in the batched form -- the end-effector position T[0:3, 3]
// (cli.py:60, inverse.py:130, tests/forward_unit.py:30) and ||pos - target||.  fk_transforms_kernel
// returns all four cumulative 4x4 matrices (or the joint origins) for the (T, [T1..T4]) return value of fkine, and
// from the same chain the arm Jacobian and its manipulability.
// HBM-bound: 16 B angles + 12 B target in, 4 B error out per row (fp32 buffers).
#include <cstdlib>

#include "fk_device.cuh"

namespace {

struct FkArgs {
    const void *angles;
    int angles_f64;
    long long n;
    long long index_base;
    void *pos_out;        // nullable, n x 3 (angles dtype)
    const void *targets;  // nullable, n x 3 (xyz dtype)
    int xyz_f64;
    void *err_out;        // nullable, n (angles dtype)
    IkbDeviceStats *stats;
    IkbRobot rc;
};

// FK_ROWS rows per thread and loop trip (2 rows x 4 resident CTAs measured best), all of their loads issued
// before any arithmetic: at 28 B of
// input per row the kernel needs ~5 MB in flight chip-wide to cover HBM latency.
#ifndef FK_ROWS
#define FK_ROWS 2
#endif
#ifndef FK_MINB
#define FK_MINB 4
#endif

// Real = dtype of the angle / position / error buffers, XYZ_F64 = dtype of the target buffer: both compile-time, so the
// row loop carries no dtype branches.
template <typename Real, bool XYZ_F64>
__global__ void __launch_bounds__(256, FK_MINB) fk_kernel(const FkArgs a)
{
    constexpr bool ANG_F64 = sizeof(Real) == 8;
    const long long stride = (long long)gridDim.x * blockDim.x;
    double err_sum = 0.0;
    unsigned err_cnt = 0;
    bool alpha_ok = true;
#pragma unroll
    for (int j = 0; j < 4; ++j)
        alpha_ok &= !(a.rc.alpha[j] < -6.283185307179586) & !(a.rc.alpha[j] > 6.283185307179586);
    for (long long base = (long long)blockIdx.x * blockDim.x + threadIdx.x; base < a.n; base += stride * FK_ROWS) {
        Real err_part = 0;  // per-trip partial sum in the working precision, folded into the fp64 total once
        Real th[FK_ROWS][4];
        Real tg[FK_ROWS][3];
#pragma unroll
        for (int u = 0; u < FK_ROWS; ++u) {
            const long long i = base + u * stride;
            if (i < a.n) {
                if (ANG_F64) {
                    const double2 *p = reinterpret_cast<const double2 *>(a.angles) + 2 * i;
                    const double2 v0 = __ldg(p), v1 = __ldg(p + 1);
                    th[u][0] = (Real)v0.x; th[u][1] = (Real)v0.y; th[u][2] = (Real)v1.x; th[u][3] = (Real)v1.y;
                } else {
                    const float4 v = __ldg(reinterpret_cast<const float4 *>(a.angles) + i);
                    th[u][0] = (Real)v.x; th[u][1] = (Real)v.y; th[u][2] = (Real)v.z; th[u][3] = (Real)v.w;
                }
                if (a.targets) {
                    if (XYZ_F64) {
                        const double *p = reinterpret_cast<const double *>(a.targets) + 3 * i;
                        tg[u][0] = (Real)__ldg(p); tg[u][1] = (Real)__ldg(p + 1); tg[u][2] = (Real)__ldg(p + 2);
                    } else {  // no detour through double for fp32 buffers
                        const float *p = reinterpret_cast<const float *>(a.targets) + 3 * i;
                        tg[u][0] = (Real)__ldg(p); tg[u][1] = (Real)__ldg(p + 1); tg[u][2] = (Real)__ldg(p + 2);
                    }
                }
            }
        }
#pragma unroll
        for (int u = 0; u < FK_ROWS; ++u) {
            const long long i = base + u * stride;
            if (i >= a.n)
                break;
            Real px, py, pz;
            const bool ok = fk_position<Real>(a.rc, th[u], px, py, pz) & alpha_ok;
            if (!ok) {
                px = py = pz = (Real)__int_as_float(0x7fc00000);
                atomicMin(&a.stats->first_fk_angle_range, a.index_base + i);
            }
            if (a.pos_out) {
                if (ANG_F64) {
                    double *o = reinterpret_cast<double *>(a.pos_out) + 3 * i;
                    o[0] = px; o[1] = py; o[2] = pz;
                } else {
                    float *o = reinterpret_cast<float *>(a.pos_out) + 3 * i;
                    o[0] = (float)px; o[1] = (float)py; o[2] = (float)pz;
                }
            }
            if (a.targets) {
                const Real dx = px - tg[u][0], dy = py - tg[u][1], dz = pz - tg[u][2];
                const Real err = sqrt(dx * dx + dy * dy + dz * dz);
                if (a.err_out) {
                    if (ANG_F64)
                        reinterpret_cast<double *>(a.err_out)[i] = err;
                    else
                        reinterpret_cast<float *>(a.err_out)[i] = (float)err;
                }
                if (isfinite(err)) {
                    err_part += err;
                    ++err_cnt;
                }
            }
        }
        err_sum += (double)err_part;
    }
    if (a.targets) {
        err_sum = ikb_warp_sum(err_sum);
        err_cnt = ikb_warp_sum(err_cnt);
        if ((threadIdx.x & 31) == 0 && err_cnt) {
            atomicAdd(&a.stats->sum_fk_error, err_sum);
            atomicAdd(&a.stats->n_fk_error, (unsigned long long)err_cnt);
        }
    }
}

// ---- the common case at HBM speed: fp32 buffers, closed-form arm, position error only ----------------------------------
// The generic kernel above is bound by instruction issue (194 instructions per row, 69 % of the HBM roofline).  Here a
// thread takes two ADJACENT rows per trip -- angles as two 16-byte loads, the six target floats as three 8-byte loads,
// the two errors as one 8-byte store -- and evaluates the eight sin/cos pairs two at a time on the packed fp32 pipe
// (ikb_sincos2: bit-identical to the scalar code, about half its instructions).  The chain arithmetic is the same inline
// function as everywhere else, so the errors are the ones the generic kernel and the solvers' fused epilogues produce.
#ifndef FK_PAIR_MINB
#define FK_PAIR_MINB 3  // 80 registers: room for the software-pipelined loads without spills (4 CTAs: 64 registers, spills)
#endif
__global__ void __launch_bounds__(256, FK_PAIR_MINB) fk_error_pairs_kernel(const FkArgs a)
{
    const long long n_pairs = a.n >> 1;  // the odd last row (if any) is handled by one thread after the loop
    const long long stride = (long long)gridDim.x * blockDim.x;
    const float *k = a.rc.fkc_f;
    const float TWO_PI = IKB_TWO_PI_F32;
    double err_sum = 0.0;
    unsigned err_cnt = 0;
    const float4 *ang = reinterpret_cast<const float4 *>(a.angles);
    const float2 *tgt = reinterpret_cast<const float2 *>(a.targets);
    float2 *out = reinterpret_cast<float2 *>(a.err_out);
    auto row_error = [&](const float (&s)[4], const float (&c)[4], const float4 &th, float tx, float ty, float tz) {
        float px, py, pz;
        fk_planar_tail_position<float>(s, c, k[0], k[1], k[2], k[3], k[4], k[5], k[6], k[7], px, py, pz);
        const float dx = px - tx, dy = py - ty, dz = pz - tz;
        // sqrt.approx (one MUFU, 1 ulp) instead of the IEEE root with its fix-up branch: the error is a diagnostic
        // in metres, and the kernel is bound by instruction issue
        float err;
        asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(err) : "f"(dx * dx + dy * dy + dz * dz));
        const bool ok = !(fabsf(th.x) > TWO_PI) & !(fabsf(th.y) > TWO_PI) & !(fabsf(th.z) > TWO_PI) & !(fabsf(th.w) > TWO_PI);
        return ok ? err : __int_as_float(0x7fc00000);
    };
#ifndef FK_PAIR_PREFETCH
#define FK_PAIR_PREFETCH 1
#endif
    long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    float4 n_th0, n_th1;
    float2 n_t0, n_t1, n_t2;
    if (FK_PAIR_PREFETCH && p < n_pairs) {  // software pipeline: the next trip's loads are in flight during this trip's arithmetic
        n_th0 = __ldg(ang + 2 * p); n_th1 = __ldg(ang + 2 * p + 1);
        n_t0 = __ldg(tgt + 3 * p); n_t1 = __ldg(tgt + 3 * p + 1); n_t2 = __ldg(tgt + 3 * p + 2);
    }
    for (; p < n_pairs; p += stride) {
        float4 th0, th1;
        float2 t0, t1, t2;
        if (FK_PAIR_PREFETCH) {
            th0 = n_th0; th1 = n_th1; t0 = n_t0; t1 = n_t1; t2 = n_t2;
            const long long pn = p + stride;
            if (pn < n_pairs) {
                n_th0 = __ldg(ang + 2 * pn); n_th1 = __ldg(ang + 2 * pn + 1);
                n_t0 = __ldg(tgt + 3 * pn); n_t1 = __ldg(tgt + 3 * pn + 1); n_t2 = __ldg(tgt + 3 * pn + 2);
            }
        } else {
            th0 = __ldg(ang + 2 * p); th1 = __ldg(ang + 2 * p + 1);
            t0 = __ldg(tgt + 3 * p); t1 = __ldg(tgt + 3 * p + 1); t2 = __ldg(tgt + 3 * p + 2);
        }
        float s0[4], c0[4], s1[4], c1[4];
        ikb_sincos2(th0.x, th1.x, s0[0], c0[0], s1[0], c1[0]);
        ikb_sincos2(th0.y, th1.y, s0[1], c0[1], s1[1], c1[1]);
        ikb_sincos2(th0.z, th1.z, s0[2], c0[2], s1[2], c1[2]);
        ikb_sincos2(th0.w, th1.w, s0[3], c0[3], s1[3], c1[3]);
        const float e0 = row_error(s0, c0, th0, t0.x, t0.y, t1.x);
        const float e1 = row_error(s1, c1, th1, t1.y, t2.x, t2.y);
        if (e0 != e0)  // NaN from the angle guard of forward.py:23-25 (or from NaN input: then the row index is not recorded)
            if (fabsf(th0.x) > TWO_PI || fabsf(th0.y) > TWO_PI || fabsf(th0.z) > TWO_PI || fabsf(th0.w) > TWO_PI)
                atomicMin(&a.stats->first_fk_angle_range, a.index_base + 2 * p);
        if (e1 != e1)
            if (fabsf(th1.x) > TWO_PI || fabsf(th1.y) > TWO_PI || fabsf(th1.z) > TWO_PI || fabsf(th1.w) > TWO_PI)
                atomicMin(&a.stats->first_fk_angle_range, a.index_base + 2 * p + 1);
        if (out)
            out[p] = make_float2(e0, e1);
        float part = 0.f;
        if (isfinite(e0)) { part += e0; ++err_cnt; }
        if (isfinite(e1)) { part += e1; ++err_cnt; }
        err_sum += (double)part;
    }
    if ((a.n & 1) && blockIdx.x == 0 && threadIdx.x == 0) {  // the odd last row: scalar code, same arithmetic
        const long long i = a.n - 1;
        const float4 v = __ldg(ang + i);
        const float th[4] = {v.x, v.y, v.z, v.w};
        const float *t = reinterpret_cast<const float *>(a.targets) + 3 * i;
        const float e = ikb_fk_error_planar_tail<float>(th, __ldg(t), __ldg(t + 1), __ldg(t + 2), k[0], k[1], k[2], k[3], k[4],
                                                        k[5], k[6], k[7]);
        if (e != e && (fabsf(v.x) > TWO_PI || fabsf(v.y) > TWO_PI || fabsf(v.z) > TWO_PI || fabsf(v.w) > TWO_PI))
            atomicMin(&a.stats->first_fk_angle_range, a.index_base + i);
        if (a.err_out)
            reinterpret_cast<float *>(a.err_out)[i] = e;
        if (isfinite(e)) { err_sum += (double)e; ++err_cnt; }
    }
    err_sum = ikb_warp_sum(err_sum);
    err_cnt = ikb_warp_sum(err_cnt);
    if ((threadIdx.x & 31) == 0 && err_cnt) {
        atomicAdd(&a.stats->sum_fk_error, err_sum);
        atomicAdd(&a.stats->n_fk_error, (unsigned long long)err_cnt);
    }
}

// ---- the same rows through an asynchronous-copy ring -------------------------------------------------------------------
// With the instruction count down, what keeps the pair kernel at ~0.8 of the HBM roofline is bytes in flight: a thread
// holds its next loads in registers (56 B) and 24 warps per SM make 43 KB.  Here a WARP owns 32 consecutive pairs per
// trip (1 KB of angles + 768 B of targets, both contiguous) and streams them global -> shared with cp.async through a
// ring of FK_STREAM_STAGES trips, no registers involved: up to 3.5 KB per warp in flight, 32 warps per SM.  Arithmetic
// and results are those of fk_error_pairs_kernel.  Needs 16-byte aligned buffers; the last partial trip goes to the
// pair kernel.
#ifndef FK_STREAM_STAGES
#define FK_STREAM_STAGES 3
#endif
#define FK_STREAM_WARPS 8
struct FkStage {
    float4 ang[64];   // 32 pairs x 2 rows
    float2 tgt[96];   // 32 pairs x 6 floats
};

__device__ __forceinline__ void cp_async16(void *smem, const void *gmem)
{
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((unsigned)__cvta_generic_to_shared(smem)), "l"(gmem)
                 : "memory");
}

__global__ void __launch_bounds__(FK_STREAM_WARPS * 32, 4) fk_error_stream_kernel(const FkArgs a, long long n_trips)
{
    __shared__ __align__(16) FkStage s_ring[FK_STREAM_WARPS][FK_STREAM_STAGES];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    FkStage *ring = s_ring[warp];
    const long long w = (long long)blockIdx.x * FK_STREAM_WARPS + warp, W = (long long)gridDim.x * FK_STREAM_WARPS;
    const float *k = a.rc.fkc_f;
    const float TWO_PI = IKB_TWO_PI_F32;
    const char *ang = reinterpret_cast<const char *>(a.angles);
    const char *tgt = reinterpret_cast<const char *>(a.targets);
    float2 *out = reinterpret_cast<float2 *>(a.err_out);
    double err_sum = 0.0;
    unsigned err_cnt = 0;
    auto issue = [&](long long trip, int stage) {
        if (trip < n_trips) {
            const char *ga = ang + trip * 1024, *gt = tgt + trip * 768;
            char *sa = reinterpret_cast<char *>(ring[stage].ang), *st = reinterpret_cast<char *>(ring[stage].tgt);
            cp_async16(sa + lane * 16, ga + lane * 16);
            cp_async16(sa + 512 + lane * 16, ga + 512 + lane * 16);
            cp_async16(st + lane * 16, gt + lane * 16);
            if (lane < 16)
                cp_async16(st + 512 + lane * 16, gt + 512 + lane * 16);
        }
        asm volatile("cp.async.commit_group;" ::: "memory");  // one group per trip, possibly empty: the wait below counts groups
    };
    auto row_error = [&](const float (&s)[4], const float (&c)[4], const float4 &th, float tx, float ty, float tz) {
        float px, py, pz;
        fk_planar_tail_position<float>(s, c, k[0], k[1], k[2], k[3], k[4], k[5], k[6], k[7], px, py, pz);
        const float dx = px - tx, dy = py - ty, dz = pz - tz;
        float err;
        asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(err) : "f"(dx * dx + dy * dy + dz * dz));
        const bool ok = !(fabsf(th.x) > TWO_PI) & !(fabsf(th.y) > TWO_PI) & !(fabsf(th.z) > TWO_PI) & !(fabsf(th.w) > TWO_PI);
        return ok ? err : __int_as_float(0x7fc00000);
    };
#pragma unroll
    for (int sidx = 0; sidx < FK_STREAM_STAGES - 1; ++sidx)
        issue(w + sidx * W, sidx);
    int stage = 0;
    for (long long trip = w; trip < n_trips; trip += W) {
        int ahead = stage + FK_STREAM_STAGES - 1;
        ahead -= ahead >= FK_STREAM_STAGES ? FK_STREAM_STAGES : 0;
        issue(trip + (FK_STREAM_STAGES - 1) * W, ahead);
        asm volatile("cp.async.wait_group %0;" ::"n"(FK_STREAM_STAGES - 1) : "memory");
        __syncwarp();
        const float4 th0 = ring[stage].ang[2 * lane], th1 = ring[stage].ang[2 * lane + 1];
        const float2 t0 = ring[stage].tgt[3 * lane], t1 = ring[stage].tgt[3 * lane + 1], t2 = ring[stage].tgt[3 * lane + 2];
        __syncwarp();  // every lane has read its rows: the stage may be refilled by the next issue()
        float s0[4], c0[4], s1[4], c1[4];
        ikb_sincos2(th0.x, th1.x, s0[0], c0[0], s1[0], c1[0]);
        ikb_sincos2(th0.y, th1.y, s0[1], c0[1], s1[1], c1[1]);
        ikb_sincos2(th0.z, th1.z, s0[2], c0[2], s1[2], c1[2]);
        ikb_sincos2(th0.w, th1.w, s0[3], c0[3], s1[3], c1[3]);
        const float e0 = row_error(s0, c0, th0, t0.x, t0.y, t1.x);
        const float e1 = row_error(s1, c1, th1, t1.y, t2.x, t2.y);
        const long long p = trip * 32 + lane;
        if (e0 != e0)
            if (fabsf(th0.x) > TWO_PI || fabsf(th0.y) > TWO_PI || fabsf(th0.z) > TWO_PI || fabsf(th0.w) > TWO_PI)
                atomicMin(&a.stats->first_fk_angle_range, a.index_base + 2 * p);
        if (e1 != e1)
            if (fabsf(th1.x) > TWO_PI || fabsf(th1.y) > TWO_PI || fabsf(th1.z) > TWO_PI || fabsf(th1.w) > TWO_PI)
                atomicMin(&a.stats->first_fk_angle_range, a.index_base + 2 * p + 1);
        if (out)
            out[p] = make_float2(e0, e1);
        float part = 0.f;
        if (isfinite(e0)) { part += e0; ++err_cnt; }
        if (isfinite(e1)) { part += e1; ++err_cnt; }
        err_sum += (double)part;
        stage = stage + 1 == FK_STREAM_STAGES ? 0 : stage + 1;
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    err_sum = ikb_warp_sum(err_sum);
    err_cnt = ikb_warp_sum(err_cnt);
    if (lane == 0 && err_cnt) {
        atomicAdd(&a.stats->sum_fk_error, err_sum);
        atomicAdd(&a.stats->n_fk_error, (unsigned long long)err_cnt);
    }
}

// ---- all four cumulative DH matrices of a batch (forward.py:79-94) -----------------------------------------------------
// Row r of T_j = T_{j-1} D_j depends only on row r of T_{j-1} and on D_j, so one angle set is served by four lanes (a
// quad): lane r computes sincos of joint r, the quad exchanges the four (sin, cos) pairs with shuffles, and lane r
// carries row r of T_1..T_4.  Every matrix element is the expression the single-pose path has always used (fp64,
// default contraction: `acc += T * D` in m order), so a row's bits do not depend on the batch it is in.
//
// The workload is store-bound (fp64: 32 B of angles in, 512 B of matrices out per angle set).  A CTA computes a tile of
// FKT_ROWS consecutive angle sets into shared memory -- one contiguous span of the output -- and one thread sends it
// to global memory with a 1-D bulk copy (cp.async.bulk, the TMA engine) while the CTA computes the next tile into the
// other buffer.  An output base that is not 16-byte aligned takes coalesced element stores from the same tile instead.

// row r of T_j from row r of T_{j-1} (`t`) and D_j = Rz(theta) Tz(eps) Tx(a) Rx(alpha) of joint j
__device__ __forceinline__ void fk_dh_step_row(const double (&t)[4], double s, double c, double ca, double sa, double aj,
                                               double ej, double (&out)[4])
{
    const double D[16] = {c, -s * ca, s * sa, aj * c,
                          s, c * ca, -c * sa, aj * s,
                          0, sa, ca, ej,
                          0, 0, 0, 1};
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        double acc = 0;
#pragma unroll
        for (int m = 0; m < 4; ++m)
            acc += t[m] * D[4 * m + q];
        out[q] = acc;
    }
}

// Row r of the 3 x 4 position Jacobian, for the quad lane r that carries row r of T_1..T_4 (zs[j], ps[j]: element r
// of z_j and p_j, columns 2 and 3 of T_j, with T_0 = I; ps[4] = element r of p_4).  Column i-1 (joint i) is
// z_{i-1} x (p_4 - p_{i-1}).  Lane r < 3 computes element r: z[r+1] * d[r+2] - z[r+2] * d[r+1] (indices mod 3: y*z' -
// z*y' for x, ...), with the operands of the other two elements fetched from their lanes.  Every operation is
// explicitly rounded (no contraction), so a NumPy restatement on fkine_batch's matrices reproduces the bits.  Lane 3
// computes an unused value.  All four lanes of the quad must call it (quad shuffles).
__device__ __forceinline__ void fk_quad_position_jacobian_row(int r, const double (&zs)[4], const double (&ps)[5],
                                                              double (&lin)[4])
{
    const int r1 = r < 2 ? r + 1 : r - 2, r2 = r == 0 ? 2 : r - 1;
    const double p4a = __shfl_sync(IKB_FULL_MASK, ps[4], r1, 4), p4b = __shfl_sync(IKB_FULL_MASK, ps[4], r2, 4);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        // z_0 = (0, 0, 1) and p_0 = 0 are constants
        const double za = k ? __shfl_sync(IKB_FULL_MASK, zs[k], r1, 4) : (r1 == 2 ? 1.0 : 0.0);
        const double zb = k ? __shfl_sync(IKB_FULL_MASK, zs[k], r2, 4) : (r2 == 2 ? 1.0 : 0.0);
        const double pa = k ? __shfl_sync(IKB_FULL_MASK, ps[k], r1, 4) : 0.0;
        const double pb = k ? __shfl_sync(IKB_FULL_MASK, ps[k], r2, 4) : 0.0;
        lin[k] = __dsub_rn(__dmul_rn(za, __dsub_rn(p4b, pb)), __dmul_rn(zb, __dsub_rn(p4a, pa)));
    }
}

__device__ __forceinline__ unsigned fkt_smem_u32(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }

// shared -> global 1-D bulk copy (SASS: UBLKCP); dst 16-byte aligned, bytes a multiple of 16
__device__ __forceinline__ void fkt_bulk_store(void *dst, const void *src, unsigned bytes)
{
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(fkt_smem_u32(src)),
                 "r"(bytes)
                 : "memory");
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}

constexpr int FKT_ROWS = 64;              // angle sets per tile
constexpr int FKT_THREADS = 4 * FKT_ROWS;  // one quad per angle set

// What fk_transforms_kernel writes per angle set (the tile row, in elements):
//   FKT_MATRICES      T_1..T_4, 4 x 4 x 4 (64)
//   FKT_JOINTS        column 3 of T_1..T_4, 4 x 3 (12)
//   FKT_JAC_GEOMETRIC the 6 x 4 geometric Jacobian (24)
//   FKT_JAC_POSITION  its rows 0-2, the 3 x 4 position Jacobian (12)
//   FKT_MANIP_ONLY    no tile; only the manipulability below
// The Jacobian kinds may also write the manipulability w (template MANIP), one element per angle set straight from the
// quad to `manip`.
enum FktKind { FKT_MATRICES, FKT_JOINTS, FKT_JAC_GEOMETRIC, FKT_JAC_POSITION, FKT_MANIP_ONLY };

constexpr int fkt_row_elems(int kind)
{
    return kind == FKT_MATRICES ? 64 : kind == FKT_JAC_GEOMETRIC ? 24 : kind == FKT_MANIP_ONLY ? 0 : 12;
}

// Real: dtype of angles and outputs.  Dynamic shared memory: two tiles of FKT_ROWS * fkt_row_elems(KIND) elements.
template <typename Real, int KIND, bool MANIP>
__global__ void __launch_bounds__(FKT_THREADS) fk_transforms_kernel(const Real *__restrict__ angles, long long n,
                                                                    long long index_base, Real *out,
                                                                    IkbDeviceStats *stats, const IkbRobot rc,
                                                                    Real *manip)
{
    constexpr bool JOINTS = KIND == FKT_JOINTS;
    constexpr bool JAC = KIND >= FKT_JAC_GEOMETRIC;
    constexpr int ROW_ELEMS = fkt_row_elems(KIND);
    constexpr bool TILED = ROW_ELEMS > 0;
    constexpr int TILE_ELEMS = FKT_ROWS * ROW_ELEMS;
    extern __shared__ __align__(128) unsigned char fkt_smem[];
    Real *const tiles = reinterpret_cast<Real *>(fkt_smem);
    const double TWO_PI = 6.283185307179586;
    const int tid = threadIdx.x, r = tid & 3, lrow = tid >> 2;
    const int odd = lrow & 1;
    const bool bulk = TILED && ((uintptr_t)out & 15) == 0;  // every row size here is a multiple of 16 bytes
    const bool alpha_bad = rc.alpha[r] < -TWO_PI || rc.alpha[r] > TWO_PI;
    const long long n_tiles = (n + FKT_ROWS - 1) / FKT_ROWS;
    int buf = 0;
    for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, buf ^= 1) {
        const long long row0 = tile * FKT_ROWS;
        const int rows = (int)(n - row0 < FKT_ROWS ? n - row0 : FKT_ROWS);
        const bool live = lrow < rows;
        const double th = live ? (double)__ldg(angles + 4 * (row0 + lrow) + r) : 0.0;  // a warp reads 256 or 128 B
        // angle guard of forward.py:23-25 (NaN passes): the lowest offending row of the warp, one atomic per warp
        const unsigned bad = __ballot_sync(IKB_FULL_MASK, live && (th < -TWO_PI || th > TWO_PI || alpha_bad));
        if (bad && (tid & 31) == __ffs(bad) - 1)
            atomicMin(&stats->first_fk_angle_range, index_base + row0 + lrow);
        double s, c;
        sincos(th, &s, &c);
        // the bulk copy that last read this buffer (two tiles ago) must be done reading it
        if (bulk && tid == 0)
            asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
        if (TILED)
            __syncthreads();
        Real *const dst = tiles + buf * TILE_ELEMS + lrow * ROW_ELEMS;
        double t[4] = {r == 0 ? 1.0 : 0.0, r == 1 ? 1.0 : 0.0, r == 2 ? 1.0 : 0.0, r == 3 ? 1.0 : 0.0};
        double prev[4];
        double zs[4], ps[5];  // Jacobian kinds: element r of z_j and p_j, columns 2 and 3 of T_j (T_0 = I)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const double sj = __shfl_sync(IKB_FULL_MASK, s, j, 4), cj = __shfl_sync(IKB_FULL_MASK, c, j, 4);
            double nr[4];
            zs[j] = t[2];
            ps[j] = t[3];
            fk_dh_step_row(t, sj, cj, rc.cos_alpha[j], rc.sin_alpha[j], rc.a[j], rc.eps[j], nr);
            if (!JAC && live) {
                // Stores are arranged so that the 8 lanes of a 16-byte shared-memory phase (two angle sets) hit 8
                // different bank groups: an unrotated 512-B (or 256-B) row stride would put them all in one.
                if (JOINTS) {
                    if (r < 3)
                        dst[3 * j + r] = (Real)nr[3];
                } else if (sizeof(Real) == 8) {
                    // row r of T_j is two 16-byte halves; odd angle sets store the second half first
                    double2 *p = reinterpret_cast<double2 *>(dst + 16 * j + 4 * r);
                    const double2 lo = make_double2(nr[0], nr[1]), hi = make_double2(nr[2], nr[3]);
                    p[odd] = odd ? hi : lo;
                    p[odd ^ 1] = odd ? lo : hi;
                } else if (j & 1) {
                    // row r of T_j is one float4; T_{j-1} and T_j go out together, odd angle sets T_j first
                    float4 *p = reinterpret_cast<float4 *>(dst + 4 * r);
                    const float4 a = make_float4((float)prev[0], (float)prev[1], (float)prev[2], (float)prev[3]);
                    const float4 b = make_float4((float)nr[0], (float)nr[1], (float)nr[2], (float)nr[3]);
                    p[4 * (j - 1 + odd)] = odd ? b : a;
                    p[4 * (j - odd)] = odd ? a : b;
                }
            }
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                prev[q] = nr[q];
                t[q] = nr[q];
            }
        }
        ps[4] = t[3];
        if (JAC) {
            double lin[4];
            fk_quad_position_jacobian_row(r, zs, ps, lin);
            if (MANIP) {
                // w^2 = sum over the four 3-column subsets of det^2 (Cauchy-Binet).  Lane r takes the subset without
                // column 3 - r: (0,1,2), (0,1,3), (0,2,3), (1,2,3) for r = 0..3, det = a . (b x c), b x c in the
                // order of the linear rows, the dot product summed (x + y) + z; then w = sqrt((s0 + s1) + (s2 + s3)).
                double J[3][4];
#pragma unroll
                for (int q = 0; q < 3; ++q)
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                        J[q][k] = __shfl_sync(IKB_FULL_MASK, lin[k], q, 4);
                double a[3], b[3], cc[3];
#pragma unroll
                for (int q = 0; q < 3; ++q) {
                    a[q] = r == 3 ? J[q][1] : J[q][0];
                    b[q] = r >= 2 ? J[q][2] : J[q][1];
                    cc[q] = r >= 1 ? J[q][3] : J[q][2];
                }
                const double m0 = __dsub_rn(__dmul_rn(b[1], cc[2]), __dmul_rn(b[2], cc[1]));
                const double m1 = __dsub_rn(__dmul_rn(b[2], cc[0]), __dmul_rn(b[0], cc[2]));
                const double m2 = __dsub_rn(__dmul_rn(b[0], cc[1]), __dmul_rn(b[1], cc[0]));
                const double det = __dadd_rn(__dadd_rn(__dmul_rn(a[0], m0), __dmul_rn(a[1], m1)), __dmul_rn(a[2], m2));
                double w2 = __dmul_rn(det, det);
                w2 = __dadd_rn(w2, __shfl_xor_sync(IKB_FULL_MASK, w2, 1, 4));  // lanes 0, 1: s0 + s1 (addition commutes)
                w2 = __dadd_rn(w2, __shfl_xor_sync(IKB_FULL_MASK, w2, 2, 4));
                if (live && r == 0)
                    manip[row0 + lrow] = (Real)__dsqrt_rn(w2);
            }
            if (TILED && live && r < 3) {
                // row r (linear) and row 3 + r (angular: z_{i-1}, i.e. element r of zs) of the 6 x 4 Jacobian.
                // As for the matrices, the stores are arranged so that the two angle sets of a 16-byte shared-memory
                // phase hit distinct bank groups.
                if (sizeof(Real) == 8) {
                    // each row is two 16-byte halves; odd angle sets store the second half first
                    double2 *pl = reinterpret_cast<double2 *>(dst + 4 * r);
                    const double2 l0 = make_double2(lin[0], lin[1]), l1 = make_double2(lin[2], lin[3]);
                    pl[odd] = odd ? l1 : l0;
                    pl[odd ^ 1] = odd ? l0 : l1;
                    if (KIND == FKT_JAC_GEOMETRIC) {
                        double2 *pa = reinterpret_cast<double2 *>(dst + 12 + 4 * r);
                        const double2 a0 = make_double2(zs[0], zs[1]), a1 = make_double2(zs[2], zs[3]);
                        pa[odd] = odd ? a1 : a0;
                        pa[odd ^ 1] = odd ? a0 : a1;
                    }
                } else {
                    float4 *q = reinterpret_cast<float4 *>(dst);
                    const float4 L = make_float4((float)lin[0], (float)lin[1], (float)lin[2], (float)lin[3]);
                    if (KIND == FKT_JAC_POSITION) {
                        q[r] = L;  // 48-B rows: the two angle sets of a phase already cover six distinct bank groups
                    } else {
                        // 96-B rows, six 16-B slots: lane 2 of an odd angle set stores its angular row first
                        const float4 A = make_float4((float)zs[0], (float)zs[1], (float)zs[2], (float)zs[3]);
                        const bool swap = odd && r == 2;
                        q[swap ? 3 + r : r] = swap ? A : L;
                        q[swap ? r : 3 + r] = swap ? L : A;
                    }
                }
            }
        }
        if (TILED) {
            const Real *src = tiles + buf * TILE_ELEMS;
            Real *gdst = out + row0 * ROW_ELEMS;
            if (bulk) {
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // make the stores visible to the copy engine
                __syncthreads();
                if (tid == 0)
                    fkt_bulk_store(gdst, src, (unsigned)(rows * ROW_ELEMS * sizeof(Real)));
            } else {
                __syncthreads();
                for (int w = tid; w < rows * ROW_ELEMS; w += FKT_THREADS)
                    gdst[w] = src[w];
            }
        }
    }
    if (bulk && tid == 0)
        asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}

// ---- damped-least-squares refinement of joint angles onto position targets ---------------------------------------
// One quad per row, as in fk_transforms_kernel: lane r holds joint r's angle, runs the chain with fk_dh_step_row and
// forms the position Jacobian with fk_quad_position_jacobian_row, so p_4 and Jv are the bits of joint_positions and
// jacobian_batch(..., "position").  After the chain every lane of the quad holds all of Jv, p_4 and e, and solves the
// 3 x 3 damped system redundantly (explicitly rounded fp64 in the order of include/ikb200.h); lane k applies
// Delta theta_k.  Iteration counts are bimodal (a few steps from a good seed, max_iter for a target out of reach), so
// the warps are persistent: a quad whose row finishes stores it and takes the next row, one atomicAdd per warp and
// trip on the work counter.  Rows finish out of order, so each quad stores its own row (one 32-B or 16-B angle row).
struct DlsArgs {
    const void *xyz;     // n x 3, xyz dtype
    int xyz_f64;
    const void *seed;    // n_seed x 4 (n_seed 1 or n), angles dtype; may equal angles_out when n_seed == n
    long long n_seed;
    void *angles_out;    // n x 4, angles dtype
    int *iters;          // nullable, n
    void *err_out;       // nullable, n (angles dtype)
    long long n;
    long long index_base;  // global row of row 0 (host pipeline chunks): the row numbers in the statistics
    double lam2;         // damping^2, rounded once
    double tol;
    int max_iter;
    IkbDeviceStats *stats;
    unsigned long long *work_counter;  // zero at launch
    IkbRobot rc;
};

constexpr int DLS_THREADS = 256;

template <typename Real>
__global__ void __launch_bounds__(DLS_THREADS) dls_refine_kernel(const DlsArgs a)
{
    const double TWO_PI = 6.283185307179586, PI = 3.141592653589793;
    const int lane = threadIdx.x & 31, r = lane & 3;
    const unsigned quads_below = (1u << (lane & ~3)) - 1u;  // lanes of the lower quads of this warp
    const bool alpha_bad = a.rc.alpha[r] < -TWO_PI || a.rc.alpha[r] > TWO_PI;
    double th = 0.0, tx = 0.0, ty = 0.0, tz = 0.0;
    long long row = 0;
    int k = 0;
    bool live = false, exhausted = false;
    unsigned long long n_solved = 0, sum_k = 0, capped = 0, n_err = 0;
    double err_sum = 0.0;
    long long first_limits = IKB_I64_MAX, first_range = IKB_I64_MAX;
    for (;;) {
        if (!exhausted) {  // refill: every quad without a row takes the next one
            const unsigned want = __ballot_sync(IKB_FULL_MASK, !live) & 0x11111111u;  // lane 0 of each idle quad
            if (want) {
                unsigned long long base = 0;
                if (lane == 0)
                    base = atomicAdd(a.work_counter, (unsigned long long)__popc(want));
                base = __shfl_sync(IKB_FULL_MASK, base, 0);
                if (!live) {
                    const long long rw = (long long)base + __popc(want & quads_below);
                    if (rw < a.n) {
                        row = rw;
                        k = 0;
                        live = true;
                        // plain loads: seed may be angles_out (in place), whose rows other quads are writing
                        th = (double)reinterpret_cast<const Real *>(a.seed)[4 * (a.n_seed == 1 ? 0 : rw) + r];
                        ikb_load_xyz(a.xyz, a.xyz_f64, rw, tx, ty, tz);
                        // the guards of fk_transforms_kernel (angles) and K0 (targets); NaN passes both
                        if (th < -TWO_PI || th > TWO_PI || alpha_bad)
                            first_range = min(first_range, a.index_base + rw);
                        if (ikb_out_of_limits(a.rc, tx, ty, tz))
                            first_limits = min(first_limits, a.index_base + rw);
                    }
                }
                exhausted = (long long)(base + __popc(want)) >= a.n;
            }
        }
        if (__ballot_sync(IKB_FULL_MASK, live) == 0)
            break;
        // the chain, at full warp width (quads without a row compute on stale registers and write nothing)
        double s, c;
        sincos(th, &s, &c);
        double t[4] = {r == 0 ? 1.0 : 0.0, r == 1 ? 1.0 : 0.0, r == 2 ? 1.0 : 0.0, r == 3 ? 1.0 : 0.0};
        double zs[4], ps[5];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const double sj = __shfl_sync(IKB_FULL_MASK, s, j, 4), cj = __shfl_sync(IKB_FULL_MASK, c, j, 4);
            double nr[4];
            zs[j] = t[2];
            ps[j] = t[3];
            fk_dh_step_row(t, sj, cj, a.rc.cos_alpha[j], a.rc.sin_alpha[j], a.rc.a[j], a.rc.eps[j], nr);
#pragma unroll
            for (int q = 0; q < 4; ++q)
                t[q] = nr[q];
        }
        ps[4] = t[3];
        double lin[4];
        fk_quad_position_jacobian_row(r, zs, ps, lin);
        double J[3][4];
#pragma unroll
        for (int q = 0; q < 3; ++q)
#pragma unroll
            for (int m = 0; m < 4; ++m)
                J[q][m] = __shfl_sync(IKB_FULL_MASK, lin[m], q, 4);
        const double ex = __dsub_rn(tx, __shfl_sync(IKB_FULL_MASK, ps[4], 0, 4));
        const double ey = __dsub_rn(ty, __shfl_sync(IKB_FULL_MASK, ps[4], 1, 4));
        const double ez = __dsub_rn(tz, __shfl_sync(IKB_FULL_MASK, ps[4], 2, 4));
        const double err = __dsqrt_rn(__dadd_rn(__dadd_rn(__dmul_rn(ex, ex), __dmul_rn(ey, ey)), __dmul_rn(ez, ez)));
        if (live && (err <= a.tol || k >= a.max_iter)) {  // quad-uniform: every lane holds the same err and k
            const long long o = 4 * row + r;
            reinterpret_cast<Real *>(a.angles_out)[o] = (Real)th;
            if (r == 0) {
                if (a.iters)
                    a.iters[row] = k;
                if (a.err_out)
                    reinterpret_cast<Real *>(a.err_out)[row] = (Real)err;
                ++n_solved;
                sum_k += (unsigned)k;
                capped += err <= a.tol ? 0u : 1u;  // NaN rows included
                if (isfinite(err)) {
                    err_sum += err;
                    ++n_err;
                }
            }
            live = false;
        }
        if (live) {
            // A = Jv Jv^T + lambda^2 I, element (i, j) summed as (j0 + j1) + (j2 + j3)
            double A[3][3];
#pragma unroll
            for (int i = 0; i < 3; ++i)
#pragma unroll
                for (int j = i; j < 3; ++j)
                    A[i][j] = __dadd_rn(__dadd_rn(__dmul_rn(J[i][0], J[j][0]), __dmul_rn(J[i][1], J[j][1])),
                                        __dadd_rn(__dmul_rn(J[i][2], J[j][2]), __dmul_rn(J[i][3], J[j][3])));
#pragma unroll
            for (int i = 0; i < 3; ++i)
                A[i][i] = __dadd_rn(A[i][i], a.lam2);
            // A y = e by LDL^T (no square root)
            const double l10 = __ddiv_rn(A[0][1], A[0][0]), l20 = __ddiv_rn(A[0][2], A[0][0]);
            const double d1 = __dsub_rn(A[1][1], __dmul_rn(l10, A[0][1]));
            const double t12 = __dsub_rn(A[1][2], __dmul_rn(l20, A[0][1]));
            const double l21 = __ddiv_rn(t12, d1);
            const double d2 = __dsub_rn(__dsub_rn(A[2][2], __dmul_rn(l20, A[0][2])), __dmul_rn(l21, t12));
            const double z1 = __dsub_rn(ey, __dmul_rn(l10, ex));
            const double z2 = __dsub_rn(__dsub_rn(ez, __dmul_rn(l20, ex)), __dmul_rn(l21, z1));
            const double y2 = __ddiv_rn(z2, d2);
            const double y1 = __dsub_rn(__ddiv_rn(z1, d1), __dmul_rn(l21, y2));
            const double y0 = __dsub_rn(__dsub_rn(__ddiv_rn(ex, A[0][0]), __dmul_rn(l10, y1)), __dmul_rn(l20, y2));
            // lane k: column k of Jv
            const double c0 = r == 0 ? J[0][0] : r == 1 ? J[0][1] : r == 2 ? J[0][2] : J[0][3];
            const double c1 = r == 0 ? J[1][0] : r == 1 ? J[1][1] : r == 2 ? J[1][2] : J[1][3];
            const double c2 = r == 0 ? J[2][0] : r == 1 ? J[2][1] : r == 2 ? J[2][2] : J[2][3];
            th = __dadd_rn(th, __dadd_rn(__dadd_rn(__dmul_rn(c0, y0), __dmul_rn(c1, y1)), __dmul_rn(c2, y2)));
            if (fabs(th) > PI)
                th = remainder(th, TWO_PI);  // exact: the angle stays inside the FK guard
            ++k;
        }
    }
    // statistics: one atomic per warp and counter (lane 0 of each quad counted its rows)
    n_solved = ikb_warp_sum(n_solved);
    sum_k = ikb_warp_sum(sum_k);
    capped = ikb_warp_sum(capped);
    n_err = ikb_warp_sum(n_err);
    err_sum = ikb_warp_sum(err_sum);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        first_limits = min(first_limits, __shfl_xor_sync(IKB_FULL_MASK, first_limits, o));
        first_range = min(first_range, __shfl_xor_sync(IKB_FULL_MASK, first_range, o));
    }
    if (lane == 0 && n_solved != 0) {
        atomicAdd(&a.stats->n_solved, n_solved);
        atomicAdd(&a.stats->sum_iterations, sum_k);
        if (capped)
            atomicAdd(&a.stats->n_iter_capped, capped);
        if (n_err) {
            atomicAdd(&a.stats->sum_fk_error, err_sum);
            atomicAdd(&a.stats->n_fk_error, n_err);
        }
        if (first_limits != IKB_I64_MAX)
            atomicMin(&a.stats->first_out_of_limits, first_limits);
        if (first_range != IKB_I64_MAX)
            atomicMin(&a.stats->first_fk_angle_range, first_range);
    }
}

// ---- damped-least-squares refinement of joint angles onto full effector poses --------------------------------------
// The sibling of dls_refine_kernel for a 6-D task: position and orientation of T_4, weighted per axis.  Same quad per
// row, chain, guards, refill loop, statistics and stores.  Lane r < 3 holds row r of the target ([R_d | p_d] row r),
// row r of T_4, element r of every z_j and row r of the position Jacobian, so it owns task rows r (linear) and 3 + r
// (angular).  Row r of R_e = R_d R^T needs the rows of R from the other lanes (quad shuffles); the quaternion error is
// then formed redundantly in every lane.  A = J^T W J + lambda^2 I and b = J^T W e are summed over the task rows as
// per-lane partials reduced across the quad (lane 3 contributes zero), and every lane solves the 4 x 4 system by
// LDL^T; lane k applies Delta theta_k.  Operation order: include/ikb200.h (ikb_dls_pose_refine_*).
struct DlsPoseArgs {
    const void *poses;   // n x 4 x 4 row-major, pose dtype; row 3 is not read
    int pose_f64;
    const void *seed;    // n_seed x 4 (n_seed 1 or n), angles dtype; may equal angles_out when n_seed == n
    long long n_seed;
    void *angles_out;    // n x 4, angles dtype
    int *iters;          // nullable, n
    void *err_out;       // nullable, n (angles dtype)
    long long n;
    long long index_base;  // global row of row 0 (host pipeline chunks): the row numbers in the statistics
    double w[6];         // task weights: x, y, z, then the three orientation axes
    double lam2;         // damping^2, rounded once
    double tol;
    int max_iter;
    IkbDeviceStats *stats;
    unsigned long long *work_counter;  // zero at launch
    IkbRobot rc;
};

__device__ __forceinline__ double ikb_load_elem(const void *p, int f64, long long i)
{
    return f64 ? __ldg(reinterpret_cast<const double *>(p) + i) : (double)__ldg(reinterpret_cast<const float *>(p) + i);
}

// a + b over the four lanes of a quad, as (lane 0 + lane 1) + (lane 2 + lane 3) in every lane (addition commutes)
__device__ __forceinline__ double ikb_quad_sum(double v)
{
    v = __dadd_rn(v, __shfl_xor_sync(IKB_FULL_MASK, v, 1, 4));
    return __dadd_rn(v, __shfl_xor_sync(IKB_FULL_MASK, v, 2, 4));
}

template <typename Real>
__global__ void __launch_bounds__(DLS_THREADS) dls_pose_refine_kernel(const DlsPoseArgs a)
{
    const double TWO_PI = 6.283185307179586, PI = 3.141592653589793;
    const int lane = threadIdx.x & 31, r = lane & 3;
    const unsigned quads_below = (1u << (lane & ~3)) - 1u;
    const bool alpha_bad = a.rc.alpha[r] < -TWO_PI || a.rc.alpha[r] > TWO_PI;
    const bool task = r < 3;  // lane r owns task rows r and 3 + r
    const double w_lin = r == 0 ? a.w[0] : r == 1 ? a.w[1] : a.w[2];
    const double w_ang = r == 0 ? a.w[3] : r == 1 ? a.w[4] : a.w[5];
    double th = 0.0, rd0 = 0.0, rd1 = 0.0, rd2 = 0.0, pd = 0.0;  // row r of the target: R_d row r and p_d[r]
    long long row = 0;
    int k = 0;
    bool live = false, exhausted = false;
    unsigned long long n_solved = 0, sum_k = 0, capped = 0, n_err = 0;
    double err_sum = 0.0;
    long long first_limits = IKB_I64_MAX, first_range = IKB_I64_MAX;
    for (;;) {
        if (!exhausted) {  // refill: every quad without a row takes the next one
            const unsigned want = __ballot_sync(IKB_FULL_MASK, !live) & 0x11111111u;
            if (want) {
                unsigned long long base = 0;
                if (lane == 0)
                    base = atomicAdd(a.work_counter, (unsigned long long)__popc(want));
                base = __shfl_sync(IKB_FULL_MASK, base, 0);
                if (!live) {
                    const long long rw = (long long)base + __popc(want & quads_below);
                    if (rw < a.n) {
                        row = rw;
                        k = 0;
                        live = true;
                        th = (double)reinterpret_cast<const Real *>(a.seed)[4 * (a.n_seed == 1 ? 0 : rw) + r];
                        if (task) {
                            const long long o = 16 * rw + 4 * r;
                            rd0 = ikb_load_elem(a.poses, a.pose_f64, o);
                            rd1 = ikb_load_elem(a.poses, a.pose_f64, o + 1);
                            rd2 = ikb_load_elem(a.poses, a.pose_f64, o + 2);
                            pd = ikb_load_elem(a.poses, a.pose_f64, o + 3);
                        }
                        if (th < -TWO_PI || th > TWO_PI || alpha_bad)
                            first_range = min(first_range, a.index_base + rw);
                        if (r == 0 && ikb_out_of_limits(a.rc, pd, ikb_load_elem(a.poses, a.pose_f64, 16 * rw + 7),
                                                        ikb_load_elem(a.poses, a.pose_f64, 16 * rw + 11)))
                            first_limits = min(first_limits, a.index_base + rw);
                    }
                }
                exhausted = (long long)(base + __popc(want)) >= a.n;
            }
        }
        if (__ballot_sync(IKB_FULL_MASK, live) == 0)
            break;
        // the chain, at full warp width (quads without a row compute on stale registers and write nothing)
        double s, c;
        sincos(th, &s, &c);
        double t[4] = {r == 0 ? 1.0 : 0.0, r == 1 ? 1.0 : 0.0, r == 2 ? 1.0 : 0.0, r == 3 ? 1.0 : 0.0};
        double zs[4], ps[5];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const double sj = __shfl_sync(IKB_FULL_MASK, s, j, 4), cj = __shfl_sync(IKB_FULL_MASK, c, j, 4);
            double nr[4];
            zs[j] = t[2];
            ps[j] = t[3];
            fk_dh_step_row(t, sj, cj, a.rc.cos_alpha[j], a.rc.sin_alpha[j], a.rc.a[j], a.rc.eps[j], nr);
#pragma unroll
            for (int q = 0; q < 4; ++q)
                t[q] = nr[q];
        }
        ps[4] = t[3];
        double lin[4];
        fk_quad_position_jacobian_row(r, zs, ps, lin);
        // row r of R_e = R_d R^T: (R_e)_rj = (Rd_r0 R_j0 + Rd_r1 R_j1) + Rd_r2 R_j2, row j of R from lane j
        double me[3];
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            const double r0 = __shfl_sync(IKB_FULL_MASK, t[0], j, 4), r1 = __shfl_sync(IKB_FULL_MASK, t[1], j, 4);
            const double r2 = __shfl_sync(IKB_FULL_MASK, t[2], j, 4);
            me[j] = __dadd_rn(__dadd_rn(__dmul_rn(rd0, r0), __dmul_rn(rd1, r1)), __dmul_rn(rd2, r2));
        }
        double M[3][3];
#pragma unroll
        for (int i = 0; i < 3; ++i)
#pragma unroll
            for (int j = 0; j < 3; ++j)
                M[i][j] = __shfl_sync(IKB_FULL_MASK, me[j], i, 4);
        // e_o = 2 x the vector part of R_e's unit quaternion, scalar part >= 0 (Shepperd: branch on the largest of
        // the trace and the diagonal, first on ties; h = 2 |q_w| or 2 |q_x|, 2 |q_y|, 2 |q_z|)
        const double tr = __dadd_rn(__dadd_rn(M[0][0], M[1][1]), M[2][2]);
        const double dx = __dsub_rn(M[2][1], M[1][2]), dy = __dsub_rn(M[0][2], M[2][0]), dz = __dsub_rn(M[1][0], M[0][1]);
        double eo0, eo1, eo2;
        if (tr >= M[0][0] && tr >= M[1][1] && tr >= M[2][2]) {  // a NaN diagonal falls through to the last case
            const double h = __dsqrt_rn(__dadd_rn(1.0, tr));
            eo0 = __ddiv_rn(dx, h); eo1 = __ddiv_rn(dy, h); eo2 = __ddiv_rn(dz, h);
        } else if (M[0][0] >= M[1][1] && M[0][0] >= M[2][2]) {
            const double h = __dsqrt_rn(__dsub_rn(__dsub_rn(__dadd_rn(1.0, M[0][0]), M[1][1]), M[2][2]));
            eo0 = h; eo1 = __ddiv_rn(__dadd_rn(M[0][1], M[1][0]), h); eo2 = __ddiv_rn(__dadd_rn(M[0][2], M[2][0]), h);
            if (dx < 0.0) { eo0 = -eo0; eo1 = -eo1; eo2 = -eo2; }
        } else if (M[1][1] >= M[2][2]) {
            const double h = __dsqrt_rn(__dsub_rn(__dsub_rn(__dadd_rn(1.0, M[1][1]), M[0][0]), M[2][2]));
            eo0 = __ddiv_rn(__dadd_rn(M[0][1], M[1][0]), h); eo1 = h; eo2 = __ddiv_rn(__dadd_rn(M[1][2], M[2][1]), h);
            if (dy < 0.0) { eo0 = -eo0; eo1 = -eo1; eo2 = -eo2; }
        } else {
            const double h = __dsqrt_rn(__dsub_rn(__dsub_rn(__dadd_rn(1.0, M[2][2]), M[0][0]), M[1][1]));
            eo0 = __ddiv_rn(__dadd_rn(M[0][2], M[2][0]), h); eo1 = __ddiv_rn(__dadd_rn(M[1][2], M[2][1]), h); eo2 = h;
            if (dz < 0.0) { eo0 = -eo0; eo1 = -eo1; eo2 = -eo2; }
        }
        const double ep = __dsub_rn(pd, t[3]);  // e_p[r]
        const double ex = __shfl_sync(IKB_FULL_MASK, ep, 0, 4), ey = __shfl_sync(IKB_FULL_MASK, ep, 1, 4);
        const double ez = __shfl_sync(IKB_FULL_MASK, ep, 2, 4);
        const double sp = __dadd_rn(__dadd_rn(__dmul_rn(a.w[0], __dmul_rn(ex, ex)), __dmul_rn(a.w[1], __dmul_rn(ey, ey))),
                                    __dmul_rn(a.w[2], __dmul_rn(ez, ez)));
        const double so = __dadd_rn(__dadd_rn(__dmul_rn(a.w[3], __dmul_rn(eo0, eo0)), __dmul_rn(a.w[4], __dmul_rn(eo1, eo1))),
                                    __dmul_rn(a.w[5], __dmul_rn(eo2, eo2)));
        const double err = __dsqrt_rn(__dadd_rn(sp, so));
        // A = J^T W J (upper triangle) and b = J^T W e at full warp width, since the quad sums shuffle (a row that
        // stops below does not use them).  g = w_r J_r, ga = w_{3+r} J_{3+r}: this lane's weighted task rows
        const double eor = r == 0 ? eo0 : r == 1 ? eo1 : eo2;
        double g[4], ga[4];
#pragma unroll
        for (int m = 0; m < 4; ++m) {
            g[m] = __dmul_rn(w_lin, lin[m]);
            ga[m] = __dmul_rn(w_ang, zs[m]);
        }
        double A[4][4], b[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
#pragma unroll
            for (int j = i; j < 4; ++j)
                A[i][j] = ikb_quad_sum(task ? __dadd_rn(__dmul_rn(g[i], lin[j]), __dmul_rn(ga[i], zs[j])) : 0.0);
            b[i] = ikb_quad_sum(task ? __dadd_rn(__dmul_rn(g[i], ep), __dmul_rn(ga[i], eor)) : 0.0);
        }
        if (live && (err <= a.tol || k >= a.max_iter)) {  // quad-uniform: every lane holds the same err and k
            reinterpret_cast<Real *>(a.angles_out)[4 * row + r] = (Real)th;
            if (r == 0) {
                if (a.iters)
                    a.iters[row] = k;
                if (a.err_out)
                    reinterpret_cast<Real *>(a.err_out)[row] = (Real)err;
                ++n_solved;
                sum_k += (unsigned)k;
                capped += err <= a.tol ? 0u : 1u;  // NaN rows included
                if (isfinite(err)) {
                    err_sum += err;
                    ++n_err;
                }
            }
            live = false;
        }
        if (live) {
#pragma unroll
            for (int i = 0; i < 4; ++i)
                A[i][i] = __dadd_rn(A[i][i], a.lam2);
            // A y = b by LDL^T (no square root)
            const double l10 = __ddiv_rn(A[0][1], A[0][0]), l20 = __ddiv_rn(A[0][2], A[0][0]);
            const double l30 = __ddiv_rn(A[0][3], A[0][0]);
            const double d1 = __dsub_rn(A[1][1], __dmul_rn(l10, A[0][1]));
            const double t21 = __dsub_rn(A[1][2], __dmul_rn(l20, A[0][1]));
            const double t31 = __dsub_rn(A[1][3], __dmul_rn(l30, A[0][1]));
            const double l21 = __ddiv_rn(t21, d1), l31 = __ddiv_rn(t31, d1);
            const double d2 = __dsub_rn(__dsub_rn(A[2][2], __dmul_rn(l20, A[0][2])), __dmul_rn(l21, t21));
            const double t32 = __dsub_rn(__dsub_rn(A[2][3], __dmul_rn(l30, A[0][2])), __dmul_rn(l31, t21));
            const double l32 = __ddiv_rn(t32, d2);
            const double d3 = __dsub_rn(__dsub_rn(__dsub_rn(A[3][3], __dmul_rn(l30, A[0][3])), __dmul_rn(l31, t31)),
                                        __dmul_rn(l32, t32));
            const double z1 = __dsub_rn(b[1], __dmul_rn(l10, b[0]));
            const double z2 = __dsub_rn(__dsub_rn(b[2], __dmul_rn(l20, b[0])), __dmul_rn(l21, z1));
            const double z3 = __dsub_rn(__dsub_rn(__dsub_rn(b[3], __dmul_rn(l30, b[0])), __dmul_rn(l31, z1)),
                                        __dmul_rn(l32, z2));
            const double y3 = __ddiv_rn(z3, d3);
            const double y2 = __dsub_rn(__ddiv_rn(z2, d2), __dmul_rn(l32, y3));
            const double y1 = __dsub_rn(__dsub_rn(__ddiv_rn(z1, d1), __dmul_rn(l21, y2)), __dmul_rn(l31, y3));
            const double y0 = __dsub_rn(__dsub_rn(__dsub_rn(__ddiv_rn(b[0], A[0][0]), __dmul_rn(l10, y1)),
                                                  __dmul_rn(l20, y2)),
                                        __dmul_rn(l30, y3));
            th = __dadd_rn(th, r == 0 ? y0 : r == 1 ? y1 : r == 2 ? y2 : y3);
            if (fabs(th) > PI)
                th = remainder(th, TWO_PI);  // exact: the angle stays inside the FK guard
            ++k;
        }
    }
    n_solved = ikb_warp_sum(n_solved);
    sum_k = ikb_warp_sum(sum_k);
    capped = ikb_warp_sum(capped);
    n_err = ikb_warp_sum(n_err);
    err_sum = ikb_warp_sum(err_sum);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        first_limits = min(first_limits, __shfl_xor_sync(IKB_FULL_MASK, first_limits, o));
        first_range = min(first_range, __shfl_xor_sync(IKB_FULL_MASK, first_range, o));
    }
    if (lane == 0 && n_solved != 0) {
        atomicAdd(&a.stats->n_solved, n_solved);
        atomicAdd(&a.stats->sum_iterations, sum_k);
        if (capped)
            atomicAdd(&a.stats->n_iter_capped, capped);
        if (n_err) {
            atomicAdd(&a.stats->sum_fk_error, err_sum);
            atomicAdd(&a.stats->n_fk_error, n_err);
        }
        if (first_limits != IKB_I64_MAX)
            atomicMin(&a.stats->first_out_of_limits, first_limits);
        if (first_range != IKB_I64_MAX)
            atomicMin(&a.stats->first_fk_angle_range, first_range);
    }
}

struct LimitsArgs {
    const void *xyz;
    int xyz_f64;
    long long n;
    long long index_base;
    IkbDeviceStats *stats;
    IkbRobot rc;
};

// K0: reference InverseKinematics.check_limits (inverse.py:26-35) as a min-index reduction.
__global__ void __launch_bounds__(256) check_limits_kernel(const LimitsArgs a)
{
    const long long stride = (long long)gridDim.x * blockDim.x;
    long long first = IKB_I64_MAX;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < a.n; i += stride) {
        double x, y, z;
        ikb_load_xyz(a.xyz, a.xyz_f64, i, x, y, z);
        if (ikb_out_of_limits(a.rc, x, y, z) && i < first)
            first = i;  // grid-stride order is increasing per thread
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const long long other = __shfl_xor_sync(IKB_FULL_MASK, first, o);
        first = other < first ? other : first;
    }
    if ((threadIdx.x & 31) == 0 && first != IKB_I64_MAX)
        atomicMin(&a.stats->first_out_of_limits, a.index_base + first);
}

// Dependent-FMA-chain microbenchmark: 8 independent chains per thread keep the pipe full.
template <typename Real>
__global__ void __launch_bounds__(256) fma_peak_kernel(Real *sink, int iters, Real seed)
{
    Real v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j)
        v[j] = seed + (Real)(threadIdx.x + j);
    const Real m = (Real)0.999, c = (Real)0.001;
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int u = 0; u < 4; ++u)
#pragma unroll
            for (int j = 0; j < 8; ++j)
                v[j] = fma(v[j], m, c);
    }
    Real s = 0;
#pragma unroll
    for (int j = 0; j < 8; ++j)
        s += v[j];
    if (s == (Real)-1)
        sink[0] = s;
}

}  // namespace

static unsigned ikb_stream_grid(long long n, int num_sms, int threads, int ctas_per_sm)
{
    long long want = (n + threads - 1) / threads;
    long long cap = (long long)num_sms * ctas_per_sm;
    return (unsigned)(want < cap ? (want > 0 ? want : 1) : cap);
}

cudaError_t ikb_launch_fk(const void *angles, int angles_f64, long long n, long long index_base,
                          void *pos_out, const void *targets, int xyz_f64, void *err_out,
                          IkbDeviceStats *stats, const IkbRobot &rc, int num_sms, cudaStream_t stream)
{
    if (n <= 0)
        return cudaSuccess;
    FkArgs a;
    a.angles = angles; a.angles_f64 = angles_f64; a.n = n; a.index_base = index_base;
    a.pos_out = pos_out; a.targets = targets; a.xyz_f64 = xyz_f64; a.err_out = err_out;
    a.stats = stats; a.rc = rc;
    // fp32 buffers, closed-form arm with alpha inside the guard, error only, 8-byte aligned rows: the pair kernel
    bool alpha_ok = rc.fk_planar_tail != 0;
    for (int j = 0; j < 4; ++j)
        alpha_ok = alpha_ok && !(rc.alpha[j] < -6.283185307179586) && !(rc.alpha[j] > 6.283185307179586);
    if (!angles_f64 && !xyz_f64 && targets && !pos_out && alpha_ok && ((uintptr_t)targets & 7) == 0 &&
        ((uintptr_t)err_out & 7) == 0 && n >= 2) {
        static const bool use_stream = [] { const char *v = std::getenv("IKB_FK_STREAM"); return !v || v[0] != '0'; }();
        const long long n_trips = n / 64;  // full trips of 32 pairs for the asynchronous-copy kernel
        if (use_stream && n_trips >= 4LL * num_sms * FK_STREAM_WARPS && ((uintptr_t)targets & 15) == 0 &&
            ((uintptr_t)angles & 15) == 0) {
            const long long want = (n_trips + FK_STREAM_WARPS - 1) / FK_STREAM_WARPS, cap = (long long)num_sms * 4;
            static const cudaError_t carve = cudaFuncSetAttribute(fk_error_stream_kernel, cudaFuncAttributePreferredSharedMemoryCarveout,
                                                                  (int)cudaSharedmemCarveoutMaxShared);
            if (carve != cudaSuccess)
                return carve;
            fk_error_stream_kernel<<<(unsigned)(want < cap ? want : cap), FK_STREAM_WARPS * 32, 0, stream>>>(a, n_trips);
            cudaError_t err = cudaGetLastError();
            const long long done = n_trips * 64;
            if (err != cudaSuccess || done == n)
                return err;
            // the last partial trip (< 64 rows): the pair kernel on the tail, same arithmetic
            FkArgs t = a;
            t.n = n - done;
            t.index_base = index_base + done;
            t.angles = reinterpret_cast<const float *>(angles) + 4 * done;
            t.targets = reinterpret_cast<const float *>(targets) + 3 * done;
            t.err_out = err_out ? reinterpret_cast<float *>(err_out) + done : nullptr;
            if (t.n >= 2) {
                fk_error_pairs_kernel<<<1, 256, 0, stream>>>(t);
                return cudaGetLastError();
            }
            a = t;  // a single odd row: the generic kernel below
            fk_kernel<float, false><<<1, 256, 0, stream>>>(a);
            return cudaGetLastError();
        }
        const unsigned pgrid = ikb_stream_grid(n / 2, num_sms, 256, FK_PAIR_MINB);
        fk_error_pairs_kernel<<<pgrid, 256, 0, stream>>>(a);
        return cudaGetLastError();
    }
    const unsigned grid = ikb_stream_grid(n, num_sms, 256, 8);
    if (angles_f64) {
        if (xyz_f64)
            fk_kernel<double, true><<<grid, 256, 0, stream>>>(a);
        else
            fk_kernel<double, false><<<grid, 256, 0, stream>>>(a);
    } else {
        if (xyz_f64)
            fk_kernel<float, true><<<grid, 256, 0, stream>>>(a);
        else
            fk_kernel<float, false><<<grid, 256, 0, stream>>>(a);
    }
    return cudaGetLastError();
}

// Persistent grid: as many CTAs as fit the SMs at once (shared memory bounds it for fp64 matrices: 64 KB per CTA).
template <typename Real, int KIND, bool MANIP = false>
static cudaError_t launch_fk_transforms(const void *angles, long long n, long long index_base, void *out,
                                        IkbDeviceStats *stats, const IkbRobot &rc, int num_sms, cudaStream_t stream,
                                        void *manip = nullptr)
{
    constexpr int smem = 2 * FKT_ROWS * fkt_row_elems(KIND) * (int)sizeof(Real);
    constexpr int kMaxDevices = 64;
    static int ctas_per_sm[kMaxDevices] = {};  // 0: the attribute is not set on that device yet (it is per device)
    int dev = 0;
    cudaError_t err = cudaGetDevice(&dev);
    if (err != cudaSuccess)
        return err;
    int ctas = dev < kMaxDevices ? ctas_per_sm[dev] : 0;
    if (ctas == 0) {
        err = cudaFuncSetAttribute(fk_transforms_kernel<Real, KIND, MANIP>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   smem);
        if (err == cudaSuccess)
            err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctas, fk_transforms_kernel<Real, KIND, MANIP>,
                                                                FKT_THREADS, smem);
        if (err != cudaSuccess)
            return err;
        ctas = ctas > 0 ? ctas : 1;
        if (dev < kMaxDevices)
            ctas_per_sm[dev] = ctas;
    }
    const long long tiles = (n + FKT_ROWS - 1) / FKT_ROWS, cap = (long long)num_sms * ctas;
    fk_transforms_kernel<Real, KIND, MANIP><<<(unsigned)(tiles < cap ? tiles : cap), FKT_THREADS, smem, stream>>>(
        reinterpret_cast<const Real *>(angles), n, index_base, reinterpret_cast<Real *>(out), stats, rc,
        reinterpret_cast<Real *>(manip));
    return cudaGetLastError();
}

cudaError_t ikb_launch_fk_transforms(const void *angles, int angles_f64, long long n, long long index_base, int what,
                                     void *out, IkbDeviceStats *stats, const IkbRobot &rc, int num_sms,
                                     cudaStream_t stream)
{
    if (n <= 0)
        return cudaSuccess;
    const bool joints = what == IKB_FK_JOINTS;
    if (angles_f64)
        return joints ? launch_fk_transforms<double, FKT_JOINTS>(angles, n, index_base, out, stats, rc, num_sms, stream)
                      : launch_fk_transforms<double, FKT_MATRICES>(angles, n, index_base, out, stats, rc, num_sms, stream);
    return joints ? launch_fk_transforms<float, FKT_JOINTS>(angles, n, index_base, out, stats, rc, num_sms, stream)
                  : launch_fk_transforms<float, FKT_MATRICES>(angles, n, index_base, out, stats, rc, num_sms, stream);
}

template <typename Real>
static cudaError_t launch_jacobian(const void *angles, long long n, long long index_base, bool geometric, void *jac,
                                   void *manip, IkbDeviceStats *stats, const IkbRobot &rc, int num_sms,
                                   cudaStream_t stream)
{
    if (!jac)
        return launch_fk_transforms<Real, FKT_MANIP_ONLY, true>(angles, n, index_base, nullptr, stats, rc, num_sms,
                                                                stream, manip);
    if (geometric)
        return manip ? launch_fk_transforms<Real, FKT_JAC_GEOMETRIC, true>(angles, n, index_base, jac, stats, rc, num_sms,
                                                                           stream, manip)
                     : launch_fk_transforms<Real, FKT_JAC_GEOMETRIC, false>(angles, n, index_base, jac, stats, rc,
                                                                            num_sms, stream);
    return manip ? launch_fk_transforms<Real, FKT_JAC_POSITION, true>(angles, n, index_base, jac, stats, rc, num_sms,
                                                                      stream, manip)
                 : launch_fk_transforms<Real, FKT_JAC_POSITION, false>(angles, n, index_base, jac, stats, rc, num_sms,
                                                                       stream);
}

// the arm Jacobian (what: IKB_JAC_GEOMETRIC / IKB_JAC_POSITION) into jac and/or the manipulability into manip
cudaError_t ikb_launch_jacobian(const void *angles, int angles_f64, long long n, long long index_base, int what,
                                void *jac, void *manip, IkbDeviceStats *stats, const IkbRobot &rc, int num_sms,
                                cudaStream_t stream)
{
    if (n <= 0)
        return cudaSuccess;
    const bool geometric = what == IKB_JAC_GEOMETRIC;
    return angles_f64 ? launch_jacobian<double>(angles, n, index_base, geometric, jac, manip, stats, rc, num_sms, stream)
                      : launch_jacobian<float>(angles, n, index_base, geometric, jac, manip, stats, rc, num_sms, stream);
}

// damped-least-squares refinement (ikb_dls_refine_*); work_counter: a counter of the engine's ring (reset here)
cudaError_t ikb_launch_dls_refine(const void *xyz, int xyz_f64, const void *seed, long long n_seed, void *angles_out,
                                  int angles_f64, int *iters, void *err_out, long long n, long long index_base,
                                  double damping, double tol, int max_iter, IkbDeviceStats *stats,
                                  unsigned long long *work_counter, const IkbRobot &rc, int num_sms,
                                  cudaStream_t stream)
{
    if (n <= 0)
        return cudaSuccess;
    DlsArgs a;
    a.xyz = xyz; a.xyz_f64 = xyz_f64; a.seed = seed; a.n_seed = n_seed; a.angles_out = angles_out;
    a.iters = iters; a.err_out = err_out; a.n = n; a.index_base = index_base;
    a.lam2 = damping * damping; a.tol = tol; a.max_iter = max_iter;
    a.stats = stats; a.work_counter = work_counter; a.rc = rc;
    void (*kern)(DlsArgs) = angles_f64 ? dls_refine_kernel<double> : dls_refine_kernel<float>;
    static int blocks_per_sm[2] = {};
    int &bps = blocks_per_sm[angles_f64 ? 1 : 0];
    if (bps == 0) {
        cudaError_t err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, kern, DLS_THREADS, 0);
        if (err != cudaSuccess)
            return err;
        bps = bps > 0 ? bps : 1;
    }
    cudaError_t err = cudaMemsetAsync(work_counter, 0, sizeof(unsigned long long), stream);
    if (err != cudaSuccess)
        return err;
    // persistent grid: resident CTAs per SM x SM count, trimmed for small batches (one quad per row)
    const long long want = (n + DLS_THREADS / 4 - 1) / (DLS_THREADS / 4), cap = (long long)num_sms * bps;
    kern<<<(unsigned)(want < cap ? want : cap), DLS_THREADS, 0, stream>>>(a);
    return cudaGetLastError();
}

// damped-least-squares refinement onto poses (ikb_dls_pose_refine_*); work_counter as for ikb_launch_dls_refine
cudaError_t ikb_launch_dls_pose_refine(const void *poses, int pose_f64, const void *seed, long long n_seed,
                                       void *angles_out, int angles_f64, int *iters, void *err_out, long long n,
                                       long long index_base, const double weights[6], double damping, double tol,
                                       int max_iter, IkbDeviceStats *stats, unsigned long long *work_counter,
                                       const IkbRobot &rc, int num_sms, cudaStream_t stream)
{
    if (n <= 0)
        return cudaSuccess;
    DlsPoseArgs a;
    a.poses = poses; a.pose_f64 = pose_f64; a.seed = seed; a.n_seed = n_seed; a.angles_out = angles_out;
    a.iters = iters; a.err_out = err_out; a.n = n; a.index_base = index_base;
    for (int i = 0; i < 6; ++i)
        a.w[i] = weights[i];
    a.lam2 = damping * damping; a.tol = tol; a.max_iter = max_iter;
    a.stats = stats; a.work_counter = work_counter; a.rc = rc;
    void (*kern)(DlsPoseArgs) = angles_f64 ? dls_pose_refine_kernel<double> : dls_pose_refine_kernel<float>;
    static int blocks_per_sm[2] = {};
    int &bps = blocks_per_sm[angles_f64 ? 1 : 0];
    if (bps == 0) {
        cudaError_t err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, kern, DLS_THREADS, 0);
        if (err != cudaSuccess)
            return err;
        bps = bps > 0 ? bps : 1;
    }
    cudaError_t err = cudaMemsetAsync(work_counter, 0, sizeof(unsigned long long), stream);
    if (err != cudaSuccess)
        return err;
    const long long want = (n + DLS_THREADS / 4 - 1) / (DLS_THREADS / 4), cap = (long long)num_sms * bps;
    kern<<<(unsigned)(want < cap ? want : cap), DLS_THREADS, 0, stream>>>(a);
    return cudaGetLastError();
}

cudaError_t ikb_launch_check_limits(const void *xyz, int xyz_f64, long long n, long long index_base,
                                    IkbDeviceStats *stats, const IkbRobot &rc, int num_sms,
                                    cudaStream_t stream)
{
    if (n <= 0)
        return cudaSuccess;
    LimitsArgs a;
    a.xyz = xyz; a.xyz_f64 = xyz_f64; a.n = n; a.index_base = index_base; a.stats = stats; a.rc = rc;
    check_limits_kernel<<<ikb_stream_grid(n, num_sms, 256, 8), 256, 0, stream>>>(a);
    return cudaGetLastError();
}

cudaError_t ikb_launch_fma_peak(int f64, void *sink, int iters, int num_sms, cudaStream_t stream)
{
    if (f64)
        fma_peak_kernel<double><<<num_sms * 8, 256, 0, stream>>>((double *)sink, iters, 1.0);
    else
        fma_peak_kernel<float><<<num_sms * 8, 256, 0, stream>>>((float *)sink, iters, 1.0f);
    return cudaGetLastError();
}

// analytic.cu -- closed-form inverse kinematics (ikb_analytic_ik_*) for arms with a turning base and three parallel
// joints: alpha_2 = alpha_3 = alpha_4 = 0, |cos alpha_1| <= 1e-12, a_2, a_3 > 0.  include/ikb200.h states the
// arithmetic.  One thread per row computes every branch of that row.
#include "ikb_common.cuh"

namespace {

constexpr int AIK_THREADS = 256;

struct AnalyticArgs {
    const void *in;       // n x 4 x 4 poses or n x 3 positions
    int in_f64;
    const void *pitch;    // position kind: n_pitch values of the input's dtype
    int per_row_pitch;
    void *out;            // n x B x 4
    int vec_out;          // out is 16-byte aligned: vector stores
    int *status;          // nullable
    long long n, index_base;
    // the family's constants: s = sign(sin alpha_1), d = (eps_2 + eps_3) + eps_4, sd = -s d + 0 (never -0)
    double a1, a2, a3, a4, eps1, s, d, sd, a23p, a23m;
    IkbDeviceStats *stats;
    IkbRobot rc;
};

// element i of an fp32 / fp64 input, widened exactly; + 0 reads -0 as +0, so that signed zeros give the same bits
__device__ __forceinline__ double aik_load(const void *p, int f64, long long i)
{
    const double v = f64 ? __ldg(reinterpret_cast<const double *>(p) + i)
                         : (double)__ldg(reinterpret_cast<const float *>(p) + i);
    return v + 0.0;
}

__device__ __forceinline__ double aik_wrap(double th)
{
    const double TWO_PI = 6.283185307179586, PI = 3.141592653589793;
    return fabs(th) > PI ? remainder(th, TWO_PI) : th;  // exact: every answer stays inside the FK guard
}

// The two-link triangle to the wrist point: th[0..3] = (theta_2, theta_3, theta_4) of the theta_3 >= 0 branch into
// th[0], th[1]; of the theta_3 <= 0 branch into th[2], th[3] -- laid out as out[b][1..3].  Returns "does not reach".
__device__ __forceinline__ bool aik_triangle(const AnalyticArgs &a, double u, double v, double phi, double cphi,
                                             double sphi, double (&br)[2][3])
{
    const double uw = u - a.a4 * cphi, vw = v - a.a4 * sphi;
    const double r = sqrt(uw * uw + vw * vw);
    const double num = (a.a23p - r) * (a.a23p + r);  // < 0: stretched toward the wrist
    const double den = (r - a.a23m) * (r + a.a23m);  // < 0: folded toward the wrist
    const double t = 2.0 * atan2(sqrt(num > 0.0 ? num : 0.0), sqrt(den > 0.0 ? den : 0.0));
    double st, ct;
    sincos(t, &st, &ct);
    const double beta = atan2(vw, uw);
    const double g = atan2(a.a3 * st, a.a2 + a.a3 * ct);
    const double th2p = beta - g, th2m = beta - (0.0 - g), th3m = 0.0 - t;  // 0 - x: t = 0 gives +0 in both
    br[0][0] = aik_wrap(th2p);
    br[0][1] = t;
    br[0][2] = aik_wrap((phi - th2p) - t);
    br[1][0] = aik_wrap(th2m);
    br[1][1] = th3m;
    br[1][2] = aik_wrap((phi - th2m) - th3m);
    return num < 0.0 || den < 0.0;
}

// branch b of row i: (theta_1, br) or, for a row with a non-finite input, NaN
template <typename Out, int B>
__device__ __forceinline__ void aik_store(const AnalyticArgs &a, long long i, int b, bool finite, double th1,
                                          const double (&br)[3])
{
    const double nan = __longlong_as_double(0x7ff8000000000000LL);
    const double t0 = finite ? th1 : nan, t1 = finite ? br[0] : nan, t2 = finite ? br[1] : nan;
    const double t3 = finite ? br[2] : nan;
    Out *o = reinterpret_cast<Out *>(a.out) + ((long long)B * i + b) * 4;
    if (a.vec_out) {
        if constexpr (sizeof(Out) == 8) {
            reinterpret_cast<double2 *>(o)[0] = make_double2(t0, t1);
            reinterpret_cast<double2 *>(o)[1] = make_double2(t2, t3);
        } else {
            *reinterpret_cast<float4 *>(o) = make_float4((float)t0, (float)t1, (float)t2, (float)t3);
        }
    } else {
        o[0] = (Out)t0; o[1] = (Out)t1; o[2] = (Out)t2; o[3] = (Out)t3;
    }
}

// KIND: IKB_AIK_POSE (B = 2) or IKB_AIK_POSITION_PITCH (B = 4)
template <int KIND, typename Out>
__global__ void __launch_bounds__(AIK_THREADS) analytic_ik_kernel(const AnalyticArgs a)
{
    constexpr int B = KIND == IKB_AIK_POSE ? 2 : 4;
    const double PI = 3.141592653589793;
    const long long stride = (long long)gridDim.x * blockDim.x;
    unsigned long long n_rows = 0;
    long long first_limits = IKB_I64_MAX;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < a.n; i += stride) {
        int bad = 0;
        bool finite;
        double px, py, pz;
        if constexpr (KIND == IKB_AIK_POSE) {
            double m[3][4];
#pragma unroll
            for (int r = 0; r < 3; ++r)
#pragma unroll
                for (int c = 0; c < 4; ++c)
                    m[r][c] = aik_load(a.in, a.in_f64, 16 * i + 4 * r + c);
            finite = true;
#pragma unroll
            for (int r = 0; r < 3; ++r)
#pragma unroll
                for (int c = 0; c < 4; ++c)
                    finite = finite && isfinite(m[r][c]);
            px = m[0][3]; py = m[1][3]; pz = m[2][3];
            // theta_1 from the joint axis z (column 2), phi = theta_2 + theta_3 + theta_4 from the tool axis x (column 0)
            const double th1 = atan2(a.s * m[0][2], -a.s * m[1][2]);
            double s1, c1;
            sincos(th1, &s1, &c1);
            const double phi = atan2(a.s * m[2][0], c1 * m[0][0] + s1 * m[1][0]);
            double sphi, cphi;
            sincos(phi, &sphi, &cphi);
            const double u = (c1 * px + s1 * py) - a.a1, v = a.s * (pz - a.eps1);
            double br[2][3];
            bad = aik_triangle(a, u, v, phi, cphi, sphi, br) ? 3 : 0;
            aik_store<Out, B>(a, i, 0, finite, th1, br[0]);
            aik_store<Out, B>(a, i, 1, finite, th1, br[1]);
        } else {
            px = aik_load(a.in, a.in_f64, 3 * i);
            py = aik_load(a.in, a.in_f64, 3 * i + 1);
            pz = aik_load(a.in, a.in_f64, 3 * i + 2);
            const double pitch = aik_load(a.pitch, a.in_f64, a.per_row_pitch ? i : 0);
            finite = isfinite(px) && isfinite(py) && isfinite(pz) && isfinite(pitch);
            const double rho2 = px * px + py * py, d2 = a.d * a.d;
            const bool inside = rho2 < d2;  // closer to the base axis than the lateral offset: q = 0
            const double q = sqrt(inside ? 0.0 : rho2 - d2);
            const double azim = atan2(py, px), v = a.s * (pz - a.eps1);
#pragma unroll
            for (int side = 0; side < 2; ++side) {  // front (q >= 0, phi = pitch), back (-q, phi = pi - pitch)
                const double qq = side ? -q : q, phi = side ? PI - pitch : pitch;
                const double th1 = aik_wrap(azim - atan2(a.sd, qq));
                double sphi, cphi;
                sincos(phi, &sphi, &cphi);
                double br[2][3];
                if (aik_triangle(a, qq - a.a1, v, phi, cphi, sphi, br) || inside)
                    bad |= 3 << (2 * side);
                aik_store<Out, B>(a, i, 2 * side, finite, th1, br[0]);
                aik_store<Out, B>(a, i, 2 * side + 1, finite, th1, br[1]);
            }
        }
        if (a.status)
            a.status[i] = finite ? bad : (1 << B) - 1;
        if (ikb_out_of_limits(a.rc, px, py, pz))
            first_limits = min(first_limits, a.index_base + i);
        ++n_rows;
    }
    n_rows = ikb_warp_sum(n_rows);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
        first_limits = min(first_limits, __shfl_xor_sync(IKB_FULL_MASK, first_limits, o));
    if ((threadIdx.x & 31) == 0 && n_rows != 0) {
        atomicAdd(&a.stats->n_solved, n_rows);
        if (first_limits != IKB_I64_MAX)
            atomicMin(&a.stats->first_out_of_limits, first_limits);
    }
}

template <int KIND>
cudaError_t launch_kind(const AnalyticArgs &a, int out_f64, int num_sms, cudaStream_t stream)
{
    void (*kern)(AnalyticArgs) = out_f64 ? analytic_ik_kernel<KIND, double> : analytic_ik_kernel<KIND, float>;
    static int blocks_per_sm[2] = {};
    int &bps = blocks_per_sm[out_f64 ? 1 : 0];
    if (bps == 0) {
        cudaError_t err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, kern, AIK_THREADS, 0);
        if (err != cudaSuccess)
            return err;
        bps = bps > 0 ? bps : 1;
    }
    // one resident wave of CTAs striding over the rows: the statistics go out once per warp
    const long long want = (a.n + AIK_THREADS - 1) / AIK_THREADS, cap = (long long)num_sms * bps;
    kern<<<(unsigned)(want < cap ? want : cap), AIK_THREADS, 0, stream>>>(a);
    return cudaGetLastError();
}

}  // namespace

// closed-form inverse kinematics (ikb_analytic_ik_*); the caller has checked the arguments and the DH family
cudaError_t ikb_launch_analytic_ik(int kind, const void *in, int in_f64, long long n, long long index_base,
                                   const void *pitch, int per_row_pitch, void *angles_out, int angles_f64,
                                   int *status, IkbDeviceStats *stats, const IkbRobot &rc, int num_sms,
                                   cudaStream_t stream)
{
    if (n <= 0)
        return cudaSuccess;
    AnalyticArgs a;
    a.in = in; a.in_f64 = in_f64; a.pitch = pitch; a.per_row_pitch = per_row_pitch;
    a.out = angles_out; a.vec_out = ((uintptr_t)angles_out & 15) == 0; a.status = status;
    a.n = n; a.index_base = index_base;
    a.a1 = rc.a[0]; a.a2 = rc.a[1]; a.a3 = rc.a[2]; a.a4 = rc.a[3]; a.eps1 = rc.eps[0];
    a.s = rc.sin_alpha[0] > 0.0 ? 1.0 : -1.0;
    a.d = (rc.eps[1] + rc.eps[2]) + rc.eps[3];
    a.sd = -a.s * a.d + 0.0;
    a.a23p = rc.a[1] + rc.a[2]; a.a23m = rc.a[1] - rc.a[2];
    a.stats = stats; a.rc = rc;
    return kind == IKB_AIK_POSE ? launch_kind<IKB_AIK_POSE>(a, angles_f64, num_sms, stream)
                                : launch_kind<IKB_AIK_POSITION_PITCH>(a, angles_f64, num_sms, stream);
}

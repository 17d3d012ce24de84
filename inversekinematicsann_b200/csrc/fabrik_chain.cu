// fabrik_chain.cu -- batched Fabrik.calculate (reference fabrik.py:19-67) for chains of J = 1..256 points (sm_100a).
//
// Per row: chain P[0..J-1], links d[0..J-1], goal T, S = P[0];
//   while (se > tol or ge > tol) and max_iter > k:
//     b = T; for j = J-2 .. 0: b = PB(b, P[j], d[j]); P[j] = b        backward, fabrik.py:19-29
//     se = |P[0] - S|; P[0] = S                                          fabrik.py:61
//     for j = 1 .. J-1: P[j] = PB(P[j-1], j == J-1 ? T : P[j], d[j])    forward, fabrik.py:32-42
//     ge = |P[J-1] - T|; k += 1                                          fabrik.py:63
// in IEEE fp64 with the reference's operation order (vec3.cuh), so chains and iteration counts equal a plain C or
// Python restatement of the loop bit for bit.  A row's result is a pure function of the row.
//
// Design (DESIGN.md "Fabrik.calculate for J-point chains"):
//  * Persistent warps with per-lane refill.  Iteration counts are bimodal (a few passes for a reachable goal, exactly
//    max_iter for an unreachable one), so a lane whose row finishes stores its chain and takes the next row in the same
//    step: one warp-aggregated atomicAdd of popc(ballot) on a 64-bit work counter.  The pass itself is branch-free at
//    full warp width (lanes without a row compute on stale registers and write nothing).
//  * Statistics are accumulated in registers and flushed with one atomic per warp and counter.
//  * J <= IKB_CHAIN_JREG: one instantiation per J with the chain in registers, updated in place.  Larger J: one
//    runtime-length instantiation of the same source with the chain in local memory.
#include <array>
#include <utility>

#include "ikb_common.cuh"
#include "vec3.cuh"

#ifndef IKB_CHAIN_JREG
#define IKB_CHAIN_JREG 32
#endif
#define IKB_CHAIN_THREADS 256

namespace {

struct ChainArgs {
    const double *init;  // n_init x J x 3 (n_init is 1 or n)
    long long n_init;
    const double *goals;  // n x 3
    long long n;
    long long index_base;  // global row of goals[0] (host pipeline chunks): the row numbers in the statistics
    double *chain_out;     // n x J x 3
    int *iters;            // nullable
    IkbDeviceStats *stats;
    unsigned long long *work_counter;  // zero at launch
    double tol;
    int max_iter;
    int J;
    int fresh_go;  // (1 > tol) and (max_iter > 0): whether a freshly loaded row takes a pass at all
    double d[IKB_CHAIN_MAX_POINTS];
};

// JR > 0: the chain has exactly JR points and lives in registers; JR == 0: a.J points in local memory
template <int JR>
__global__ void __launch_bounds__(IKB_CHAIN_THREADS) fabrik_chain_kernel(const ChainArgs a)
{
    constexpr int JA = JR > 0 ? JR : IKB_CHAIN_MAX_POINTS;
    constexpr int UNROLL = JR > 0 ? JR : 1;
    const int J = JR > 0 ? JR : a.J;
    const int lane = threadIdx.x & 31;
    const unsigned lt = ikb_lanemask_lt();
    Vec3 P[JA];
    Vec3 S{0, 0, 0}, T{0, 0, 0};
    long long row = 0;
    int k = 0;
    double se = 1.0, ge = 1.0;
    bool live = false, exhausted = false;
    unsigned long long n_solved = 0, sum_k = 0, capped = 0;
    long long first_zero = IKB_I64_MAX;

    for (;;) {
        const bool go = ((se > a.tol) | (ge > a.tol)) & (a.max_iter > k);  // fabrik.py:57-59
        if (live & !go) {
            double *o = a.chain_out + 3LL * J * row;
            bool bad = false;
#pragma unroll UNROLL
            for (int j = 0; j < J; ++j) {
                o[3 * j] = P[j].x; o[3 * j + 1] = P[j].y; o[3 * j + 2] = P[j].z;
                bad |= !(isfinite(P[j].x) & isfinite(P[j].y) & isfinite(P[j].z));
            }
            if (a.iters)
                a.iters[row] = k;
            // a segment of length 0 (ZeroDivisionError upstream, point.py:40) leaves a non-finite chain
            if (bad & isfinite(T.x) & isfinite(T.y) & isfinite(T.z))
                first_zero = min(first_zero, a.index_base + row);
            ++n_solved;
            sum_k += (unsigned)k;
            capped += (((se > a.tol) | (ge > a.tol)) & (k > 0)) ? 1u : 0u;
            live = false;
        }
        if (!exhausted) {  // refill: every lane without a row takes the next one
            const unsigned want = __ballot_sync(IKB_FULL_MASK, !live);
            if (want) {
                unsigned long long base = 0;
                if (lane == 0)
                    base = atomicAdd(a.work_counter, (unsigned long long)__popc(want));
                base = __shfl_sync(IKB_FULL_MASK, base, 0);
                if (!live) {
                    const long long r = (long long)base + __popc(want & lt);
                    if (r < a.n) {
                        const double *ip = a.init + (a.n_init == 1 ? 0LL : 3LL * J * r);
#pragma unroll UNROLL
                        for (int j = 0; j < J; ++j)
                            P[j] = Vec3{__ldg(ip + 3 * j), __ldg(ip + 3 * j + 1), __ldg(ip + 3 * j + 2)};
                        S = P[0];
                        const double *g = a.goals + 3 * r;
                        T = Vec3{__ldg(g), __ldg(g + 1), __ldg(g + 2)};
                        row = r;
                        k = 0;
                        se = ge = 1.0;
                        live = true;
                    }
                }
                exhausted = (long long)(base + __popc(want)) >= a.n;
            }
        }
        if (__ballot_sync(IKB_FULL_MASK, live) == 0)
            break;
        if (!a.fresh_go)  // no row takes a pass (tol >= 1 or max_iter <= 0): store the initial chains
            continue;
        // one pass on every lane: each live row has go == true here (finished rows were just replaced)
        Vec3 b = T;
#pragma unroll UNROLL
        for (int j = J - 2; j >= 0; --j) {
            b = point_between3(b, P[j], a.d[j]);
            P[j] = b;
        }
        se = dist3(P[0], S);
        P[0] = S;
#pragma unroll UNROLL
        for (int j = 1; j < J - 1; ++j)
            P[j] = point_between3(P[j - 1], P[j], a.d[j]);
        if (J > 1)
            P[J - 1] = point_between3(P[J - 2], T, a.d[J - 1]);
        ge = dist3(P[J - 1], T);
        ++k;
    }

    // statistics: one atomic per warp and counter
    n_solved = ikb_warp_sum(n_solved);
    sum_k = ikb_warp_sum(sum_k);
    capped = ikb_warp_sum(capped);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
        first_zero = min(first_zero, __shfl_xor_sync(IKB_FULL_MASK, first_zero, o));
    if (lane == 0 && n_solved != 0) {
        atomicAdd(&a.stats->n_solved, n_solved);
        atomicAdd(&a.stats->sum_iterations, sum_k);
        if (capped)
            atomicAdd(&a.stats->n_iter_capped, capped);
        if (first_zero != IKB_I64_MAX)
            atomicMin(&a.stats->first_zero_division, first_zero);
    }
}

using ChainKernel = void (*)(ChainArgs);

template <size_t... I>
constexpr std::array<ChainKernel, sizeof...(I)> chain_kernels(std::index_sequence<I...>)
{
    return {{&fabrik_chain_kernel<(int)I>...}};
}
// index J for 1 <= J <= IKB_CHAIN_JREG, index 0 (runtime length) above
constexpr std::array<ChainKernel, IKB_CHAIN_JREG + 1> kChainKernels =
    chain_kernels(std::make_index_sequence<IKB_CHAIN_JREG + 1>());

}  // namespace

// work_counter: a counter of the engine's ring (reset here).  links: n_points doubles in host memory.
cudaError_t ikb_launch_fabrik_chain(int n_points, const double *links, double tol, int max_iter, const double *init,
                                    long long n_init, const double *goals, long long n, long long index_base,
                                    double *chain_out, int *iters, IkbDeviceStats *stats,
                                    unsigned long long *work_counter, int num_sms, cudaStream_t stream)
{
    if (n <= 0)
        return cudaSuccess;
    ChainArgs a;
    a.init = init; a.n_init = n_init; a.goals = goals; a.n = n; a.index_base = index_base;
    a.chain_out = chain_out; a.iters = iters; a.stats = stats; a.work_counter = work_counter;
    a.tol = tol; a.max_iter = max_iter; a.J = n_points;
    a.fresh_go = (1.0 > tol) && (max_iter > 0);
    for (int j = 0; j < IKB_CHAIN_MAX_POINTS; ++j)
        a.d[j] = j < n_points ? links[j] : 0.0;
    const int idx = n_points <= IKB_CHAIN_JREG ? n_points : 0;
    const ChainKernel kern = kChainKernels[idx];
    static int blocks_per_sm[IKB_CHAIN_JREG + 1] = {};
    if (blocks_per_sm[idx] == 0) {
        cudaError_t err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks_per_sm[idx], kern, IKB_CHAIN_THREADS, 0);
        if (err != cudaSuccess)
            return err;
        if (blocks_per_sm[idx] < 1)
            blocks_per_sm[idx] = 1;
    }
    cudaError_t err = cudaMemsetAsync(work_counter, 0, sizeof(unsigned long long), stream);
    if (err != cudaSuccess)
        return err;
    // persistent grid: resident CTAs per SM x SM count, trimmed for small batches
    long long grid = (long long)num_sms * blocks_per_sm[idx];
    const long long want = (n + IKB_CHAIN_THREADS - 1) / IKB_CHAIN_THREADS;
    if (want < grid)
        grid = want;
    kern<<<(unsigned)grid, IKB_CHAIN_THREADS, 0, stream>>>(a);
    return cudaGetLastError();
}

// capi.cu -- the C ABI of libikb200 (include/ikb200.h): engine lifetime, statistics, host-side
// H2D -> kernel -> D2H pipelines.  No torch types, no CPU fallback: every compute entry point
// needs a CUDA device.
#include <cmath>
#include <cstdio>
#include <algorithm>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#include "ikb_common.cuh"
#include "mlp.cuh"

// launchers implemented next to their kernels
cudaError_t ikb_launch_fabrik_planar(const void *xyz, int xyz_f64, long long n, long long index_base,
                                     void *angles, int angles_f64, int *iters, void *fk_err, int fk_stats,
                                     int precision, IkbDeviceStats *stats, unsigned long long *work_counter,
                                     const IkbRobot &rc, int num_sms, cudaStream_t stream);
cudaError_t ikb_launch_fabrik_chain(int n_points, const double *links, double tol, int max_iter, const double *init,
                                    long long n_init, const double *goals, long long n, long long index_base,
                                    double *chain_out, int *iters, IkbDeviceStats *stats,
                                    unsigned long long *work_counter, int num_sms, cudaStream_t stream);
cudaError_t ikb_launch_fabrik_generic_ikine(const void *xyz, int xyz_f64, long long n, long long index_base,
                                            void *angles, int angles_f64, int *iters, IkbDeviceStats *stats,
                                            const IkbRobot &rc, cudaStream_t stream);
cudaError_t ikb_launch_fk(const void *angles, int angles_f64, long long n, long long index_base,
                          void *pos_out, const void *targets, int xyz_f64, void *err_out,
                          IkbDeviceStats *stats, const IkbRobot &rc, int num_sms, cudaStream_t stream);
cudaError_t ikb_launch_fk_transforms(const void *angles, int angles_f64, long long n, long long index_base, int what,
                                     void *out, IkbDeviceStats *stats, const IkbRobot &rc, int num_sms,
                                     cudaStream_t stream);
cudaError_t ikb_launch_jacobian(const void *angles, int angles_f64, long long n, long long index_base, int what,
                                void *jac, void *manip, IkbDeviceStats *stats, const IkbRobot &rc, int num_sms,
                                cudaStream_t stream);
cudaError_t ikb_launch_dls_refine(const void *xyz, int xyz_f64, const void *seed, long long n_seed, void *angles_out,
                                  int angles_f64, int *iters, void *err_out, long long n, long long index_base,
                                  double damping, double tol, int max_iter, IkbDeviceStats *stats,
                                  unsigned long long *work_counter, const IkbRobot &rc, int num_sms,
                                  cudaStream_t stream);
cudaError_t ikb_launch_dls_pose_refine(const void *poses, int pose_f64, const void *seed, long long n_seed,
                                       void *angles_out, int angles_f64, int *iters, void *err_out, long long n,
                                       long long index_base, const double weights[6], double damping, double tol,
                                       int max_iter, IkbDeviceStats *stats, unsigned long long *work_counter,
                                       const IkbRobot &rc, int num_sms, cudaStream_t stream);
cudaError_t ikb_launch_analytic_ik(int kind, const void *in, int in_f64, long long n, long long index_base,
                                   const void *pitch, int per_row_pitch, void *angles_out, int angles_f64,
                                   int *status, IkbDeviceStats *stats, const IkbRobot &rc, int num_sms,
                                   cudaStream_t stream);
cudaError_t ikb_launch_check_limits(const void *xyz, int xyz_f64, long long n, long long index_base,
                                    IkbDeviceStats *stats, const IkbRobot &rc, int num_sms,
                                    cudaStream_t stream);
cudaError_t ikb_launch_fma_peak(int f64, void *sink, int iters, int num_sms, cudaStream_t stream);
cudaError_t ikb_launch_generate(int kind, const double *params, int n_params, long long n, long long row_offset,
                                void *out, int out_f64, unsigned long long seed, int num_sms, cudaStream_t stream);

namespace {

constexpr int kCounterRing = 16;
constexpr long long kHostChunkRows = 1LL << 22;  // rows per pipeline stage of the *_host entry points

// Rows of the pipeline stage that starts at row `lo`: full-size stages, except that a long call ramps up through two
// short ones so that the device-to-host stream (the PCIe-bound direction: 16 B of angles per row) starts after a
// tenth of a stage time instead of a whole one.
inline long long host_chunk_rows(long long lo, long long n)
{
    long long m = kHostChunkRows;
    if (n > 4 * kHostChunkRows) {
        if (lo == 0)
            m = kHostChunkRows / 8;
        else if (lo == kHostChunkRows / 8)
            m = kHostChunkRows / 2;
    }
    return std::min<long long>(m, n - lo);
}
constexpr int kSlots = 3;

std::string g_create_error;

struct Slot {
    cudaStream_t stream = nullptr;
    void *d_in = nullptr;    // kHostChunkRows x 4 doubles: holds xyz (3) or angles (4), f32 or f64
    void *d_in2 = nullptr;   // second input (FK targets)
    void *d_out = nullptr;   // kHostChunkRows x 4 doubles
    int *d_aux = nullptr;    // kHostChunkRows ints (iterations) / floats (fk error)
};

}  // namespace

struct ikb_engine {
    ikb_config cfg;
    IkbRobot rc;
    int device = 0;
    int num_sms = 0;
    IkbDeviceStats *d_stats = nullptr;
    IkbDeviceStats *h_stats = nullptr;  // pinned
    unsigned long long *d_counters = nullptr;     // kCounterRing work counters of the persistent kernels
    cudaEvent_t counter_free[kCounterRing] = {};  // recorded after the last launch that used each counter
    int counter_seq = 0;
    Slot slots[kSlots];
    long long slot_rows = 0;  // current capacity of every slot buffer, grows on demand
    IkbMlp mlp;
    std::string err;
    long long launches = 0;
    bool analytic_family = false;  // the DH table has the closed-form inverse kinematics of ikb_analytic_ik_*
};

namespace {

int fail(ikb_engine *e, int code, const std::string &msg)
{
    if (e)
        e->err = msg;
    else
        g_create_error = msg;
    return code;
}

#define IKB_CUDA(e, call)                                                                         \
    do {                                                                                          \
        cudaError_t _err = (call);                                                                \
        if (_err != cudaSuccess)                                                                  \
            return fail((e), IKB_ERR_CUDA,                                                        \
                        std::string(#call) + ": " + cudaGetErrorString(_err));                    \
    } while (0)

IkbDeviceStats fresh_stats()
{
    IkbDeviceStats s;
    memset(&s, 0, sizeof s);
    s.first_out_of_limits = s.first_zero_division = s.first_domain_error = s.first_fk_angle_range =
        IKB_I64_MAX;
    return s;
}

void to_public(const IkbDeviceStats &d, ikb_stats *o)
{
    auto idx = [](long long v) { return v == IKB_I64_MAX ? (int64_t)-1 : (int64_t)v; };
    o->n_solved = (int64_t)d.n_solved;
    o->sum_iterations = (int64_t)d.sum_iterations;
    o->n_iter_capped = (int64_t)d.n_iter_capped;
    o->first_out_of_limits = idx(d.first_out_of_limits);
    o->first_zero_division = idx(d.first_zero_division);
    o->first_domain_error = idx(d.first_domain_error);
    o->first_fk_angle_range = idx(d.first_fk_angle_range);
    o->sum_fk_error = d.sum_fk_error;
    o->n_fk_error = (int64_t)d.n_fk_error;
}

// The work counter of the next persistent launch, taken round-robin from the engine's ring.  Launches on different
// streams may overlap, so a counter is only handed out once the last launch that used it has finished: `stream` first
// waits for that launch's event (a no-op for an event that was never recorded).  After the launch, call
// counter_release(e, slot, stream) with the slot returned here.
cudaError_t counter_claim(ikb_engine *e, cudaStream_t stream, unsigned long long **counter, int *slot)
{
    *slot = e->counter_seq % kCounterRing;
    e->counter_seq++;
    *counter = e->d_counters + *slot;
    return cudaStreamWaitEvent(stream, e->counter_free[*slot], 0);
}

cudaError_t counter_release(ikb_engine *e, int slot, cudaStream_t stream)
{
    return cudaEventRecord(e->counter_free[slot], stream);
}

// staging buffers of the host pipelines: sized for min(rows, kHostChunkRows), grown on demand
int ensure_slots(ikb_engine *e, long long rows)
{
    long long want = 1024;
    while (want < rows && want < kHostChunkRows)
        want <<= 1;
    if (want <= e->slot_rows)
        return IKB_OK;
    for (int i = 0; i < kSlots; ++i) {
        Slot &s = e->slots[i];
        if (!s.stream)
            IKB_CUDA(e, cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking));
        IKB_CUDA(e, cudaStreamSynchronize(s.stream));
        if (s.d_in) cudaFree(s.d_in);
        if (s.d_in2) cudaFree(s.d_in2);
        if (s.d_out) cudaFree(s.d_out);
        if (s.d_aux) cudaFree(s.d_aux);
        s.d_in = s.d_in2 = s.d_out = nullptr;
        s.d_aux = nullptr;
        IKB_CUDA(e, cudaMalloc(&s.d_in, want * 4 * sizeof(double)));
        IKB_CUDA(e, cudaMalloc(&s.d_in2, want * 3 * sizeof(double)));
        IKB_CUDA(e, cudaMalloc(&s.d_out, want * 4 * sizeof(double)));
        IKB_CUDA(e, cudaMalloc(&s.d_aux, want * sizeof(int)));
    }
    e->slot_rows = want;
    return IKB_OK;
}

int host_begin(ikb_engine *e, long long rows)
{
    IKB_CUDA(e, cudaSetDevice(e->device));
    int rc = ensure_slots(e, rows);
    if (rc)
        return rc;
    *e->h_stats = fresh_stats();
    IKB_CUDA(e, cudaMemcpy(e->d_stats, e->h_stats, sizeof(IkbDeviceStats), cudaMemcpyHostToDevice));
    return IKB_OK;
}

int host_end(ikb_engine *e, ikb_stats *stats)
{
    for (int i = 0; i < kSlots; ++i)
        IKB_CUDA(e, cudaStreamSynchronize(e->slots[i].stream));
    IKB_CUDA(e, cudaMemcpy(e->h_stats, e->d_stats, sizeof(IkbDeviceStats), cudaMemcpyDeviceToHost));
    if (stats)
        to_public(*e->h_stats, stats);
    return IKB_OK;
}

size_t esize(int dtype) { return dtype == IKB_F64 ? sizeof(double) : sizeof(float); }

bool bad_dtype(int d) { return d != IKB_F32 && d != IKB_F64; }

}  // namespace

extern "C" {

const char *ikb_version(void) { return "ikb200 0.1 sm_100a"; }

int ikb_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess)
        return 0;
    return n;
}

const char *ikb_last_error(const ikb_engine *e) { return e ? e->err.c_str() : g_create_error.c_str(); }

int64_t ikb_launch_count(const ikb_engine *e) { return e ? e->launches : 0; }

int ikb_engine_create(const ikb_config *cfg, ikb_engine **out)
{
    if (!cfg || !out)
        return fail(nullptr, IKB_ERR_INVALID, "ikb_engine_create: NULL argument");
    *out = nullptr;
    int ndev = 0;
    cudaError_t cerr = cudaGetDeviceCount(&ndev);
    if (cerr != cudaSuccess || ndev == 0)
        return fail(nullptr, IKB_ERR_CUDA,
                    std::string("no CUDA device: libikb200 has no CPU fallback (") +
                        cudaGetErrorString(cerr) + ")");
    if (cfg->device < 0 || cfg->device >= ndev)
        return fail(nullptr, IKB_ERR_INVALID, "ikb_engine_create: device ordinal out of range");
    ikb_engine *e = new (std::nothrow) ikb_engine();
    if (!e)
        return fail(nullptr, IKB_ERR_INVALID, "out of host memory");
    e->cfg = *cfg;
    e->device = cfg->device;
    auto bail = [&](int code) {
        g_create_error = e->err;
        ikb_engine_destroy(e);
        return code;
    };
#define IKB_CREATE_CUDA(call)                                                                     \
    do {                                                                                          \
        cudaError_t _err = (call);                                                                \
        if (_err != cudaSuccess) {                                                                \
            e->err = std::string(#call) + ": " + cudaGetErrorString(_err);                        \
            return bail(IKB_ERR_CUDA);                                                            \
        }                                                                                         \
    } while (0)
    IKB_CREATE_CUDA(cudaSetDevice(e->device));
    cudaDeviceProp prop;
    IKB_CREATE_CUDA(cudaGetDeviceProperties(&prop, e->device));
    e->num_sms = prop.multiProcessorCount;
    IKB_CREATE_CUDA(cudaMalloc(&e->d_stats, sizeof(IkbDeviceStats)));
    IKB_CREATE_CUDA(cudaMallocHost(&e->h_stats, sizeof(IkbDeviceStats)));
    IKB_CREATE_CUDA(cudaMalloc(&e->d_counters, kCounterRing * sizeof(unsigned long long)));
    for (int i = 0; i < kCounterRing; ++i)
        IKB_CREATE_CUDA(cudaEventCreateWithFlags(&e->counter_free[i], cudaEventDisableTiming));
    *e->h_stats = fresh_stats();
    IKB_CREATE_CUDA(cudaMemcpy(e->d_stats, e->h_stats, sizeof(IkbDeviceStats), cudaMemcpyHostToDevice));

    IkbRobot &rc = e->rc;
    memset(&rc, 0, sizeof rc);
    for (int j = 0; j < 4; ++j) {
        rc.links[j] = cfg->links[j];
        rc.eps[j] = cfg->dh[4 + j];
        rc.a[j] = cfg->dh[8 + j];
        rc.alpha[j] = cfg->dh[12 + j];
        rc.cos_alpha[j] = std::cos(rc.alpha[j]);
        rc.sin_alpha[j] = std::sin(rc.alpha[j]);
    }
    rc.fk_planar_tail = (rc.alpha[1] == 0.0 && rc.alpha[2] == 0.0 && rc.alpha[3] == 0.0) ? 1 : 0;
    for (int j = 0; j < 4; ++j)
        rc.link_k[j] = ikb_scaled_rsqrt_constants(cfg->links[j]);
    {
        const double fkc[8] = {rc.a[0], rc.a[1], rc.a[2], rc.a[3], rc.eps[0], rc.eps[1] + rc.eps[2] + rc.eps[3],
                               rc.cos_alpha[0], rc.sin_alpha[0]};
        for (int j = 0; j < 8; ++j) {
            rc.fkc[j] = fkc[j];
            rc.fkc_f[j] = (float)fkc[j];
        }
    }
    for (int j = 0; j < 6; ++j)
        rc.limits[j] = cfg->limits[j];
    rc.tol = cfg->tol;
    for (int j = 0; j < 2; ++j) {
        const double d = cfg->links[j == 0 ? 0 : 3];
        const double lo = d - cfg->tol, hi = d + cfg->tol;
        rc.band_lo2[j] = lo > 0.0 ? lo * lo : -1.0;  // -1: every squared length is above the lower edge
        rc.band_hi2[j] = hi * hi;
        rc.band_lo2_f[j] = (float)rc.band_lo2[j];
        rc.band_hi2_f[j] = (float)rc.band_hi2[j];
    }
    rc.max_iter = cfg->max_iter;
    rc.zero_iter = (!(1.0 > cfg->tol) || cfg->max_iter <= 0) ? 1 : 0;  // fabrik.py:54-59
    // seed chain: FK of [0, dh[0][1], dh[0][2], dh[0][3]] on the device (inverse.py:123-130)
    {
        double seed[4] = {0.0, cfg->dh[1], cfg->dh[2], cfg->dh[3]};
        double chain[64];
        double *d_ang = nullptr, *d_chain = nullptr;
        IKB_CREATE_CUDA(cudaMalloc(&d_ang, sizeof seed));
        IKB_CREATE_CUDA(cudaMalloc(&d_chain, sizeof chain));
        IKB_CREATE_CUDA(cudaMemcpy(d_ang, seed, sizeof seed, cudaMemcpyHostToDevice));
        IKB_CREATE_CUDA(ikb_launch_fk_transforms(d_ang, 1, 1, 0, IKB_FK_MATRICES, d_chain, e->d_stats, rc, e->num_sms,
                                                 nullptr));
        e->launches++;
        IKB_CREATE_CUDA(cudaMemcpy(chain, d_chain, sizeof chain, cudaMemcpyDeviceToHost));
        IKB_CREATE_CUDA(cudaMemcpy(e->h_stats, e->d_stats, sizeof(IkbDeviceStats), cudaMemcpyDeviceToHost));
        const bool status = e->h_stats->first_fk_angle_range != IKB_I64_MAX;
        // the guard of the seed chain is the engine's business, not its callers': start them with a clean block
        *e->h_stats = fresh_stats();
        IKB_CREATE_CUDA(cudaMemcpy(e->d_stats, e->h_stats, sizeof(IkbDeviceStats), cudaMemcpyHostToDevice));
        cudaFree(d_ang); cudaFree(d_chain);
        rc.planar = 1;
        for (int j = 0; j < 4; ++j) {
            const double x = chain[16 * j + 3], y = chain[16 * j + 7], z = chain[16 * j + 11];
            rc.seed_xyz[3 * j] = x; rc.seed_xyz[3 * j + 1] = y; rc.seed_xyz[3 * j + 2] = z;
            rc.seed_r[j] = x; rc.seed_z[j] = z;
            if (std::fabs(y) > 1e-9 || !(std::fabs(x) < 1e300))
                rc.planar = 0;
        }
        if (status)
            rc.planar = 0;
        e->analytic_family = rc.fk_planar_tail && std::fabs(rc.cos_alpha[0]) <= 1e-12 && rc.a[1] > 0.0 &&
                             rc.a[2] > 0.0;
        rc.seed_ab = std::sqrt(rc.seed_r[0] * rc.seed_r[0] + rc.seed_z[0] * rc.seed_z[0]);
        rc.seed_ab2 = rc.seed_ab * rc.seed_ab;
        rc.half_inv_ab = 0.5 / rc.seed_ab;
        const double d1 = cfg->links[1], d2 = cfg->links[2], d3 = cfg->links[3];
        rc.cos_sum[0] = rc.seed_ab2 + d1 * d1; rc.cos_inv[0] = 1.0 / (2.0 * rc.seed_ab * d1);
        rc.cos_sum[1] = d1 * d1 + d2 * d2;     rc.cos_inv[1] = 1.0 / (2.0 * d1 * d2);
        rc.cos_sum[2] = d2 * d2 + d3 * d3;     rc.cos_inv[2] = 1.0 / (2.0 * d2 * d3);
    }
    *out = e;
    return IKB_OK;
#undef IKB_CREATE_CUDA
}

void ikb_engine_destroy(ikb_engine *e)
{
    if (!e)
        return;
    cudaSetDevice(e->device);
    for (int i = 0; i < kSlots; ++i) {
        Slot &s = e->slots[i];
        if (s.stream) cudaStreamSynchronize(s.stream);
        if (s.d_in) cudaFree(s.d_in);
        if (s.d_in2) cudaFree(s.d_in2);
        if (s.d_out) cudaFree(s.d_out);
        if (s.d_aux) cudaFree(s.d_aux);
        if (s.stream) cudaStreamDestroy(s.stream);
    }
    ikb_mlp_free(e->mlp);
    if (e->d_stats) cudaFree(e->d_stats);
    if (e->h_stats) cudaFreeHost(e->h_stats);
    if (e->d_counters) cudaFree(e->d_counters);
    for (int i = 0; i < kCounterRing; ++i)
        if (e->counter_free[i]) cudaEventDestroy(e->counter_free[i]);
    delete e;
}

int ikb_stats_reset(ikb_engine *e, void *stream)
{
    if (!e)
        return IKB_ERR_INVALID;
    IKB_CUDA(e, cudaSetDevice(e->device));
    cudaStream_t st = (cudaStream_t)stream;
    // h_stats may still be in flight from a previous async copy on another stream: use a
    // stack copy through a synchronous-with-respect-to-host memcpy on this stream
    IkbDeviceStats s = fresh_stats();
    IKB_CUDA(e, cudaMemcpyAsync(e->d_stats, &s, sizeof s, cudaMemcpyHostToDevice, st));
    IKB_CUDA(e, cudaStreamSynchronize(st));
    return IKB_OK;
}

int ikb_stats_fetch(ikb_engine *e, void *stream, ikb_stats *out)
{
    if (!e || !out)
        return IKB_ERR_INVALID;
    IKB_CUDA(e, cudaSetDevice(e->device));
    cudaStream_t st = (cudaStream_t)stream;
    IKB_CUDA(e, cudaMemcpyAsync(e->h_stats, e->d_stats, sizeof(IkbDeviceStats), cudaMemcpyDeviceToHost, st));
    IKB_CUDA(e, cudaStreamSynchronize(st));
    to_public(*e->h_stats, out);
    return IKB_OK;
}

// ---- check_limits ---------------------------------------------------------------------------------
int ikb_check_limits_device(ikb_engine *e, const void *xyz, int xyz_dtype, int64_t n, void *stream)
{
    if (!e || n < 0 || (n > 0 && !xyz) || bad_dtype(xyz_dtype))
        return fail(e, IKB_ERR_INVALID, "ikb_check_limits_device: bad argument");
    IKB_CUDA(e, cudaSetDevice(e->device));
    IKB_CUDA(e, ikb_launch_check_limits(xyz, xyz_dtype == IKB_F64, n, 0, e->d_stats, e->rc, e->num_sms,
                                        (cudaStream_t)stream));
    e->launches += (n > 0);
    return IKB_OK;
}

int ikb_check_limits_host(ikb_engine *e, const void *xyz, int xyz_dtype, int64_t n, int64_t *first_bad)
{
    if (!e || n < 0 || (n > 0 && !xyz) || bad_dtype(xyz_dtype) || !first_bad)
        return fail(e, IKB_ERR_INVALID, "ikb_check_limits_host: bad argument");
    int rc = host_begin(e, n);
    if (rc)
        return rc;
    const size_t row = 3 * esize(xyz_dtype);
    int it = 0;
    for (long long lo = 0, m = 0; lo < n; lo += m, ++it) {
        Slot &s = e->slots[it % kSlots];
        m = host_chunk_rows(lo, n);
        IKB_CUDA(e, cudaMemcpyAsync(s.d_in, (const char *)xyz + lo * row, m * row, cudaMemcpyHostToDevice, s.stream));
        IKB_CUDA(e, ikb_launch_check_limits(s.d_in, xyz_dtype == IKB_F64, m, lo, e->d_stats, e->rc,
                                            e->num_sms, s.stream));
        e->launches++;
    }
    ikb_stats st;
    rc = host_end(e, &st);
    *first_bad = st.first_out_of_limits;
    return rc;
}

// ---- FABRIK ---------------------------------------------------------------------------------------
// K1's fused error epilogue uses the closed-form FK (joints 2..4 about parallel axes, alpha inside the guard of
// forward.py:23-25); any other DH table gets K3 as a second launch.
// Measured on B200 (100 M rows): the fused epilogue adds 2.2 ms to the 21.2 ms solve (K1 is latency-bound on the
// fp64 pipe with a tight register budget, and the extra fp32 work competes for its issue slots), K3 as a second launch
// 0.8 ms (it runs at HBM speed while K1 hardly touches HBM); at 1e5 rows 21 us against 12 us, at 4096 rows 12 us
// against 5 us.  So the fusion only pays while the saved launch dominates: CLI-sized batches.
constexpr long long kFuseFkMaxRows = 1LL << 10;
static bool fk_fusable(const IkbRobot &rc, long long rows)
{
    bool ok = rc.fk_planar_tail != 0 && rows <= kFuseFkMaxRows;
    for (int j = 0; j < 4; ++j)
        ok = ok && !(rc.alpha[j] < -6.283185307179586) && !(rc.alpha[j] > 6.283185307179586);
    return ok;
}

int ikb_fabrik_solve_device(ikb_engine *e, const void *xyz, int xyz_dtype, int64_t n, void *angles_out,
                            int angles_dtype, int32_t *iters_out, void *fk_err_out, int fk_stats, int precision,
                            void *stream)
{
    if (!e || n < 0 || (n > 0 && (!xyz || !angles_out)) || bad_dtype(xyz_dtype) || bad_dtype(angles_dtype) ||
        (precision != IKB_FABRIK_F64 && precision != IKB_FABRIK_F32) || n > 0x7fffffffLL)
        return fail(e, IKB_ERR_INVALID, "ikb_fabrik_solve_device: bad argument (n must be < 2^31 per call)");
    if (((uintptr_t)angles_out & 15))  // rows are stored as float4 / double2 pairs
        return fail(e, IKB_ERR_INVALID, "ikb_fabrik_solve_device: angles must be 16-byte aligned");
    IKB_CUDA(e, cudaSetDevice(e->device));
    const bool want_fk = n > 0 && (fk_err_out || fk_stats);
    const bool fuse = want_fk && e->rc.planar && fk_fusable(e->rc, n);
    if (!e->rc.planar) {  // general DH table: the seed chain leaves the vertical plane -> 3-D kernel
        IKB_CUDA(e, ikb_launch_fabrik_generic_ikine(xyz, xyz_dtype == IKB_F64, n, 0, angles_out,
                                                    angles_dtype == IKB_F64, iters_out, e->d_stats, e->rc,
                                                    (cudaStream_t)stream));
    } else {
        unsigned long long *counter;
        int slot;
        IKB_CUDA(e, counter_claim(e, (cudaStream_t)stream, &counter, &slot));
        IKB_CUDA(e, ikb_launch_fabrik_planar(xyz, xyz_dtype == IKB_F64, n, 0, angles_out, angles_dtype == IKB_F64,
                                             iters_out, fuse ? fk_err_out : nullptr, fuse ? fk_stats : 0, precision,
                                             e->d_stats, counter, e->rc, e->num_sms, (cudaStream_t)stream));
        IKB_CUDA(e, counter_release(e, slot, (cudaStream_t)stream));
    }
    if (want_fk && !fuse) {  // no closed-form FK for this DH table: K3 as a second launch
        IKB_CUDA(e, ikb_launch_fk(angles_out, angles_dtype == IKB_F64, n, 0, nullptr, xyz, xyz_dtype == IKB_F64,
                                  fk_err_out, e->d_stats, e->rc, e->num_sms, (cudaStream_t)stream));
        e->launches++;
    }
    e->launches += (n > 0);
    return IKB_OK;
}

int ikb_fabrik_solve_host(ikb_engine *e, const void *xyz, int xyz_dtype, int64_t n, void *angles_out,
                          int angles_dtype, int32_t *iters_out, void *fk_err_out, int fk_stats, int precision,
                          ikb_stats *stats)
{
    if (!e || n < 0 || (n > 0 && (!xyz || !angles_out)) || bad_dtype(xyz_dtype) || bad_dtype(angles_dtype) ||
        (precision != IKB_FABRIK_F64 && precision != IKB_FABRIK_F32))
        return fail(e, IKB_ERR_INVALID, "ikb_fabrik_solve_host: bad argument");
    int rc = host_begin(e, n);
    if (rc)
        return rc;
    const size_t in_row = 3 * esize(xyz_dtype), out_row = 4 * esize(angles_dtype), err_row = esize(angles_dtype);
    const bool want_fk = fk_err_out || fk_stats;
    const bool fuse = want_fk && e->rc.planar && fk_fusable(e->rc, n);
    int it = 0;
    for (long long lo = 0, m = 0; lo < n; lo += m, ++it) {
        Slot &s = e->slots[it % kSlots];
        m = host_chunk_rows(lo, n);
        void *d_err = fk_err_out ? s.d_in2 : nullptr;  // d_in2 is free here (FK targets only)
        IKB_CUDA(e, cudaMemcpyAsync(s.d_in, (const char *)xyz + lo * in_row, m * in_row, cudaMemcpyHostToDevice, s.stream));
        if (!e->rc.planar) {
            IKB_CUDA(e, ikb_launch_fabrik_generic_ikine(s.d_in, xyz_dtype == IKB_F64, m, lo, s.d_out,
                                                        angles_dtype == IKB_F64, iters_out ? s.d_aux : nullptr,
                                                        e->d_stats, e->rc, s.stream));
        } else {
            unsigned long long *counter;
            int slot;
            IKB_CUDA(e, counter_claim(e, s.stream, &counter, &slot));
            IKB_CUDA(e, ikb_launch_fabrik_planar(s.d_in, xyz_dtype == IKB_F64, m, lo, s.d_out,
                                                 angles_dtype == IKB_F64, iters_out ? s.d_aux : nullptr,
                                                 fuse ? d_err : nullptr, fuse ? fk_stats : 0, precision, e->d_stats,
                                                 counter, e->rc, e->num_sms, s.stream));
            IKB_CUDA(e, counter_release(e, slot, s.stream));
        }
        if (want_fk && !fuse) {
            IKB_CUDA(e, ikb_launch_fk(s.d_out, angles_dtype == IKB_F64, m, lo, nullptr, s.d_in, xyz_dtype == IKB_F64,
                                      d_err, e->d_stats, e->rc, e->num_sms, s.stream));
            e->launches++;
        }
        e->launches++;
        IKB_CUDA(e, cudaMemcpyAsync((char *)angles_out + lo * out_row, s.d_out, m * out_row, cudaMemcpyDeviceToHost, s.stream));
        if (iters_out)
            IKB_CUDA(e, cudaMemcpyAsync(iters_out + lo, s.d_aux, m * sizeof(int), cudaMemcpyDeviceToHost, s.stream));
        if (fk_err_out)
            IKB_CUDA(e, cudaMemcpyAsync((char *)fk_err_out + lo * err_row, d_err, m * err_row, cudaMemcpyDeviceToHost, s.stream));
    }
    return host_end(e, stats);
}

// ---- Fabrik.calculate on J-point chains (fabrik.py:44-67) ----------------------------------------
static int chain_args_error(ikb_engine *e, const char *what, int32_t n_points, const double *links, const double *init,
                            int64_t n_init, const double *goals, int64_t n, const double *chain_out)
{
    if (!e)
        return IKB_ERR_INVALID;
    if (n_points < 1 || n_points > IKB_CHAIN_MAX_POINTS)
        return fail(e, IKB_ERR_UNSUPPORTED, std::string(what) + ": n_points must be 1.." +
                                                std::to_string(IKB_CHAIN_MAX_POINTS) + ", got " + std::to_string(n_points));
    if (!links || n < 0 || (n_init != 1 && n_init != n) || (n > 0 && (!init || !goals || !chain_out)))
        return fail(e, IKB_ERR_INVALID, std::string(what) + ": bad argument (n_init must be 1 or n)");
    return IKB_OK;
}

int ikb_fabrik_chain_device(ikb_engine *e, int32_t n_points, const double *links, double tol, int32_t max_iter,
                            const double *init, int64_t n_init, const double *goals, int64_t n, double *chain_out,
                            int32_t *iters_out, void *stream)
{
    int rc = chain_args_error(e, "ikb_fabrik_chain_device", n_points, links, init, n_init, goals, n, chain_out);
    if (rc)
        return rc;
    IKB_CUDA(e, cudaSetDevice(e->device));
    unsigned long long *counter;
    int slot;
    IKB_CUDA(e, counter_claim(e, (cudaStream_t)stream, &counter, &slot));
    IKB_CUDA(e, ikb_launch_fabrik_chain(n_points, links, tol, max_iter, init, n_init, goals, n, 0, chain_out, iters_out,
                                        e->d_stats, counter, e->num_sms, (cudaStream_t)stream));
    IKB_CUDA(e, counter_release(e, slot, (cudaStream_t)stream));
    e->launches += (n > 0);
    return IKB_OK;
}

// Chunks of the host pipeline: goals in d_in2 (3 doubles per slot row), chains in d_out and per-row initial chains in
// d_in (4 doubles per slot row each), iterations in d_aux.  A single initial chain (n_init == 1) is copied to d_in of
// every slot once.
int ikb_fabrik_chain_host(ikb_engine *e, int32_t n_points, const double *links, double tol, int32_t max_iter,
                          const double *init, int64_t n_init, const double *goals, int64_t n, double *chain_out,
                          int32_t *iters_out, ikb_stats *stats)
{
    int rc = chain_args_error(e, "ikb_fabrik_chain_host", n_points, links, init, n_init, goals, n, chain_out);
    if (rc)
        return rc;
    const long long row_doubles = 3LL * n_points;
    rc = host_begin(e, std::max<long long>(n, (n * row_doubles + 3) / 4));
    if (rc)
        return rc;
    const long long m_max = std::max(1LL, std::min(e->slot_rows, 4 * e->slot_rows / row_doubles));
    const bool per_row_init = n_init != 1;
    if (n > 0 && !per_row_init)
        for (int i = 0; i < kSlots; ++i)
            IKB_CUDA(e, cudaMemcpyAsync(e->slots[i].d_in, init, row_doubles * sizeof(double), cudaMemcpyHostToDevice,
                                        e->slots[i].stream));
    int it = 0;
    for (long long lo = 0, m = 0; lo < n; lo += m, ++it) {
        Slot &s = e->slots[it % kSlots];
        m = std::min(m_max, n - lo);
        double *d_init = (double *)s.d_in, *d_goals = (double *)s.d_in2, *d_chain = (double *)s.d_out;
        if (per_row_init)
            IKB_CUDA(e, cudaMemcpyAsync(d_init, init + lo * row_doubles, m * row_doubles * sizeof(double),
                                        cudaMemcpyHostToDevice, s.stream));
        IKB_CUDA(e, cudaMemcpyAsync(d_goals, goals + 3 * lo, m * 3 * sizeof(double), cudaMemcpyHostToDevice, s.stream));
        unsigned long long *counter;
        int slot;
        IKB_CUDA(e, counter_claim(e, s.stream, &counter, &slot));
        IKB_CUDA(e, ikb_launch_fabrik_chain(n_points, links, tol, max_iter, d_init, per_row_init ? m : 1, d_goals, m, lo,
                                            d_chain, iters_out ? s.d_aux : nullptr, e->d_stats, counter, e->num_sms,
                                            s.stream));
        IKB_CUDA(e, counter_release(e, slot, s.stream));
        e->launches++;
        IKB_CUDA(e, cudaMemcpyAsync(chain_out + lo * row_doubles, d_chain, m * row_doubles * sizeof(double),
                                    cudaMemcpyDeviceToHost, s.stream));
        if (iters_out)
            IKB_CUDA(e, cudaMemcpyAsync(iters_out + lo, s.d_aux, m * sizeof(int), cudaMemcpyDeviceToHost, s.stream));
    }
    return host_end(e, stats);
}

int ikb_fabrik_calculate_host(ikb_engine *e, const double *init, int64_t n_init, const double *goals,
                              int64_t n, double *chain_out, int32_t *iters_out, ikb_stats *stats)
{
    if (!e)
        return IKB_ERR_INVALID;
    return ikb_fabrik_chain_host(e, 4, e->rc.links, e->cfg.tol, e->cfg.max_iter, init, n_init, goals, n, chain_out,
                                 iters_out, stats);
}

// ---- forward kinematics ---------------------------------------------------------------------------
int ikb_fk_device(ikb_engine *e, const void *angles, int angles_dtype, int64_t n, void *pos_out,
                  const void *targets, int xyz_dtype, void *err_out, void *stream)
{
    if (!e || n < 0 || (n > 0 && !angles) || bad_dtype(angles_dtype) || bad_dtype(xyz_dtype) ||
        (err_out && !targets))
        return fail(e, IKB_ERR_INVALID, "ikb_fk_device: bad argument");
    if (((uintptr_t)angles & 15))  // rows are loaded as float4 / double2 pairs
        return fail(e, IKB_ERR_INVALID, "ikb_fk_device: angles must be 16-byte aligned");
    IKB_CUDA(e, cudaSetDevice(e->device));
    IKB_CUDA(e, ikb_launch_fk(angles, angles_dtype == IKB_F64, n, 0, pos_out, targets, xyz_dtype == IKB_F64,
                              err_out, e->d_stats, e->rc, e->num_sms, (cudaStream_t)stream));
    e->launches += (n > 0);
    return IKB_OK;
}

int ikb_fk_host(ikb_engine *e, const void *angles, int angles_dtype, int64_t n, void *pos_out,
                const void *targets, int xyz_dtype, void *err_out, ikb_stats *stats)
{
    if (!e || n < 0 || (n > 0 && !angles) || bad_dtype(angles_dtype) || bad_dtype(xyz_dtype) ||
        (err_out && !targets))
        return fail(e, IKB_ERR_INVALID, "ikb_fk_host: bad argument");
    int rc = host_begin(e, n);
    if (rc)
        return rc;
    const size_t a_row = 4 * esize(angles_dtype), p_row = 3 * esize(angles_dtype), t_row = 3 * esize(xyz_dtype);
    const size_t e_row = esize(angles_dtype);
    int it = 0;
    for (long long lo = 0, m = 0; lo < n; lo += m, ++it) {
        Slot &s = e->slots[it % kSlots];
        m = host_chunk_rows(lo, n);
        IKB_CUDA(e, cudaMemcpyAsync(s.d_in, (const char *)angles + lo * a_row, m * a_row, cudaMemcpyHostToDevice, s.stream));
        if (targets)
            IKB_CUDA(e, cudaMemcpyAsync(s.d_in2, (const char *)targets + lo * t_row, m * t_row, cudaMemcpyHostToDevice, s.stream));
        // d_out holds positions (3 per row); errors go behind them in the same buffer
        void *d_err = err_out ? (void *)((char *)s.d_out + e->slot_rows * p_row) : nullptr;
        IKB_CUDA(e, ikb_launch_fk(s.d_in, angles_dtype == IKB_F64, m, lo, pos_out ? s.d_out : nullptr,
                                  targets ? s.d_in2 : nullptr, xyz_dtype == IKB_F64, d_err, e->d_stats,
                                  e->rc, e->num_sms, s.stream));
        e->launches++;
        if (pos_out)
            IKB_CUDA(e, cudaMemcpyAsync((char *)pos_out + lo * p_row, s.d_out, m * p_row, cudaMemcpyDeviceToHost, s.stream));
        if (err_out)
            IKB_CUDA(e, cudaMemcpyAsync((char *)err_out + lo * e_row, d_err, m * e_row, cudaMemcpyDeviceToHost, s.stream));
    }
    return host_end(e, stats);
}

static bool fk_transforms_bad_args(ikb_engine *e, const void *angles, int angles_dtype, int64_t n, int what,
                                   const void *out)
{
    const uintptr_t align = esize(angles_dtype) - 1;
    return !e || n < 0 || (n > 0 && (!angles || !out)) || bad_dtype(angles_dtype) ||
           (what != IKB_FK_MATRICES && what != IKB_FK_JOINTS) || ((uintptr_t)angles & align) || ((uintptr_t)out & align);
}

static size_t fk_transforms_row_bytes(int angles_dtype, int what)
{
    return (what == IKB_FK_JOINTS ? 12 : 64) * esize(angles_dtype);
}

int ikb_fk_transforms_device(ikb_engine *e, const void *angles, int angles_dtype, int64_t n, int what, void *out,
                             void *stream)
{
    if (fk_transforms_bad_args(e, angles, angles_dtype, n, what, out))
        return fail(e, IKB_ERR_INVALID, "ikb_fk_transforms_device: bad argument");
    IKB_CUDA(e, cudaSetDevice(e->device));
    IKB_CUDA(e, ikb_launch_fk_transforms(angles, angles_dtype == IKB_F64, n, 0, what, out, e->d_stats, e->rc,
                                         e->num_sms, (cudaStream_t)stream));
    e->launches += (n > 0);
    return IKB_OK;
}

// Chunks of the host pipeline: angles in d_in (32 B per slot row holds a row of either dtype), results in d_out, as
// many rows as its 32 B per slot row hold at the output row size.
int ikb_fk_transforms_host(ikb_engine *e, const void *angles, int angles_dtype, int64_t n, int what, void *out,
                           ikb_stats *stats)
{
    if (fk_transforms_bad_args(e, angles, angles_dtype, n, what, out))
        return fail(e, IKB_ERR_INVALID, "ikb_fk_transforms_host: bad argument");
    int rc = host_begin(e, n);
    if (rc)
        return rc;
    const size_t in_row = 4 * esize(angles_dtype), out_row = fk_transforms_row_bytes(angles_dtype, what);
    const long long m_max = e->slot_rows * 32 / (long long)out_row;
    int it = 0;
    for (long long lo = 0, m = 0; lo < n; lo += m, ++it) {
        Slot &s = e->slots[it % kSlots];
        m = std::min(m_max, n - lo);
        IKB_CUDA(e, cudaMemcpyAsync(s.d_in, (const char *)angles + lo * in_row, m * in_row, cudaMemcpyHostToDevice,
                                    s.stream));
        IKB_CUDA(e, ikb_launch_fk_transforms(s.d_in, angles_dtype == IKB_F64, m, lo, what, s.d_out, e->d_stats, e->rc,
                                             e->num_sms, s.stream));
        e->launches++;
        IKB_CUDA(e, cudaMemcpyAsync((char *)out + lo * out_row, s.d_out, m * out_row, cudaMemcpyDeviceToHost, s.stream));
    }
    return host_end(e, stats);
}

// ---- arm Jacobian and manipulability --------------------------------------------------------------
// what is wrong with the arguments, or nullptr; the engine is checked last, so that each refusal can be told apart
// without one
static const char *jacobian_bad_args(const ikb_engine *e, const void *angles, int angles_dtype, int64_t n, int what,
                                     const void *jac_out, const void *manip_out)
{
    if (n < 0)
        return "negative n";
    if (bad_dtype(angles_dtype))
        return "unknown dtype";
    if (what != IKB_JAC_GEOMETRIC && what != IKB_JAC_POSITION)
        return "unknown `what`";
    if (!jac_out && !manip_out)
        return "both outputs are NULL";
    if (n > 0 && !angles)
        return "NULL angles";
    const uintptr_t align = esize(angles_dtype) - 1;
    if (((uintptr_t)angles | (uintptr_t)jac_out | (uintptr_t)manip_out) & align)
        return "angles and outputs must be aligned to their element size";
    if (!e)
        return "NULL engine";
    return nullptr;
}

static size_t jacobian_row_bytes(int angles_dtype, int what)
{
    return (what == IKB_JAC_GEOMETRIC ? 24 : 12) * esize(angles_dtype);
}

int ikb_jacobian_device(ikb_engine *e, const void *angles, int angles_dtype, int64_t n, int what, void *jac_out,
                        void *manip_out, void *stream)
{
    if (const char *why = jacobian_bad_args(e, angles, angles_dtype, n, what, jac_out, manip_out))
        return fail(e, IKB_ERR_INVALID, std::string("ikb_jacobian_device: ") + why);
    IKB_CUDA(e, cudaSetDevice(e->device));
    IKB_CUDA(e, ikb_launch_jacobian(angles, angles_dtype == IKB_F64, n, 0, what, jac_out, manip_out, e->d_stats, e->rc,
                                    e->num_sms, (cudaStream_t)stream));
    e->launches += (n > 0);
    return IKB_OK;
}

// Chunks of the host pipeline: angles in d_in (32 B per slot row), Jacobians in d_out (as many rows as its 32 B per
// slot row hold at the Jacobian's row size, at most one per slot row), manipulabilities in d_in2 (24 B per slot row).
int ikb_jacobian_host(ikb_engine *e, const void *angles, int angles_dtype, int64_t n, int what, void *jac_out,
                      void *manip_out, ikb_stats *stats)
{
    if (const char *why = jacobian_bad_args(e, angles, angles_dtype, n, what, jac_out, manip_out))
        return fail(e, IKB_ERR_INVALID, std::string("ikb_jacobian_host: ") + why);
    int rc = host_begin(e, n);
    if (rc)
        return rc;
    const size_t in_row = 4 * esize(angles_dtype), jac_row = jacobian_row_bytes(angles_dtype, what);
    const size_t w_row = esize(angles_dtype);
    const long long m_max = jac_out ? std::min(e->slot_rows, e->slot_rows * 32 / (long long)jac_row) : e->slot_rows;
    int it = 0;
    for (long long lo = 0, m = 0; lo < n; lo += m, ++it) {
        Slot &s = e->slots[it % kSlots];
        m = std::min(m_max, n - lo);
        IKB_CUDA(e, cudaMemcpyAsync(s.d_in, (const char *)angles + lo * in_row, m * in_row, cudaMemcpyHostToDevice,
                                    s.stream));
        IKB_CUDA(e, ikb_launch_jacobian(s.d_in, angles_dtype == IKB_F64, m, lo, what, jac_out ? s.d_out : nullptr,
                                        manip_out ? s.d_in2 : nullptr, e->d_stats, e->rc, e->num_sms, s.stream));
        e->launches++;
        if (jac_out)
            IKB_CUDA(e, cudaMemcpyAsync((char *)jac_out + lo * jac_row, s.d_out, m * jac_row, cudaMemcpyDeviceToHost,
                                        s.stream));
        if (manip_out)
            IKB_CUDA(e, cudaMemcpyAsync((char *)manip_out + lo * w_row, s.d_in2, m * w_row, cudaMemcpyDeviceToHost,
                                        s.stream));
    }
    return host_end(e, stats);
}

// ---- damped-least-squares refinement --------------------------------------------------------------
// what is wrong with the arguments, or nullptr; the engine is checked last, as for the Jacobian
static const char *dls_bad_args(const ikb_engine *e, const void *xyz, int xyz_dtype, int64_t n, const void *seed,
                                int64_t n_seed, const void *angles_out, int angles_dtype, double damping, double tol,
                                int32_t max_iter, const int32_t *iters_out, const void *err_out)
{
    if (n > 0 && !xyz)
        return "NULL targets";
    if (n > 0 && !seed)
        return "NULL seeds";
    if (n > 0 && !angles_out)
        return "NULL angles_out";
    if (n < 0)
        return "negative n";
    if (n_seed != 1 && n_seed != n)
        return "n_seed must be 1 or n";
    if (bad_dtype(xyz_dtype) || bad_dtype(angles_dtype))
        return "unknown dtype";
    if (!(damping > 0.0) || !std::isfinite(damping))
        return "damping must be positive and finite";
    if (!(tol >= 0.0))
        return "tol must be >= 0 and not NaN";
    if (max_iter < 0)
        return "max_iter must be >= 0";
    const uintptr_t a_align = esize(angles_dtype) - 1;
    if (((uintptr_t)xyz & (esize(xyz_dtype) - 1)) || (((uintptr_t)seed | (uintptr_t)angles_out | (uintptr_t)err_out) & a_align) ||
        ((uintptr_t)iters_out & 3))
        return "buffers must be aligned to their element size";
    if (n > 0) {
        const uintptr_t row = 4 * esize(angles_dtype), s0 = (uintptr_t)seed, o0 = (uintptr_t)angles_out;
        const bool overlap = s0 < o0 + (uintptr_t)n * row && o0 < s0 + (uintptr_t)n_seed * row;
        if (overlap && !(s0 == o0 && n_seed == n))
            return "seed and angles_out overlap other than in place (angles_out == seed, n_seed == n)";
    }
    if (!e)
        return "NULL engine";
    return nullptr;
}

int ikb_dls_refine_device(ikb_engine *e, const void *xyz, int xyz_dtype, int64_t n, const void *seed, int64_t n_seed,
                          void *angles_out, int angles_dtype, double damping, double tol, int32_t max_iter,
                          int32_t *iters_out, void *err_out, void *stream)
{
    if (const char *why = dls_bad_args(e, xyz, xyz_dtype, n, seed, n_seed, angles_out, angles_dtype, damping, tol,
                                       max_iter, iters_out, err_out))
        return fail(e, IKB_ERR_INVALID, std::string("ikb_dls_refine_device: ") + why);
    if (n == 0)
        return IKB_OK;
    IKB_CUDA(e, cudaSetDevice(e->device));
    unsigned long long *counter;
    int slot;
    IKB_CUDA(e, counter_claim(e, (cudaStream_t)stream, &counter, &slot));
    IKB_CUDA(e, ikb_launch_dls_refine(xyz, xyz_dtype == IKB_F64, seed, n_seed, angles_out, angles_dtype == IKB_F64,
                                      iters_out, err_out, n, 0, damping, tol, max_iter, e->d_stats, counter, e->rc,
                                      e->num_sms, (cudaStream_t)stream));
    IKB_CUDA(e, counter_release(e, slot, (cudaStream_t)stream));
    e->launches++;
    return IKB_OK;
}

// Chunks of the host pipeline: targets in d_in2 (24 B per slot row), seeds in d_in, angles in d_out, iterations in
// d_aux.  The fp64 errors (8 B per row) go behind the targets in d_in2, so a chunk then holds 3 S / 4 rows (S the rows
// of a slot), else S.  A single seed (n_seed == 1) is copied to d_in of every slot once.
int ikb_dls_refine_host(ikb_engine *e, const void *xyz, int xyz_dtype, int64_t n, const void *seed, int64_t n_seed,
                        void *angles_out, int angles_dtype, double damping, double tol, int32_t max_iter,
                        int32_t *iters_out, void *err_out, ikb_stats *stats)
{
    if (const char *why = dls_bad_args(e, xyz, xyz_dtype, n, seed, n_seed, angles_out, angles_dtype, damping, tol,
                                       max_iter, iters_out, err_out))
        return fail(e, IKB_ERR_INVALID, std::string("ikb_dls_refine_host: ") + why);
    int rc = host_begin(e, n);
    if (rc)
        return rc;
    const size_t t_row = 3 * esize(xyz_dtype), a_row = 4 * esize(angles_dtype), e_row = esize(angles_dtype);
    const long long m_max = err_out ? 3 * e->slot_rows / 4 : e->slot_rows;
    const bool per_row_seed = n_seed != 1;
    if (n > 0 && !per_row_seed)
        for (int i = 0; i < kSlots; ++i)
            IKB_CUDA(e, cudaMemcpyAsync(e->slots[i].d_in, seed, a_row, cudaMemcpyHostToDevice, e->slots[i].stream));
    int it = 0;
    for (long long lo = 0, m = 0; lo < n; lo += m, ++it) {
        Slot &s = e->slots[it % kSlots];
        m = std::min(m_max, n - lo);
        void *d_err = err_out ? (void *)((char *)s.d_in2 + 24 * m_max) : nullptr;
        IKB_CUDA(e, cudaMemcpyAsync(s.d_in2, (const char *)xyz + lo * t_row, m * t_row, cudaMemcpyHostToDevice, s.stream));
        if (per_row_seed)
            IKB_CUDA(e, cudaMemcpyAsync(s.d_in, (const char *)seed + lo * a_row, m * a_row, cudaMemcpyHostToDevice,
                                        s.stream));
        unsigned long long *counter;
        int slot;
        IKB_CUDA(e, counter_claim(e, s.stream, &counter, &slot));
        IKB_CUDA(e, ikb_launch_dls_refine(s.d_in2, xyz_dtype == IKB_F64, s.d_in, per_row_seed ? m : 1, s.d_out,
                                          angles_dtype == IKB_F64, iters_out ? s.d_aux : nullptr, d_err, m, lo,
                                          damping, tol, max_iter, e->d_stats, counter, e->rc, e->num_sms, s.stream));
        IKB_CUDA(e, counter_release(e, slot, s.stream));
        e->launches++;
        IKB_CUDA(e, cudaMemcpyAsync((char *)angles_out + lo * a_row, s.d_out, m * a_row, cudaMemcpyDeviceToHost, s.stream));
        if (iters_out)
            IKB_CUDA(e, cudaMemcpyAsync(iters_out + lo, s.d_aux, m * sizeof(int), cudaMemcpyDeviceToHost, s.stream));
        if (err_out)
            IKB_CUDA(e, cudaMemcpyAsync((char *)err_out + lo * e_row, d_err, m * e_row, cudaMemcpyDeviceToHost, s.stream));
    }
    return host_end(e, stats);
}

// ---- damped-least-squares refinement onto poses ---------------------------------------------------------------------
// the weights first, then everything dls_bad_args checks (the engine last)
static const char *pose_bad_args(const ikb_engine *e, const void *poses, int pose_dtype, int64_t n, const void *seed,
                                 int64_t n_seed, const void *angles_out, int angles_dtype, const double *weights,
                                 double damping, double tol, int32_t max_iter, const int32_t *iters_out,
                                 const void *err_out)
{
    if (!weights)
        return "NULL weights";
    bool any = false;
    for (int i = 0; i < 6; ++i) {
        if (!(weights[i] >= 0.0) || !std::isfinite(weights[i]))
            return "weights must be >= 0 and finite";
        any = any || weights[i] > 0.0;
    }
    if (!any)
        return "all six weights are zero";
    return dls_bad_args(e, poses, pose_dtype, n, seed, n_seed, angles_out, angles_dtype, damping, tol, max_iter,
                        iters_out, err_out);
}

int ikb_dls_pose_refine_device(ikb_engine *e, const void *poses, int pose_dtype, int64_t n, const void *seed,
                               int64_t n_seed, void *angles_out, int angles_dtype, const double weights[6],
                               double damping, double tol, int32_t max_iter, int32_t *iters_out, void *err_out,
                               void *stream)
{
    if (const char *why = pose_bad_args(e, poses, pose_dtype, n, seed, n_seed, angles_out, angles_dtype, weights,
                                        damping, tol, max_iter, iters_out, err_out))
        return fail(e, IKB_ERR_INVALID, std::string("ikb_dls_pose_refine_device: ") + why);
    if (n == 0)
        return IKB_OK;
    IKB_CUDA(e, cudaSetDevice(e->device));
    unsigned long long *counter;
    int slot;
    IKB_CUDA(e, counter_claim(e, (cudaStream_t)stream, &counter, &slot));
    IKB_CUDA(e, ikb_launch_dls_pose_refine(poses, pose_dtype == IKB_F64, seed, n_seed, angles_out,
                                           angles_dtype == IKB_F64, iters_out, err_out, n, 0, weights, damping, tol,
                                           max_iter, e->d_stats, counter, e->rc, e->num_sms, (cudaStream_t)stream));
    IKB_CUDA(e, counter_release(e, slot, (cudaStream_t)stream));
    e->launches++;
    return IKB_OK;
}

// Chunks of the host pipeline, S / 4 rows each (S the rows of a slot): poses in d_in (32 B per slot row, so 128 B per
// chunk row), seeds in d_in2 (24 B per slot row) with the fp64 errors behind them, angles in d_out, iterations in
// d_aux.  A single seed (n_seed == 1) is copied to d_in2 of every slot once.
int ikb_dls_pose_refine_host(ikb_engine *e, const void *poses, int pose_dtype, int64_t n, const void *seed,
                             int64_t n_seed, void *angles_out, int angles_dtype, const double weights[6],
                             double damping, double tol, int32_t max_iter, int32_t *iters_out, void *err_out,
                             ikb_stats *stats)
{
    if (const char *why = pose_bad_args(e, poses, pose_dtype, n, seed, n_seed, angles_out, angles_dtype, weights,
                                        damping, tol, max_iter, iters_out, err_out))
        return fail(e, IKB_ERR_INVALID, std::string("ikb_dls_pose_refine_host: ") + why);
    int rc = host_begin(e, n);
    if (rc)
        return rc;
    const size_t p_row = 16 * esize(pose_dtype), a_row = 4 * esize(angles_dtype), e_row = esize(angles_dtype);
    const long long m_max = e->slot_rows / 4;
    const bool per_row_seed = n_seed != 1;
    if (n > 0 && !per_row_seed)
        for (int i = 0; i < kSlots; ++i)
            IKB_CUDA(e, cudaMemcpyAsync(e->slots[i].d_in2, seed, a_row, cudaMemcpyHostToDevice, e->slots[i].stream));
    int it = 0;
    for (long long lo = 0, m = 0; lo < n; lo += m, ++it) {
        Slot &s = e->slots[it % kSlots];
        m = std::min(m_max, n - lo);
        void *d_err = err_out ? (void *)((char *)s.d_in2 + 32 * m_max) : nullptr;
        IKB_CUDA(e, cudaMemcpyAsync(s.d_in, (const char *)poses + lo * p_row, m * p_row, cudaMemcpyHostToDevice,
                                    s.stream));
        if (per_row_seed)
            IKB_CUDA(e, cudaMemcpyAsync(s.d_in2, (const char *)seed + lo * a_row, m * a_row, cudaMemcpyHostToDevice,
                                        s.stream));
        unsigned long long *counter;
        int slot;
        IKB_CUDA(e, counter_claim(e, s.stream, &counter, &slot));
        IKB_CUDA(e, ikb_launch_dls_pose_refine(s.d_in, pose_dtype == IKB_F64, s.d_in2, per_row_seed ? m : 1, s.d_out,
                                               angles_dtype == IKB_F64, iters_out ? s.d_aux : nullptr, d_err, m, lo,
                                               weights, damping, tol, max_iter, e->d_stats, counter, e->rc,
                                               e->num_sms, s.stream));
        IKB_CUDA(e, counter_release(e, slot, s.stream));
        e->launches++;
        IKB_CUDA(e, cudaMemcpyAsync((char *)angles_out + lo * a_row, s.d_out, m * a_row, cudaMemcpyDeviceToHost, s.stream));
        if (iters_out)
            IKB_CUDA(e, cudaMemcpyAsync(iters_out + lo, s.d_aux, m * sizeof(int), cudaMemcpyDeviceToHost, s.stream));
        if (err_out)
            IKB_CUDA(e, cudaMemcpyAsync((char *)err_out + lo * e_row, d_err, m * e_row, cudaMemcpyDeviceToHost, s.stream));
    }
    return host_end(e, stats);
}

// ---- closed-form inverse kinematics ---------------------------------------------------------------------------------
// what is wrong with the arguments, or nullptr; the engine is checked last, the DH family after it
static const char *analytic_bad_args(const ikb_engine *e, int kind, const void *in, int in_dtype, int64_t n,
                                     const void *pitch, int64_t n_pitch, const void *angles_out, int angles_dtype,
                                     const int32_t *status_out)
{
    if (n > 0 && !in)
        return "NULL input";
    if (n > 0 && !angles_out)
        return "NULL angles_out";
    if (kind != IKB_AIK_POSE && kind != IKB_AIK_POSITION_PITCH)
        return "unknown kind";
    if (bad_dtype(in_dtype) || bad_dtype(angles_dtype))
        return "unknown dtype";
    if (n < 0)
        return "negative n";
    if (kind == IKB_AIK_POSITION_PITCH && n > 0 && !pitch)
        return "NULL pitch: the position kind needs one pitch or one per row";
    if (kind == IKB_AIK_POSE && pitch)
        return "pitch given for the pose kind, which takes none";
    if (kind == IKB_AIK_POSITION_PITCH && n_pitch != 1 && n_pitch != n)
        return "n_pitch must be 1 or n";
    const uintptr_t i_align = esize(in_dtype) - 1;
    if ((((uintptr_t)in | (uintptr_t)pitch) & i_align) || ((uintptr_t)angles_out & (esize(angles_dtype) - 1)) ||
        ((uintptr_t)status_out & 3))
        return "buffers must be aligned to their element size";
    if (!e)
        return "NULL engine";
    return nullptr;
}

static int analytic_refusal(ikb_engine *e, const char *name, int kind, const void *in, int in_dtype, int64_t n,
                            const void *pitch, int64_t n_pitch, const void *angles_out, int angles_dtype,
                            const int32_t *status_out)
{
    if (const char *why = analytic_bad_args(e, kind, in, in_dtype, n, pitch, n_pitch, angles_out, angles_dtype,
                                            status_out))
        return fail(e, IKB_ERR_INVALID, std::string(name) + ": " + why);
    if (!e->analytic_family)
        return fail(e, IKB_ERR_UNSUPPORTED,
                    std::string(name) + ": the DH table is outside the closed form's family (alpha_2 = alpha_3 = "
                    "alpha_4 = 0, |cos alpha_1| <= 1e-12, a_2 > 0, a_3 > 0); use ikine_pose / refine_pose for it");
    return IKB_OK;
}

int ikb_analytic_ik_device(ikb_engine *e, int kind, const void *in, int in_dtype, int64_t n, const void *pitch,
                           int64_t n_pitch, void *angles_out, int angles_dtype, int32_t *status_out, void *stream)
{
    if (int rc = analytic_refusal(e, "ikb_analytic_ik_device", kind, in, in_dtype, n, pitch, n_pitch, angles_out,
                                  angles_dtype, status_out))
        return rc;
    if (n == 0)
        return IKB_OK;
    IKB_CUDA(e, cudaSetDevice(e->device));
    IKB_CUDA(e, ikb_launch_analytic_ik(kind, in, in_dtype == IKB_F64, n, 0, pitch, n_pitch != 1, angles_out,
                                       angles_dtype == IKB_F64, status_out, e->d_stats, e->rc, e->num_sms,
                                       (cudaStream_t)stream));
    e->launches++;
    return IKB_OK;
}

// Chunks of the host pipeline, S / 4 rows each (S the rows of a slot): poses (128 B per fp64 row) or positions in
// d_in, per-row pitches in d_in2 (a single pitch is copied to d_in2 of every slot once), angles (up to 128 B per fp64
// row) in d_out, status in d_aux.
int ikb_analytic_ik_host(ikb_engine *e, int kind, const void *in, int in_dtype, int64_t n, const void *pitch,
                         int64_t n_pitch, void *angles_out, int angles_dtype, int32_t *status_out, ikb_stats *stats)
{
    if (int rc = analytic_refusal(e, "ikb_analytic_ik_host", kind, in, in_dtype, n, pitch, n_pitch, angles_out,
                                  angles_dtype, status_out))
        return rc;
    int rc = host_begin(e, n);
    if (rc)
        return rc;
    const bool pose = kind == IKB_AIK_POSE, per_row_pitch = !pose && n_pitch != 1;
    const size_t i_row = (pose ? 16 : 3) * esize(in_dtype), p_row = esize(in_dtype);
    const size_t a_row = (pose ? 2 : 4) * 4 * esize(angles_dtype);
    const long long m_max = e->slot_rows / 4;
    if (n > 0 && !pose && !per_row_pitch)
        for (int i = 0; i < kSlots; ++i)
            IKB_CUDA(e, cudaMemcpyAsync(e->slots[i].d_in2, pitch, p_row, cudaMemcpyHostToDevice, e->slots[i].stream));
    int it = 0;
    for (long long lo = 0, m = 0; lo < n; lo += m, ++it) {
        Slot &s = e->slots[it % kSlots];
        m = std::min(m_max, n - lo);
        IKB_CUDA(e, cudaMemcpyAsync(s.d_in, (const char *)in + lo * i_row, m * i_row, cudaMemcpyHostToDevice, s.stream));
        if (per_row_pitch)
            IKB_CUDA(e, cudaMemcpyAsync(s.d_in2, (const char *)pitch + lo * p_row, m * p_row, cudaMemcpyHostToDevice,
                                        s.stream));
        IKB_CUDA(e, ikb_launch_analytic_ik(kind, s.d_in, in_dtype == IKB_F64, m, lo, pose ? nullptr : s.d_in2,
                                           per_row_pitch, s.d_out, angles_dtype == IKB_F64,
                                           status_out ? s.d_aux : nullptr, e->d_stats, e->rc, e->num_sms, s.stream));
        e->launches++;
        IKB_CUDA(e, cudaMemcpyAsync((char *)angles_out + lo * a_row, s.d_out, m * a_row, cudaMemcpyDeviceToHost,
                                    s.stream));
        if (status_out)
            IKB_CUDA(e, cudaMemcpyAsync(status_out + lo, s.d_aux, m * sizeof(int32_t), cudaMemcpyDeviceToHost,
                                        s.stream));
    }
    return host_end(e, stats);
}

int ikb_fk_chain_host(ikb_engine *e, const double angles[4], double chain_out[64], int *status)
{
    if (!e || !angles || !chain_out || !status)
        return fail(e, IKB_ERR_INVALID, "ikb_fk_chain_host: NULL argument");
    ikb_stats st;
    int rc = ikb_fk_transforms_host(e, angles, IKB_F64, 1, IKB_FK_MATRICES, chain_out, &st);
    if (rc)
        return rc;
    *status = st.first_fk_angle_range >= 0 ? 1 : 0;
    return IKB_OK;
}

// ---- ANN ------------------------------------------------------------------------------------------
int ikb_mlp_load(ikb_engine *e, int32_t n_layers, const int32_t *dims, const float *const *weights,
                 const float *const *biases, const double mean_x[3], const double scale_x[3],
                 const double mean_y[4], const double scale_y[4])
{
    if (!e || n_layers < 1 || !dims || !weights || !biases || !mean_x || !scale_x || !mean_y || !scale_y)
        return fail(e, IKB_ERR_INVALID, "ikb_mlp_load: NULL argument");
    IKB_CUDA(e, cudaSetDevice(e->device));
    std::string msg;
    int rc = ikb_mlp_upload(e->mlp, n_layers, dims, weights, biases, mean_x, scale_x, mean_y, scale_y, msg);
    if (rc)
        return fail(e, rc, msg);
    return IKB_OK;
}

int ikb_ann_solve_device(ikb_engine *e, const void *xyz, int xyz_dtype, int64_t n, float *angles_out,
                         float *fk_err_out, int fk_stats, int mode, void *stream)
{
    if (!e || n < 0 || (n > 0 && (!xyz || !angles_out)) || bad_dtype(xyz_dtype))
        return fail(e, IKB_ERR_INVALID, "ikb_ann_solve_device: bad argument");
    if (((uintptr_t)angles_out & 15))  // rows are stored as float4
        return fail(e, IKB_ERR_INVALID, "ikb_ann_solve_device: angles must be 16-byte aligned");
    if (!e->mlp.loaded)
        return fail(e, IKB_ERR_NO_MODEL, "ikb_ann_solve: no model loaded (call ikb_mlp_load first)");
    IKB_CUDA(e, cudaSetDevice(e->device));
    std::string msg;
    int launches = 0;
    int rc = ikb_mlp_launch(e->mlp, xyz, xyz_dtype == IKB_F64, n, 0, angles_out, fk_err_out, fk_stats, mode,
                            e->d_stats, e->rc, e->num_sms, (cudaStream_t)stream, msg, launches);
    e->launches += launches;
    if (rc)
        return fail(e, rc, msg);
    return IKB_OK;
}

int ikb_ann_solve_host(ikb_engine *e, const void *xyz, int xyz_dtype, int64_t n, float *angles_out,
                       float *fk_err_out, int fk_stats, int mode, ikb_stats *stats)
{
    if (!e || n < 0 || (n > 0 && (!xyz || !angles_out)) || bad_dtype(xyz_dtype))
        return fail(e, IKB_ERR_INVALID, "ikb_ann_solve_host: bad argument");
    if (!e->mlp.loaded)
        return fail(e, IKB_ERR_NO_MODEL, "ikb_ann_solve: no model loaded (call ikb_mlp_load first)");
    int rc = host_begin(e, n);
    if (rc)
        return rc;
    const size_t in_row = 3 * esize(xyz_dtype), out_row = 4 * sizeof(float);
    int it = 0;
    for (long long lo = 0, m = 0; lo < n; lo += m, ++it) {
        Slot &s = e->slots[it % kSlots];
        m = host_chunk_rows(lo, n);
        float *d_err = fk_err_out ? (float *)s.d_in2 : nullptr;
        IKB_CUDA(e, cudaMemcpyAsync(s.d_in, (const char *)xyz + lo * in_row, m * in_row, cudaMemcpyHostToDevice, s.stream));
        std::string msg;
        int launches = 0;
        rc = ikb_mlp_launch(e->mlp, s.d_in, xyz_dtype == IKB_F64, m, lo, (float *)s.d_out, d_err, fk_stats, mode,
                            e->d_stats, e->rc, e->num_sms, s.stream, msg, launches);
        e->launches += launches;
        if (rc)
            return fail(e, rc, msg);
        IKB_CUDA(e, cudaMemcpyAsync((char *)angles_out + lo * out_row, s.d_out, m * out_row, cudaMemcpyDeviceToHost, s.stream));
        if (fk_err_out)
            IKB_CUDA(e, cudaMemcpyAsync(fk_err_out + lo, d_err, m * sizeof(float), cudaMemcpyDeviceToHost, s.stream));
    }
    return host_end(e, stats);
}

// ---- trajectory generators ------------------------------------------------------------------------
int ikb_generate_device(ikb_engine *e, int kind, const double *params, int n_params, int64_t n, int64_t row_offset,
                        void *xyz_out, int xyz_dtype, uint64_t seed, void *stream)
{
    if (!e || n < 0 || (n > 0 && !xyz_out) || bad_dtype(xyz_dtype) || kind < 0 || kind > 4 || n_params < 0 ||
        n_params > 12 || (n_params > 0 && !params))
        return fail(e, IKB_ERR_INVALID, "ikb_generate_device: bad argument");
    IKB_CUDA(e, cudaSetDevice(e->device));
    IKB_CUDA(e, ikb_launch_generate(kind, params, n_params, n, row_offset, xyz_out, xyz_dtype == IKB_F64, seed,
                                    e->num_sms, (cudaStream_t)stream));
    e->launches += (n > 0);
    return IKB_OK;
}

// ---- pinned host buffers --------------------------------------------------------------------------
int ikb_host_alloc(ikb_engine *e, size_t bytes, void **out)
{
    if (!e || !out || bytes == 0)
        return fail(e, IKB_ERR_INVALID, "ikb_host_alloc: bad argument");
    *out = nullptr;
    IKB_CUDA(e, cudaSetDevice(e->device));
    IKB_CUDA(e, cudaHostAlloc(out, bytes, cudaHostAllocDefault));
    return IKB_OK;
}

int ikb_host_free(ikb_engine *e, void *p)
{
    if (!e)
        return IKB_ERR_INVALID;
    if (!p)
        return IKB_OK;
    IKB_CUDA(e, cudaSetDevice(e->device));
    IKB_CUDA(e, cudaFreeHost(p));
    return IKB_OK;
}

int ikb_host_register(ikb_engine *e, void *p, size_t bytes, int read_only)
{
    if (!e || !p || bytes == 0)
        return fail(e, IKB_ERR_INVALID, "ikb_host_register: bad argument");
    IKB_CUDA(e, cudaSetDevice(e->device));
    cudaError_t err = cudaHostRegister(p, bytes, read_only ? cudaHostRegisterReadOnly : cudaHostRegisterDefault);
    if (err != cudaSuccess && read_only) {  // read-only registration is optional on some platforms
        (void)cudaGetLastError();
        err = cudaHostRegister(p, bytes, cudaHostRegisterDefault);
    }
    IKB_CUDA(e, err);
    return IKB_OK;
}

int ikb_host_unregister(ikb_engine *e, void *p)
{
    if (!e || !p)
        return fail(e, IKB_ERR_INVALID, "ikb_host_unregister: bad argument");
    IKB_CUDA(e, cudaSetDevice(e->device));
    IKB_CUDA(e, cudaHostUnregister(p));
    return IKB_OK;
}

// ---- measurement ----------------------------------------------------------------------------------
int ikb_copy_pipeline_host(ikb_engine *e, const void *in, int64_t in_row_bytes, int64_t n, void *out,
                           int64_t out_row_bytes)
{
    if (!e || n < 0 || in_row_bytes < 0 || out_row_bytes < 0 || in_row_bytes > 32 || out_row_bytes > 32 ||
        (n > 0 && ((in_row_bytes && !in) || (out_row_bytes && !out))))
        return fail(e, IKB_ERR_INVALID, "ikb_copy_pipeline_host: bad argument (rows of at most 32 bytes)");
    int rc = host_begin(e, n);
    if (rc)
        return rc;
    int it = 0;
    for (long long lo = 0, m = 0; lo < n; lo += m, ++it) {
        Slot &s = e->slots[it % kSlots];
        m = host_chunk_rows(lo, n);
        if (in_row_bytes)
            IKB_CUDA(e, cudaMemcpyAsync(s.d_in, (const char *)in + lo * in_row_bytes, m * in_row_bytes,
                                        cudaMemcpyHostToDevice, s.stream));
        if (out_row_bytes)
            IKB_CUDA(e, cudaMemcpyAsync((char *)out + lo * out_row_bytes, s.d_out, m * out_row_bytes,
                                        cudaMemcpyDeviceToHost, s.stream));
    }
    return host_end(e, nullptr);
}

int ikb_theoretical_fma_peak(ikb_engine *e, int dtype, double *tflops_out)
{
    if (!e || !tflops_out || bad_dtype(dtype))
        return fail(e, IKB_ERR_INVALID, "ikb_theoretical_fma_peak: bad argument");
    int khz = 0;
    IKB_CUDA(e, cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, e->device));
    const double lanes = dtype == IKB_F64 ? 64.0 : 128.0;  // sm_100: 128 fp32 / 64 fp64 FMA lanes per SM
    *tflops_out = e->num_sms * lanes * 2.0 * (double)khz * 1e3 / 1e12;
    return IKB_OK;
}

int ikb_microbench_fma(ikb_engine *e, int dtype, double *tflops_out)
{
    if (!e || !tflops_out || bad_dtype(dtype))
        return fail(e, IKB_ERR_INVALID, "ikb_microbench_fma: bad argument");
    IKB_CUDA(e, cudaSetDevice(e->device));
    void *sink = nullptr;
    IKB_CUDA(e, cudaMalloc(&sink, 64));
    cudaEvent_t t0, t1;
    IKB_CUDA(e, cudaEventCreate(&t0));
    IKB_CUDA(e, cudaEventCreate(&t1));
    const int iters = dtype == IKB_F64 ? 4096 : 8192;
    double best = 0.0;
    for (int rep = 0; rep < 6; ++rep) {
        IKB_CUDA(e, cudaEventRecord(t0, nullptr));
        IKB_CUDA(e, ikb_launch_fma_peak(dtype == IKB_F64, sink, iters, e->num_sms, nullptr));
        e->launches++;
        IKB_CUDA(e, cudaEventRecord(t1, nullptr));
        IKB_CUDA(e, cudaEventSynchronize(t1));
        float ms = 0;
        IKB_CUDA(e, cudaEventElapsedTime(&ms, t0, t1));
        const double flops = 2.0 * 32.0 * iters * 256.0 * e->num_sms * 8.0;
        const double tf = flops / (ms * 1e-3) / 1e12;
        if (rep > 0 && tf > best)
            best = tf;
    }
    cudaEventDestroy(t0); cudaEventDestroy(t1); cudaFree(sink);
    *tflops_out = best;
    return IKB_OK;
}

}  // extern "C"

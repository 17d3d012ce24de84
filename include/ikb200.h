/*
 * ikb200.h -- C ABI of the B200-native batched inverse-kinematics engine (libikb200.so).
 *
 * This is the drop-in boundary for the reference's hot path (lstar93/InverseKinematicsANN):
 * plain pointers and sizes, no torch / C++ types.  The Python host mirror of the reference's
 * `kinematics/` API (inversekinematicsann_b200/kinematics/*.py) binds these with ctypes;
 * INTEGRATION.md shows the stub a maintainer of the reference would add.
 *
 * Every entry point cites the reference interface (file:line under the reference root) it replaces.
 *
 * Conventions
 *   - All calls return IKB_OK (0) or a negative IKB_ERR_* code; ikb_last_error() gives the text.
 *   - "dtype" arguments are IKB_F32 / IKB_F64 and describe the element type of a caller buffer.
 *   - Targets are AoS rows [x, y, z]; angles are AoS rows [theta1..theta4]; row i of every output
 *     belongs to row i of the input (trajectory order is preserved).
 *   - *_device entry points take DEVICE pointers, enqueue on `stream` (a cudaStream_t passed as
 *     void*, NULL = the legacy default stream) and return without synchronising; per-call
 *     diagnostics accumulate in the engine's device-side statistics block, read with
 *     ikb_stats_fetch().
 *   - *_host entry points take HOST pointers (pinned or pageable), run a chunked
 *     H2D -> kernel -> D2H pipeline on the engine's own streams, synchronise, and fill `stats`.
 *   - The reference's whole-batch exception semantics (inverse.py:117: check_limits raises before
 *     any solve) map to stats.first_out_of_limits >= 0: the caller must then discard the outputs
 *     and raise OutOfRobotReachException for that row.
 *   - Row counts: every kernel indexes rows with 64-bit integers except K1 (FABRIK), whose shared-memory queues
 *     hold 32-bit row numbers: ikb_fabrik_solve_device refuses n >= 2^31 per call (the *_host entry points chunk
 *     internally and have no limit).
 *   - There is no CPU fallback: without a CUDA device every compute entry point fails with
 *     IKB_ERR_CUDA.
 */
#ifndef IKB200_H
#define IKB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define IKB_OK 0
#define IKB_ERR_INVALID (-1)   /* bad argument (NULL pointer, negative size, unknown enum)      */
#define IKB_ERR_CUDA (-2)      /* CUDA runtime error (no device, launch failure, OOM ...)       */
#define IKB_ERR_NO_MODEL (-3)  /* ikb_ann_* called before ikb_mlp_load                          */
#define IKB_ERR_UNSUPPORTED (-4) /* e.g. a DH table that is not 4 joints                        */

#define IKB_F32 0
#define IKB_F64 1

/* FABRIK iterate precision.  The angle extraction (reference inverse.py:54-112) forms its cosines and their 8-decimal
 * rounding in fp64 either way; what follows the rounding (acos / atan2 and the combination with pi) is evaluated in the
 * precision of the caller's angle buffer: IKB_F64 buffers <= 1e-9 rad from the reference, IKB_F32 buffers <= 1e-6 rad. */
#define IKB_FABRIK_F64 0 /* default: fp64 iterate, agrees with the reference to ~1e-12 rad       */
#define IKB_FABRIK_F32 1 /* fast: fp32 iterate; ~0.4 % of uniform-workspace targets leave the    */
                         /* 1e-4 rad band (convergence-test flips), see DESIGN.md                */

/* MLP arithmetic mode */
#define IKB_MLP_FP32_SIMT 0 /* fp32 FFMA on the CUDA cores (Keras-fp32 grade)                    */
#define IKB_MLP_FP16X3_TC 1 /* tcgen05 kind::f16, 3-term hi/lo split, fp32 accumulate in TMEM    */
#define IKB_MLP_FP16X3_TS 2 /* same arithmetic, activations as the A operand in TMEM (TS-mode MMA) */

typedef struct ikb_engine ikb_engine;

/* Robot + solver description: the constructor arguments of the reference's IK classes
 * (inverse.py:20-24,47-52) and robot/robot.py:40-42. */
typedef struct ikb_config {
    double dh[16];     /* reference DH table, row-major 4x4: rows = thetas, epsilons, a, alphas
                          (forward.py:16); row 0 holds the seed angles [.., pi/2, 0, 0]          */
    double links[4];   /* joints_distances (robot.py:42)                                        */
    double limits[6];  /* workspace box {xlo, xhi, ylo, yhi, zlo, zhi}, inclusive (robot.py:41)  */
    double tol;        /* FABRIK err_margin (fabrik.py:13, inverse.py:48), default 1e-3          */
    int32_t max_iter;  /* FABRIK max_iter_num, default 100                                      */
    int32_t device;    /* CUDA device ordinal this engine lives on                              */
} ikb_config;

/* Per-call diagnostics (what the reference signals with exceptions) and roofline accounting.   */
typedef struct ikb_stats {
    int64_t n_solved;            /* targets processed                                           */
    int64_t sum_iterations;      /* sum of FABRIK iterations (k in "114 k + 126 flops")          */
    int64_t n_iter_capped;       /* targets that stopped on max_iter, not on the tolerance       */
    int64_t first_out_of_limits; /* lowest row failing check_limits (inverse.py:26-35) or -1     */
    int64_t first_zero_division; /* lowest row where a segment length was 0 (point.py:40 raises
                                    ZeroDivisionError in the reference) or -1; its angles are NaN */
    int64_t first_domain_error;  /* lowest row with acos argument outside [-1,1] after the 8-dp
                                    rounding (ValueError in the reference) or -1                 */
    int64_t first_fk_angle_range;/* lowest row with an angle outside [-2pi, 2pi] in an FK call
                                    (forward.py:23-25 raises OutOfRobotReachException) or -1     */
    double sum_fk_error;         /* sum of ||FK(angles) - target|| over rows with a finite error */
    int64_t n_fk_error;          /* number of rows in sum_fk_error                               */
} ikb_stats;

/* ---- engine lifetime ------------------------------------------------------------------------ */
/* replaces InverseKinematics.__init__ / FabrikInverseKinematics.__init__ (inverse.py:20-24,47-52) */
int ikb_engine_create(const ikb_config *cfg, ikb_engine **out);
void ikb_engine_destroy(ikb_engine *e);
/* text of the last error on this engine (or of the last failed ikb_engine_create when e == NULL) */
const char *ikb_last_error(const ikb_engine *e);
/* library version + build arch string, e.g. "ikb200 0.1 sm_100a" */
const char *ikb_version(void);
int ikb_device_count(void);

/* ---- statistics ----------------------------------------------------------------------------- */
int ikb_stats_reset(ikb_engine *e, void *stream);
/* synchronises `stream`, copies the device statistics block to *out */
int ikb_stats_fetch(ikb_engine *e, void *stream, ikb_stats *out);

/* ---- check_limits (inverse.py:26-35) --------------------------------------------------------- */
/* first_bad = lowest row with any axis outside its inclusive bounds (NaN passes), else -1        */
int ikb_check_limits_device(ikb_engine *e, const void *xyz, int xyz_dtype, int64_t n, void *stream);
int ikb_check_limits_host(ikb_engine *e, const void *xyz, int xyz_dtype, int64_t n,
                          int64_t *first_bad);

/* ---- FABRIK ikine (inverse.py:115-139 = check_limits + per-target Fabrik.calculate
 *      (fabrik.py:44-67) + __get_angles (inverse.py:54-112)) ----------------------------------- */
/* fk_err_out (nullable, n values of angles_dtype) = ||FK(angles_out) - target|| per row, the check the reference
 * CLI draws (cli.py:56-61) -- part of the same call: fused into the solver's epilogue for batches up to 2^10 rows
 * (one launch), an fk_kernel launch on the same stream above that (measured cheaper there) and for DH tables
 * without the closed-form FK; fk_stats != 0 accumulates ikb_stats.sum_fk_error / n_fk_error even without the
 * per-row array. */
int ikb_fabrik_solve_device(ikb_engine *e, const void *xyz, int xyz_dtype, int64_t n,
                            void *angles_out, int angles_dtype,
                            int32_t *iters_out /* nullable */, void *fk_err_out /* nullable */, int fk_stats,
                            int precision, void *stream);
int ikb_fabrik_solve_host(ikb_engine *e, const void *xyz, int xyz_dtype, int64_t n,
                          void *angles_out, int angles_dtype,
                          int32_t *iters_out /* nullable */, void *fk_err_out /* nullable */, int fk_stats,
                          int precision, ikb_stats *stats);

/* ---- Fabrik.calculate with explicit initial chains (fabrik.py:44-67) -------------------------
 * A chain of n_points = J points (1 <= J <= IKB_CHAIN_MAX_POINTS, else IKB_ERR_UNSUPPORTED) with one link length per
 * point (links: J doubles in HOST memory; the backward pass uses links[J-2..0], the forward pass links[1..J-1]).
 * init: n_init x J x 3 doubles (n_init == 1 broadcasts one chain to all goals, or n_init == n);
 * goals: n x 3 doubles; chain_out: n x J x 3 doubles; iters_out: n passes per row.  3-D, IEEE fp64 with the
 * reference's operation order (sqrt and division correctly rounded, no FMA contraction): the result of a row does not
 * depend on the batch it is in.  tol and max_iter are the reference's err_margin and max_iter_num: tol >= 1 or
 * max_iter <= 0 returns the initial chains.  A zero-length segment leaves a non-finite chain and sets
 * stats.first_zero_division (ZeroDivisionError upstream).  Row counts are 64-bit, without a per-call limit.
 * _device: DEVICE pointers, enqueued on `stream`; _host: HOST pointers, staged through the engine's pipeline. */
#define IKB_CHAIN_MAX_POINTS 256
int ikb_fabrik_chain_device(ikb_engine *e, int32_t n_points, const double *links, double tol, int32_t max_iter,
                            const double *init, int64_t n_init, const double *goals, int64_t n, double *chain_out,
                            int32_t *iters_out /* nullable */, void *stream);
int ikb_fabrik_chain_host(ikb_engine *e, int32_t n_points, const double *links, double tol, int32_t max_iter,
                          const double *init, int64_t n_init, const double *goals, int64_t n, double *chain_out,
                          int32_t *iters_out /* nullable */, ikb_stats *stats);
/* the 4-point chain with the engine's own links, tol and max_iter (ikb_config) */
int ikb_fabrik_calculate_host(ikb_engine *e, const double *init, int64_t n_init,
                              const double *goals, int64_t n, double *chain_out,
                              int32_t *iters_out /* nullable */, ikb_stats *stats);

/* ---- forward kinematics (forward.py:73-94) ---------------------------------------------------
 * (fp32 buffers + err_out only + an arm whose joints 2..4 have alpha = 0 take the HBM-speed kernels of csrc/fk.cu;
 *  everything else the generic one -- same arithmetic, errors agree to 2e-6)
 * angles n x 4 -> end-effector position n x 3 (column 3 of the last cumulative DH matrix, as read
 * at cli.py:60 / inverse.py:130) and/or position error ||pos - target||.  pos_out, targets and
 * err_out are nullable (err_out needs targets); pos/err use angles_dtype, targets use xyz_dtype. */
int ikb_fk_device(ikb_engine *e, const void *angles, int angles_dtype, int64_t n,
                  void *pos_out, const void *targets, int xyz_dtype, void *err_out, void *stream);
int ikb_fk_host(ikb_engine *e, const void *angles, int angles_dtype, int64_t n,
                void *pos_out, const void *targets, int xyz_dtype, void *err_out, ikb_stats *stats);
/* all four cumulative 4x4 matrices of ONE angle set (the (T, [T1..T4]) return of fkine):
 * chain_out = 4 x 16 doubles, row-major.  Host pointers. */
int ikb_fk_chain_host(ikb_engine *e, const double angles[4], double chain_out[64], int *status);

/* ---- ANN (ann.py:70-85, inverse.py:142-155) -------------------------------------------------- */
/* replaces ANN.load_model (ann.py:78-85): upload the Keras Sequential's Dense kernels/biases and the
 * two StandardScalers.  dims[n_layers+1] = {3, 500, ..., 500, 4}; weights[l] is row-major
 * (dims[l] x dims[l+1]) float32 = Keras `kernel`, biases[l] has dims[l+1] floats.  Hidden layers
 * use tanh, the last layer is linear (ann.py:46-56).  HOST pointers; the scalers are folded into the
 * first / last layer on upload. */
int ikb_mlp_load(ikb_engine *e, int32_t n_layers, const int32_t *dims,
                 const float *const *weights, const float *const *biases,
                 const double mean_x[3], const double scale_x[3],
                 const double mean_y[4], const double scale_y[4]);
/* replaces AnnInverseKinematics.ikine / ANN.predict (inverse.py:152-155, ann.py:70-76):
 * angles_out is n x 4 float32 (Keras / sklearn return float32). */
/* fk_err_out / fk_stats as for ikb_fabrik_solve_*: fused into the default IKB_MLP_FP16X3_TS kernel's output stage,
 * a second launch (fk_kernel) on the same stream for the two cross-check modes. */
int ikb_ann_solve_device(ikb_engine *e, const void *xyz, int xyz_dtype, int64_t n,
                         float *angles_out, float *fk_err_out /* nullable */, int fk_stats, int mode, void *stream);
int ikb_ann_solve_host(ikb_engine *e, const void *xyz, int xyz_dtype, int64_t n,
                       float *angles_out, float *fk_err_out /* nullable */, int fk_stats, int mode, ikb_stats *stats);

/* ---- trajectory generators (robot/position_generator.py:26-97), written straight into device memory ----
 * kind / params (doubles):
 *   IKB_GEN_CIRCLE      {radius, cx, cy, cz}                      circle(radius, n, centre)            :26-31
 *   IKB_GEN_SPRING      {len_x, len_y, len_z, n_total}            spring(n_total, len_x, len_y, len_z) :72-78
 *   IKB_GEN_CUBE        {step, len_x, len_y, len_z, sx, sy, sz, nx, ny}   cube(step, ...), nx = len(arange(0, len_x, step)) :39-46
 *   IKB_GEN_CUBE_RANDOM {len_x, len_y, len_z, sx, sy, sz}         cube_random: start + len * U[0,1)    :48-55
 *   IKB_GEN_NORMAL      {xlo, xhi, ylo, yhi, zlo, zhi, std_dev}   random_distribution(.., 'normal', std_dev) :80-97
 * Rows [row_offset, row_offset + n) of the trajectory are produced (a shard generates only its own range).
 * The random kinds use Philox4x32-10 keyed by (seed, row): same distributions as the reference's numpy / scipy
 * calls, reproducible per seed, but not numpy's Mersenne-Twister stream. */
#define IKB_GEN_CIRCLE 0
#define IKB_GEN_SPRING 1
#define IKB_GEN_CUBE 2
#define IKB_GEN_CUBE_RANDOM 3
#define IKB_GEN_NORMAL 4
int ikb_generate_device(ikb_engine *e, int kind, const double *params, int n_params, int64_t n, int64_t row_offset,
                        void *xyz_out, int xyz_dtype, uint64_t seed, void *stream);

/* ---- pinned host buffers ------------------------------------------------------------------------
 * The reference hands results back as freshly built Python lists (inverse.py:137,155) and the broker serialises
 * them into a new message body (rpc_broker.py:88-99).  At 1e7+ rows the allocation and the pageable copy of
 * that buffer cost more than the solve, so the array-native callers (ikine(out=...), the IKB1 broker reply) write
 * into page-locked memory obtained here: allocated by the calling thread on the engine's device context
 * (cudaHostAlloc, default flags: not portable, NUMA placement follows the caller's CPU affinity).
 * ikb_host_register page-locks an existing buffer (e.g. a received request body) for the duration of one call. */
int ikb_host_alloc(ikb_engine *e, size_t bytes, void **out);
int ikb_host_free(ikb_engine *e, void *p);
int ikb_host_register(ikb_engine *e, void *p, size_t bytes, int read_only);
int ikb_host_unregister(ikb_engine *e, void *p);

/* ---- measurement helpers --------------------------------------------------------------------- */
/* dependent-FMA-chain microbenchmark on `stream`'s device: achieved TFLOP/s (2 flops per FMA) of
 * the fp32 (dtype IKB_F32) or fp64 (IKB_F64) CUDA-core pipe; the roofline denominator for FABRIK. */
int ikb_microbench_fma(ikb_engine *e, int dtype, double *tflops_out);
/* number of kernel launches this engine has issued since creation (bench.py's gpu_launches)     */
int64_t ikb_launch_count(const ikb_engine *e);
/* the *_host pipelines with the kernels removed: n rows of in_row_bytes go host -> device and n rows of
 * out_row_bytes come back device -> host through the same staging slots, streams and chunk sizes as
 * ikb_fabrik_solve_host / ikb_ann_solve_host.  What it takes is the copy ceiling `e2e` is measured against. */
int ikb_copy_pipeline_host(ikb_engine *e, const void *in, int64_t in_row_bytes, int64_t n, void *out,
                           int64_t out_row_bytes);
/* theoretical CUDA-core peak of the engine's device in TFLOP/s: SMs x lanes (128 fp32 / 64 fp64) x 2 x max SM clock */
int ikb_theoretical_fma_peak(ikb_engine *e, int dtype, double *tflops_out);

#ifdef __cplusplus
}
#endif
#endif /* IKB200_H */

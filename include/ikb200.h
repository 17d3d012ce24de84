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
 *     ikb_stats_fetch().  Calls on different streams may overlap (the engine orders only launches
 *     that would share one of its work counters); the statistics block is engine-wide and sums
 *     over them.
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
 * chain_out = 4 x 16 doubles, row-major.  Host pointers.  *status = 1 when an angle (or alpha) is outside
 * [-2pi, 2pi] (forward.py:23-25; the matrices are still written), else 0.  This is ikb_fk_transforms_host at n = 1. */
int ikb_fk_chain_host(ikb_engine *e, const double angles[4], double chain_out[64], int *status);
/* The cumulative DH matrices T_1..T_4 of n angle sets (fkine's (T, [T1..T4]) for a batch).  angles: n x 4 of
 * angles_dtype; the arithmetic is fp64 (float32 angles are widened exactly) and is the same as ikb_fk_chain_host's, so
 * a row's bits do not depend on the batch it is in.  `out` has the angles' dtype (a float32 output is the fp64 result
 * rounded once) and, by `what`:
 *   IKB_FK_MATRICES  n x 4 x 4 x 4, row-major T_1..T_4 (the layout of chain_out above): 512 B per row in fp64
 *   IKB_FK_JOINTS    n x 4 x 3, column 3 of T_1..T_4 -- the joint origins (inverse.py:128-130), which is the `init`
 *                    layout of ikb_fabrik_chain_* for fp64
 * Rows with an angle (or alpha) outside [-2pi, 2pi] are still written; the lowest such row goes to
 * stats.first_fk_angle_range (NaN passes; float32 angles are tested after widening, so float32(2pi), which is
 * above 2pi, is outside).  `angles` and `out` must be aligned to their element size; an `out` that
 * is not 16-byte aligned is written with element stores instead of bulk copies.
 * _device: DEVICE pointers, enqueued on `stream`, the guard accumulates in the statistics block; _host: HOST pointers,
 * staged through the engine's pipeline, `stats` filled (nullable). */
#define IKB_FK_MATRICES 0
#define IKB_FK_JOINTS 1
int ikb_fk_transforms_device(ikb_engine *e, const void *angles, int angles_dtype, int64_t n,
                             int what, void *out, void *stream);
int ikb_fk_transforms_host(ikb_engine *e, const void *angles, int angles_dtype, int64_t n,
                           int what, void *out, ikb_stats *stats);
/* The arm Jacobian of n angle sets: how the effector moves when the four joints turn.  With T_0 = I and the cumulative
 * DH matrices T_1..T_4 of ikb_fk_transforms_*, joint i turns about z_{i-1} through p_{i-1} (columns 2 and 3 of
 * T_{i-1}) and p_4 is the effector.  angles: n x 4 of angles_dtype; the arithmetic is fp64 (float32 angles are widened
 * exactly), outputs have the angles' dtype (a float32 output is the fp64 result rounded once).
 *   jac_out, by `what`:
 *     IKB_JAC_GEOMETRIC  n x 6 x 4, row-major: rows 0-2 the linear part z_{i-1} x (p_4 - p_{i-1}), rows 3-5 the
 *                        angular part z_{i-1}; column i-1 belongs to joint i.  192 B per row in fp64.
 *     IKB_JAC_POSITION   n x 3 x 4, rows 0-2 only.
 *   manip_out: n values, the Yoshikawa manipulability w = sqrt(det(Jv Jv^T)) of the 3 x 4 position Jacobian Jv,
 *     evaluated as sqrt(sum over the four 3-column subsets of det^2) (Cauchy-Binet): non-negative, 0 at singular poses.
 *   Either output may be NULL, not both; `what` must be valid even without jac_out.
 * Bits: z_{i-1} and p_{i-1} are the bits of ikb_fk_transforms_*'s matrices (z_0 = (0, 0, 1), p_0 = 0), and every
 * later operation is IEEE fp64 with round-to-nearest and no contraction, in this order:
 *   d = p_4 - p_{i-1};  linear = (z.y*d.z - z.z*d.y, z.z*d.x - z.x*d.z, z.x*d.y - z.y*d.x)
 *   for the column subsets c_0 = (0,1,2), c_1 = (0,1,3), c_2 = (0,2,3), c_3 = (1,2,3) of Jv, with columns (a, b, c):
 *     m = b x c in the order of the linear rows;  det_k = (a.x*m.x + a.y*m.y) + a.z*m.z;  s_k = det_k * det_k
 *   w = sqrt((s_0 + s_1) + (s_2 + s_3)), correctly rounded.
 * Rows with an angle (or alpha) outside [-2pi, 2pi] are still written; the lowest such row goes to
 * stats.first_fk_angle_range (NaN passes, as for ikb_fk_transforms_*).  `angles` and both outputs must be aligned to
 * their element size; a jac_out that is not 16-byte aligned is written with element stores instead of bulk copies.
 * _device: DEVICE pointers, enqueued on `stream`, the guard accumulates in the statistics block; _host: HOST pointers,
 * staged through the engine's pipeline, `stats` filled (nullable).  A host chunk holds min(S, 32 S / B) rows, S the
 * rows of a staging slot and B the bytes of a jac_out row (S rows without jac_out); w is staged beside the Jacobians.
 * A NULL engine with otherwise valid arguments is refused too; the text of any refusal with e == NULL is read with
 * ikb_last_error(NULL). */
#define IKB_JAC_GEOMETRIC 0
#define IKB_JAC_POSITION 1
int ikb_jacobian_device(ikb_engine *e, const void *angles, int angles_dtype, int64_t n, int what,
                        void *jac_out, void *manip_out, void *stream);
int ikb_jacobian_host(ikb_engine *e, const void *angles, int angles_dtype, int64_t n, int what,
                      void *jac_out, void *manip_out, ikb_stats *stats);

/* Damped-least-squares (DLS) refinement of joint angles onto position targets: from a seed, every row repeats
 * Delta theta = Jv^T (Jv Jv^T + lambda^2 I)^-1 e, e = target - p_4, until it meets its own tolerance.  It puts the
 * effector on the target where FABRIK stops at its err_margin and the network's prediction a few millimetres away.
 *   xyz: n x 3 targets of xyz_dtype.  seed: n_seed x 4 angles of angles_dtype, n_seed == 1 (one seed for every row,
 *   e.g. the DH table's seed row) or n.  angles_out: n x 4 of angles_dtype; angles_out == seed with n_seed == n refines
 *   in place, any other overlap of the two is refused.  iters_out (nullable): the steps taken per row.  err_out
 *   (nullable, angles_dtype): ||target - p_4(theta_out)|| per row.  damping = lambda (metres), tol in metres,
 *   max_iter >= 0; max_iter = 0 returns the seeds with their errors.
 * The arithmetic is fp64 (float32 seeds and targets are widened exactly; a float32 output is the fp64 result rounded
 * once).  p_4 and Jv of an iterate are the bits of ikb_fk_transforms_* (IKB_FK_JOINTS, column 3 of T_4) and of
 * ikb_jacobian_* (IKB_JAC_POSITION) for it.  Every later operation is IEEE fp64 with round-to-nearest and no
 * contraction.  Per row, with k = 0:
 *   1. e = target - p_4;  err = sqrt((e.x*e.x + e.y*e.y) + e.z*e.z)
 *   2. err <= tol: stop (converged).   3. k == max_iter: stop (not converged; NaN rows end here).
 *   4. A = Jv Jv^T + lambda^2 I: A_ij = (J_i0*J_j0 + J_i1*J_j1) + (J_i2*J_j2 + J_i3*J_j3), then A_ii += L, where
 *      L = lambda*lambda rounded once.  A y = e by LDL^T:
 *        l10 = A01/A00;  l20 = A02/A00;  d1 = A11 - l10*A01;  t = A12 - l20*A01;  l21 = t/d1;
 *        d2 = (A22 - l20*A02) - l21*t;
 *        z1 = e.y - l10*e.x;  z2 = (e.z - l20*e.x) - l21*z1;
 *        y2 = z2/d2;  y1 = z1/d1 - l21*y2;  y0 = (e.x/A00 - l10*y1) - l20*y2
 *      theta_k = theta_k + ((J_0k*y0 + J_1k*y1) + J_2k*y2), then theta_k = remainder(theta_k, 2pi) when
 *      |theta_k| > pi (IEEE remainder, exact: every iterate stays inside the FK guard);  k += 1;  back to 1.
 *   (pi and 2pi are the doubles nearest them.)  iters_out = k and err_out = err at the stop.
 * Guards (rows are still computed and written): a target outside the workspace box sets stats.first_out_of_limits
 * (the inclusive test of ikb_check_limits_*, NaN passes); a seed angle, or an alpha, outside [-2pi, 2pi] sets
 * stats.first_fk_angle_range (the test of ikb_fk_transforms_*).  Statistics: n_solved rows, sum_iterations steps,
 * n_iter_capped rows that ended above tol (NaN rows included), sum_fk_error / n_fk_error the final errors of the
 * finite rows.
 * Refused with IKB_ERR_INVALID before the engine is looked at, each with its own message (read with
 * ikb_last_error(NULL) when e == NULL): NULL targets, seeds or angles_out (n > 0), negative n, n_seed not 1 or n, an
 * unknown dtype, damping <= 0 or not finite, tol < 0 or NaN, max_iter < 0, a buffer not aligned to its element size
 * (iters_out: 4 bytes), a partial overlap of seed and angles_out, and a NULL engine.  Nothing is launched for a
 * refused call or for n = 0.
 * _device: DEVICE pointers, enqueued on `stream`, one launch; statistics accumulate in the engine's block.  _host:
 * HOST pointers, staged through the engine's pipeline with no per-call allocation, `stats` filled (nullable): targets
 * in the slot's target buffer, seeds in its input buffer (a single seed copied once per slot), angles in its output
 * buffer, iterations in its auxiliary buffer, and err_out behind the targets.  A host chunk, one launch, holds
 * 3 S / 4 rows with err_out and S rows without, S the rows of a staging slot. */
int ikb_dls_refine_device(ikb_engine *e, const void *xyz, int xyz_dtype, int64_t n, const void *seed, int64_t n_seed,
                          void *angles_out, int angles_dtype, double damping, double tol, int32_t max_iter,
                          int32_t *iters_out /* nullable */, void *err_out /* nullable, angles_dtype */,
                          void *stream);
int ikb_dls_refine_host(ikb_engine *e, const void *xyz, int xyz_dtype, int64_t n, const void *seed, int64_t n_seed,
                        void *angles_out, int angles_dtype, double damping, double tol, int32_t max_iter,
                        int32_t *iters_out /* nullable */, void *err_out /* nullable, angles_dtype */,
                        ikb_stats *stats);

/* Damped-least-squares refinement of joint angles onto full effector poses (position and orientation), weighted per
 * task axis: from a seed, every row repeats Delta theta = (J^T W J + lambda^2 I)^-1 J^T W e, J the 6 x 4 geometric
 * Jacobian, W = diag(weights), until it meets its own tolerance.  The arm has 4 joints and a pose 6 components, so a
 * pose that is not the FK of some angles is generally not reachable; the weights decide what is matched then.
 *   poses: n x 4 x 4 of pose_dtype, row-major, the layout of one matrix of ikb_fk_transforms_* (IKB_FK_MATRICES): rows
 *   0-2 hold [R_d | p_d], row 3 is not read.  weights: 6 HOST doubles, the position axes x, y, z then the three
 *   orientation axes, each >= 0 and finite, not all zero.  damping = lambda (joint space: A's unit is that of J^T W J),
 *   tol >= 0 on err below.  Everything else -- seeds, n_seed, in place, iters_out, err_out (angles_dtype), max_iter = 0
 *   returning the seeds with their errors -- is as for ikb_dls_refine_*.
 * The arithmetic is fp64 (float32 seeds and poses are widened exactly; a float32 output is the fp64 result rounded
 * once).  R, p = T_4 of an iterate are the bits of ikb_fk_transforms_* (IKB_FK_MATRICES) and J those of
 * ikb_jacobian_* (IKB_JAC_GEOMETRIC) for it.  Every later operation is IEEE fp64 with round-to-nearest and no
 * contraction (sqrt correctly rounded).  Per row, with k = 0:
 *   1. e_p = p_d - p.  M = R_d R^T: M_ij = (Rd_i0*R_j0 + Rd_i1*R_j1) + Rd_i2*R_j2.  tr = (M00 + M11) + M22;
 *      dx = M21 - M12, dy = M02 - M20, dz = M10 - M01.  e_o = 2 x the vector part of M's unit quaternion with a
 *      non-negative scalar part (Shepperd), zero only for no rotation, so a row 180 degrees off is not converged:
 *        tr >= M00, tr >= M11 and tr >= M22:  h = sqrt(1 + tr);  e_o = (dx/h, dy/h, dz/h)
 *        else M00 >= M11 and M00 >= M22:     h = sqrt(((1 + M00) - M11) - M22);
 *                                            e_o = (h, (M01 + M10)/h, (M02 + M20)/h), negated when dx < 0
 *        else M11 >= M22:                    h = sqrt(((1 + M11) - M00) - M22);
 *                                            e_o = ((M01 + M10)/h, h, (M12 + M21)/h), negated when dy < 0
 *        else:                               h = sqrt(((1 + M22) - M00) - M11);
 *                                            e_o = ((M02 + M20)/h, (M12 + M21)/h, h), negated when dz < 0
 *      e = (e_p, e_o), s_i = w_i*(e_i*e_i);  err = sqrt(((s0 + s1) + s2) + ((s3 + s4) + s5))
 *   2. err <= tol: stop (converged).   3. k == max_iter: stop (not converged; NaN rows end here).
 *   4. For task rows q = 0..5 (J_q: row q of J): g_q = w_q*J_q elementwise.  For i = 0, 1, 2, pairing linear row i
 *      with angular row 3 + i:  P_i[k][m] = g_ik*J_im + g_(3+i)k*J_(3+i)m  (k <= m),  c_i[k] = g_ik*e_i + g_(3+i)k*e_(3+i);
 *      A_km = (P_0 + P_1) + (P_2 + 0) and b_k = (c_0 + c_1) + (c_2 + 0) elementwise (the "+ 0" turns -0 into +0);
 *      then A_kk += L, L = lambda*lambda rounded once.  A y = b by LDL^T:
 *        l10 = A01/A00;  l20 = A02/A00;  l30 = A03/A00;
 *        d1 = A11 - l10*A01;  t21 = A12 - l20*A01;  t31 = A13 - l30*A01;  l21 = t21/d1;  l31 = t31/d1;
 *        d2 = (A22 - l20*A02) - l21*t21;  t32 = (A23 - l30*A02) - l31*t21;  l32 = t32/d2;
 *        d3 = ((A33 - l30*A03) - l31*t31) - l32*t32;
 *        z1 = b1 - l10*b0;  z2 = (b2 - l20*b0) - l21*z1;  z3 = ((b3 - l30*b0) - l31*z1) - l32*z2;
 *        y3 = z3/d3;  y2 = z2/d2 - l32*y3;  y1 = (z1/d1 - l21*y2) - l31*y3;  y0 = ((b0/A00 - l10*y1) - l20*y2) - l30*y3
 *      theta_k = theta_k + y_k, then theta_k = remainder(theta_k, 2pi) when |theta_k| > pi;  k += 1;  back to 1.
 *   iters_out = k and err_out = err at the stop.  With weights (1, 1, 1, 0, 0, 0) the step equals ikb_dls_refine_*'s
 *   mathematically (J^T (J J^T + L I)^-1 = (J^T J + L I)^-1 J^T), not in bits.
 * Guards and statistics are those of ikb_dls_refine_*, the box test on the position column p_d; sum_fk_error /
 * n_fk_error sum the final weighted errors of the finite rows.
 * Refused with IKB_ERR_INVALID before the engine is looked at, each with its own message: NULL weights, a weight
 * that is negative or not finite, all six weights zero, then every refusal of ikb_dls_refine_* (NULL poses are "NULL
 * targets"; the pose buffer must be aligned to its element size).  Nothing is launched for a refused call or n = 0.
 * _device: DEVICE pointers, enqueued on `stream`, one launch.  _host: HOST pointers, staged through the engine's
 * pipeline with no per-call allocation, `stats` filled (nullable): poses in the slot's input buffer, seeds in its
 * target buffer with err_out behind them, angles in its output buffer, iterations in its auxiliary buffer.  A host
 * chunk, one launch, holds S / 4 rows, S the rows of a staging slot. */
int ikb_dls_pose_refine_device(ikb_engine *e, const void *poses, int pose_dtype, int64_t n, const void *seed,
                               int64_t n_seed, void *angles_out, int angles_dtype, const double weights[6],
                               double damping, double tol, int32_t max_iter, int32_t *iters_out /* nullable */,
                               void *err_out /* nullable, angles_dtype */, void *stream);
int ikb_dls_pose_refine_host(ikb_engine *e, const void *poses, int pose_dtype, int64_t n, const void *seed,
                             int64_t n_seed, void *angles_out, int angles_dtype, const double weights[6],
                             double damping, double tol, int32_t max_iter, int32_t *iters_out /* nullable */,
                             void *err_out /* nullable, angles_dtype */, ikb_stats *stats);

/* Closed-form inverse kinematics: every solution branch of n effector poses, or of n positions at a given approach
 * (pitch) angle, for arms with a turning base and three parallel joints.  That family is: alpha_2 = alpha_3 =
 * alpha_4 = 0, |cos alpha_1| <= 1e-12 (treated as 0; s = sign(sin alpha_1)), a_2 > 0 and a_3 > 0; a_1, a_4 and every
 * epsilon are free, d = (eps_2 + eps_3) + eps_4 is the lateral offset.  (Indices count joints from 1 here, as the
 * DH table's columns: a_1 = dh[2][0].)  The reference's arm is in it.  Any other table is refused with
 * IKB_ERR_UNSUPPORTED: the damped-least-squares entries (ikb_dls_pose_refine_*) serve it.
 * The arithmetic is fp64 (float32 inputs are widened exactly, a float32 output is the fp64 result rounded once); every
 * input element is read as x + 0, so -0 and +0 give the same bits.  Every angle leaving [-pi, pi] is wrapped with the
 * exact IEEE remainder(theta, 2pi), as in ikb_dls_refine_*, so every answer is inside the FK guard and valid as a seed.
 *   Two-link triangle, from in-plane coordinates (u, v) of the effector and phi = theta_2 + theta_3 + theta_4:
 *     uw = u - a_4 cos phi;  vw = v - a_4 sin phi;  r = sqrt(uw^2 + vw^2)
 *     num = ((a_2 + a_3) - r)((a_2 + a_3) + r);  den = (r - (a_2 - a_3))(r + (a_2 - a_3))
 *     t = 2 atan2(sqrt(num > 0 ? num : 0), sqrt(den > 0 ? den : 0))   (half-angle form: exact near the folded arm)
 *     beta = atan2(vw, uw);  g = atan2(a_3 sin t, a_2 + a_3 cos t)
 *     elbow +: theta_3 = t,      theta_2 = beta - g
 *     elbow -: theta_3 = 0 - t,  theta_2 = beta - (0 - g)    (identical bits to elbow + at t = 0)
 *     theta_4 = (phi - theta_2) - theta_3, with the unwrapped theta_2.
 *   IKB_AIK_POSE: in = n x 4 x 4 poses of in_dtype, row-major (the layout of ikb_fk_transforms_*, rows 0-2 read), with
 *   x = column 0, z = column 2, p = column 3:
 *     theta_1 = atan2(s z_x, -s z_y);  phi = atan2(s x_z, c_1 x_x + s_1 x_y)
 *     u = (c_1 p_x + s_1 p_y) - a_1;  v = s (p_z - eps_1)
 *     2 branches per row, ordered [elbow +, elbow -].  A pose that no angles produce is projected onto the arm's plane
 *     by the same formulas: its angles are defined, and a refinement takes them on to what its weights ask for.
 *   IKB_AIK_POSITION_PITCH: in = n x 3 targets; pitch = n_pitch values (1 or n) of in_dtype, the angle of the tool axis
 *   x_4 above the horizontal:
 *     rho2 = p_x^2 + p_y^2;  q = sqrt(rho2 < d^2 ? 0 : rho2 - d^2)
 *     front: q' = q, phi = pitch;  back (reaching over the base): q' = -q, phi = pi - pitch
 *     theta_1 = atan2(p_y, p_x) - atan2(-s d + 0, q');  u = q' - a_1;  v = s (p_z - eps_1)
 *     4 branches per row, ordered [front +, front -, back +, back -].  With d = 0 all four give the same tool axis
 *     x_4 = (cos(pitch) r^, s sin(pitch)).  A target on the base axis (p_x = p_y = 0, either sign) with d = 0 gets
 *     theta_1 = 0 on the front branches and -pi on the back ones.
 * status_out (nullable, n int32): bit b is set when branch b does not reach -- num < 0 (the arm is stretched toward
 * the wrist, t = 0), den < 0 (folded toward it, t = pi), or rho2 < d^2 (position kind; q = 0 is used).  num = 0 counts
 * as reached.  A row with a non-finite input element (or pitch) gets NaN angles and every bit set.
 * Guard: a position (column 3 of a pose) outside the workspace box sets stats.first_out_of_limits (the inclusive test of
 * ikb_check_limits_*, NaN passes); the rows are still written.  n_solved counts the rows.
 * Refused with IKB_ERR_INVALID before the engine is looked at, each with its own message (read with
 * ikb_last_error(NULL) when e == NULL): NULL input or angles_out (n > 0), an unknown kind or dtype, negative n, a NULL
 * pitch for the position kind (n > 0) or a pitch for the pose kind, n_pitch not 1 or n (position kind), a buffer not
 * aligned to its element size (pitch: in_dtype, status_out: 4 bytes), then a NULL engine; then a table outside the
 * family with IKB_ERR_UNSUPPORTED.  Nothing is launched for a refused call or for n = 0.
 * _device: DEVICE pointers, enqueued on `stream`, one launch; the guard accumulates in the engine's block.  _host:
 * HOST pointers, staged through the engine's pipeline with no per-call allocation, `stats` filled (nullable).  A host
 * chunk, one launch, holds S / 4 rows, S the rows of a staging slot. */
#define IKB_AIK_POSE 0
#define IKB_AIK_POSITION_PITCH 1
int ikb_analytic_ik_device(ikb_engine *e, int kind, const void *in, int in_dtype, int64_t n, const void *pitch,
                           int64_t n_pitch, void *angles_out /* n x B x 4 */, int angles_dtype,
                           int32_t *status_out /* nullable */, void *stream);
int ikb_analytic_ik_host(ikb_engine *e, int kind, const void *in, int in_dtype, int64_t n, const void *pitch,
                         int64_t n_pitch, void *angles_out /* n x B x 4 */, int angles_dtype,
                         int32_t *status_out /* nullable */, ikb_stats *stats);

/* ---- ANN (ann.py:70-85, inverse.py:142-155)-------------------------------------------------- */
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

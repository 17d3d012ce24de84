"""Inverse kinematics front classes -- API of reference kinematics/inverse.py.

``FabrikInverseKinematics.ikine`` and ``AnnInverseKinematics.ikine`` keep the reference's
signatures, return types (list of [theta1..theta4] python floats) and exceptions, so cli.py
(--inverse-kine) and rpc_broker.py run on top of them unchanged.  The per-target python loop of the
reference (inverse.py:120-137) becomes ONE call into libikb200.so for the whole trajectory; pass
``as_array=True`` (and float32/float64 ndarrays in) to skip the python list round trip.

Differences from upstream, all documented in DESIGN.md:
  * ``ikine`` does not write theta_1 of the last target into the caller's ``dh_matrix[0][0]``
    (upstream side effect at inverse.py:125, asserted by no test).
  * degenerate targets (on the z axis / coincident joints) give defined results (NaN angles +
    ZeroDivisionError for a zero-length segment) instead of rounding-noise-dependent ones.
"""
from abc import ABC, abstractmethod

import numpy as np

from ..engine import DLS_DAMPING, DLS_MAX_ITER, DLS_TOL, POSE_DAMPING, POSE_MAX_ITER, POSE_TOL, POSE_WEIGHTS
from ..robot.robot import OutOfRobotReachException
from ._shared import get_engine, points_to_array
from .ann import ANN
from .forward import _ANGLE_MSG, ForwardKinematics


def poses_to_array(dest_poses):
    """(n, 4, 4) poses -- an array such as fkine_batch(angles)[0], or nested lists -> contiguous float array (float32
    arrays stay float32, everything else becomes float64)."""
    if isinstance(dest_poses, np.ndarray) and dest_poses.dtype in (np.float32, np.float64):
        arr = dest_poses
    else:
        arr = np.asarray(dest_poses, dtype=np.float64)
    if arr.size == 0:
        return np.zeros((0, 4, 4), dtype=np.float64)
    if arr.ndim != 3 or arr.shape[1:] != (4, 4):
        raise ValueError(f'destination poses must have shape (n, 4, 4), not {arr.shape}')
    return np.ascontiguousarray(arr)


class _PosePositions:
    """Stands in for the destination points in the exception messages: item i is pose i's position [x, y, z]."""

    def __init__(self, poses):
        self._poses = poses

    def __getitem__(self, i):
        return self._poses[i, :3, 3].tolist()


def _empty_result(dtype, as_array, return_iterations, return_fk_error):
    empty = np.zeros((0, 4), dtype=dtype)
    empty = empty if as_array else []
    extras = ((np.zeros(0, np.int32),) if return_iterations else ()) + \
             ((np.zeros(0, dtype),) if return_fk_error else ())
    return (empty,) + extras if extras else empty


class InverseKinematics(ABC):
    """Inverse kinematics base (reference inverse.py:18-40)."""

    def __init__(self, dh_matrix, joints_distances, workspace_limits, device=None):
        self.dh_matrix = dh_matrix
        self.joints_distances = joints_distances
        self.workspace_limits = workspace_limits
        self.fkine = ForwardKinematics(self.dh_matrix, device=device)
        self._device = device
        self._max_err = 0.001
        self._max_iter = 100

    def _engine(self):
        return get_engine(self.dh_matrix, self.joints_distances, self.workspace_limits,
                          self._max_err, self._max_iter, self._device)

    def _limits_error(self, dest_points, index):
        # message text of reference inverse.py:32-35; `dest_points[index]` prints as upstream does
        # ([1, 2, 7] for a list row, Point(1, 2, 7) for a Point)
        return OutOfRobotReachException(
            f'Inverse Kinematics exception, point {dest_points[index]} '
            'is out of manipulator reach area! '
            f'Limits: {self.workspace_limits}')

    def check_limits(self, dest_points):
        """Raise OutOfRobotReachException for the first point outside the workspace box."""
        arr = points_to_array(dest_points)
        if arr.shape[0] == 0:
            return
        first_bad = self._engine().check_limits(arr)
        if first_bad >= 0:
            raise self._limits_error(dest_points, first_bad)

    def _raise_from_stats(self, dest_points, stats):
        if stats.first_out_of_limits >= 0:  # whole-batch semantics: limits first (inverse.py:117)
            raise self._limits_error(dest_points, stats.first_out_of_limits)
        rows = [(r, kind) for r, kind in ((stats.first_zero_division, ZeroDivisionError),
                                          (stats.first_domain_error, ValueError)) if r >= 0]
        if rows:
            _, kind = min(rows, key=lambda t: t[0])  # same row in both classes: the division comes first upstream
            raise kind('float division by zero' if kind is ZeroDivisionError else 'math domain error')

    @abstractmethod
    def ikine(self, dest_points):
        """Calculate inverse kinematics"""

    def refine(self, dest_points, angles, damping=DLS_DAMPING, tol=DLS_TOL, max_iter=DLS_MAX_ITER, as_array=False,
               return_iterations=False, return_fk_error=False):
        """Refine joint angles onto the destination points by damped least squares on the GPU: from `angles` (one row
        per point, or one row for all of them; e.g. what `ikine` returned), each row repeats
        Delta theta = Jv^T (Jv Jv^T + damping^2 I)^-1 (point - FK(theta)) until ||FK(theta) - point|| <= tol or
        `max_iter` steps (include/ikb200.h ikb_dls_refine_* states the arithmetic).  The angles come back wrapped to
        [-pi, pi] where a step left that range.

        The result has the seeds' dtype: a list gives float64, a float32 array float32.  The network's float32
        predictions should be widened (``angles.astype(np.float64)``) to refine below about 1e-6 m, since float32
        angles cannot resolve the effector more finely than that.  Return shapes follow `ikine`: a list of rows, or an
        (n, 4) array with `as_array`, then the step counts (`return_iterations`) and ||FK(theta) - point||
        (`return_fk_error`).  A point outside the workspace box raises OutOfRobotReachException with `ikine`'s message
        (checked first), a seed angle outside [-2pi, 2pi] with the forward-kinematics one."""
        arr = points_to_array(dest_points)
        seed = angles if isinstance(angles, np.ndarray) and angles.dtype in (np.float32, np.float64) else \
            np.asarray(angles, dtype=np.float64)
        if arr.shape[0] == 0:
            empty = np.zeros((0, 4), dtype=seed.dtype)
            empty = empty if as_array else []
            extras = ((np.zeros(0, np.int32),) if return_iterations else ()) + \
                     ((np.zeros(0, seed.dtype),) if return_fk_error else ())
            return (empty,) + extras if extras else empty
        res = self._engine().dls_refine(arr, seed, damping, tol, max_iter, return_iters=return_iterations,
                                        return_error=return_fk_error)
        out, stats = res[0], res[1]
        self.last_stats = stats
        if stats.first_out_of_limits >= 0:
            raise self._limits_error(dest_points, stats.first_out_of_limits)
        if stats.first_fk_angle_range >= 0:
            raise OutOfRobotReachException(_ANGLE_MSG)
        out = out if as_array else out.tolist()
        return (out,) + tuple(res[2:]) if len(res) > 2 else out

    def refine_device(self, points, angles, out=None, iters=None, fk_err=None, damping=DLS_DAMPING, tol=DLS_TOL,
                      max_iter=DLS_MAX_ITER):
        """`refine` on CUDA tensors, enqueued on torch's current stream without a synchronisation: points (n, 3),
        angles (n, 4) or one row for all points, float32 or float64; out (n, 4) in the angles' dtype is allocated when
        None and may be `angles` itself (in place), so ``ann_solve_device`` -> ``refine_device(..., out=angles)``
        needs no host round trip.  iters (int32) and fk_err (angles' dtype), when given, receive the step counts and
        the final errors.  Returns out.  The guards set first_out_of_limits / first_fk_angle_range of the engine's
        statistics (``stats_fetch_torch``) instead of raising."""
        import torch
        if out is None:
            out = torch.empty((points.shape[0], 4), dtype=angles.dtype, device=angles.device)
        self._engine().dls_refine_device(points, angles, out, iters, fk_err, damping, tol, max_iter)
        return out

    def _raise_pose_errors(self, poses, stats):
        if stats.first_out_of_limits >= 0:
            raise self._limits_error(_PosePositions(poses), stats.first_out_of_limits)
        if stats.first_fk_angle_range >= 0:
            raise OutOfRobotReachException(_ANGLE_MSG)

    def refine_pose(self, dest_poses, angles, weights=POSE_WEIGHTS, damping=POSE_DAMPING, tol=POSE_TOL,
                    max_iter=POSE_MAX_ITER, as_array=False, return_iterations=False, return_fk_error=False):
        """Refine joint angles onto full effector poses (position and orientation) by weighted damped least squares on
        the GPU.  dest_poses: (n, 4, 4) homogeneous transforms, e.g. ``self.fkine.fkine_batch(theta)[0]``; rows 0-2
        are read.  From `angles` (one row per pose, or one row for all), each row repeats
        Delta theta = (J^T W J + damping^2 I)^-1 J^T W e over the 6 x 4 geometric Jacobian J, with e = (position error,
        2 x the vector part of the rotation error's quaternion) and W = diag(weights), until
        sqrt(sum w_i e_i^2) <= tol or `max_iter` steps (include/ikb200.h ikb_dls_pose_refine_* states the arithmetic).
        The arm has four joints: a pose that no angles produce stops at max_iter, matched as the weights ask.

        Dtypes, return shapes and exceptions follow `refine`: a pose whose position is outside the workspace box
        raises OutOfRobotReachException with `ikine`'s message naming that position [x, y, z] (checked first), a seed
        angle outside [-2pi, 2pi] the forward-kinematics one.  `return_fk_error` gives the weighted error."""
        poses = poses_to_array(dest_poses)
        seed = angles if isinstance(angles, np.ndarray) and angles.dtype in (np.float32, np.float64) else \
            np.asarray(angles, dtype=np.float64)
        if poses.shape[0] == 0:
            return _empty_result(seed.dtype, as_array, return_iterations, return_fk_error)
        res = self._engine().dls_pose_refine(poses, seed, weights, damping, tol, max_iter,
                                             return_iters=return_iterations, return_error=return_fk_error)
        out, stats = res[0], res[1]
        self.last_stats = stats
        self._raise_pose_errors(poses, stats)
        out = out if as_array else out.tolist()
        return (out,) + tuple(res[2:]) if len(res) > 2 else out

    def refine_pose_device(self, poses, angles, out=None, iters=None, fk_err=None, weights=POSE_WEIGHTS,
                           damping=POSE_DAMPING, tol=POSE_TOL, max_iter=POSE_MAX_ITER):
        """`refine_pose` on CUDA tensors, enqueued on torch's current stream without a synchronisation: poses a
        contiguous (n, 4, 4) tensor, angles (n, 4) or one row for all poses, float32 or float64; out, iters and fk_err
        as for `refine_device` (out may be `angles`: in place).  Returns out.  The guards set first_out_of_limits /
        first_fk_angle_range of the engine's statistics (``stats_fetch_torch``) instead of raising."""
        import torch
        if out is None:
            out = torch.empty((poses.shape[0], 4), dtype=angles.dtype, device=angles.device)
        self._engine().dls_pose_refine_device(poses, angles, out, iters, fk_err, weights, damping, tol, max_iter)
        return out

    def _ikine_pose(self, dest_poses, seed_on_device, weights, damping, tol, max_iter, as_array, return_iterations,
                    return_fk_error):
        """Upload the poses once, seed with `seed_on_device(poses) -> (engine, float64 seeds)` from the device poses
        (n, 4, 4), raise what `ikine` raises, refine onto the poses in place and download once."""
        import torch
        poses = poses_to_array(dest_poses)
        n = poses.shape[0]
        if n == 0:
            return _empty_result(np.float64, as_array, return_iterations, return_fk_error)
        eng = self._engine()
        d_poses = torch.from_numpy(poses).to(torch.device("cuda", eng.device))
        solver, seed = seed_on_device(d_poses)
        stats = solver.stats_fetch_torch()
        self.last_stats = stats
        self._raise_from_stats(_PosePositions(poses), stats)
        eng.stats_reset_torch()
        iters = torch.empty(n, dtype=torch.int32, device=seed.device) if return_iterations else None
        err = torch.empty(n, dtype=seed.dtype, device=seed.device) if return_fk_error else None
        eng.dls_pose_refine_device(d_poses, seed, seed, iters, err, weights, damping, tol, max_iter)
        out = seed.cpu().numpy()
        extras = tuple(t.cpu().numpy() for t in (iters, err) if t is not None)
        stats = eng.stats_fetch_torch()
        self.last_stats = stats
        self._raise_pose_errors(poses, stats)
        out = out if as_array else out.tolist()
        return (out,) + extras if extras else out


class FabrikInverseKinematics(InverseKinematics):
    """Reaching inverse kinematics using the FABRIK method (reference inverse.py:45-139)."""

    def __init__(self, dh_matrix, joints_distances, workspace_limits,
                 max_err=0.001, max_iterations_num=100, device=None, precision='f64'):
        super().__init__(dh_matrix, joints_distances, workspace_limits, device=device)
        from .fabrik import Fabrik
        self.fabrik = Fabrik(joints_distances, max_err, max_iterations_num, device=device)
        self._max_err = max_err
        self._max_iter = max_iterations_num
        self.precision = precision
        self.last_stats = None

    def ikine(self, dest_points, as_array=False, return_iterations=False, out=None, return_fk_error=False):
        """Joint angles [theta1..theta4] for every destination point.

        `out` (optional, implies as_array): a preallocated (n, 4) float32/float64 array -- e.g. pinned
        host memory -- that receives the angles.  `return_fk_error` appends ||FK(angles) - point|| per point (the
        check the reference CLI plots, cli.py:56-61), computed inside the solver kernel."""
        arr = points_to_array(dest_points)
        if arr.shape[0] == 0:
            empty = np.zeros((0, 4)) if as_array else []
            extras = ((np.zeros(0, np.int32),) if return_iterations else ()) + \
                     ((np.zeros(0),) if return_fk_error else ())
            return (empty,) + extras if extras else empty
        if out is not None:
            as_array = True
        res = self._engine().fabrik_solve(arr, out=out, precision=self.precision, return_iters=return_iterations,
                                          return_fk_error=return_fk_error, fk_stats=return_fk_error)
        angles, stats = res[0], res[1]
        self.last_stats = stats
        self._raise_from_stats(dest_points, stats)
        out = angles if as_array else angles.tolist()
        return (out,) + tuple(res[2:]) if len(res) > 2 else out

    def ikine_pose(self, dest_poses, weights=POSE_WEIGHTS, damping=POSE_DAMPING, tol=POSE_TOL, max_iter=POSE_MAX_ITER,
                   as_array=False, return_iterations=False, return_fk_error=False):
        """Joint angles that put the effector on each (4, 4) pose: FABRIK on the pose's position column, then
        `refine_pose` from there, all on the GPU (one upload of the poses, one download of the float64 angles).
        Raises what `ikine` raises for those positions, then what `refine_pose` raises; returns as `refine_pose`."""
        import torch

        def seed(poses):
            eng = self._engine()
            xyz = poses[:, :3, 3].contiguous()
            angles = torch.empty((xyz.shape[0], 4), dtype=torch.float64, device=xyz.device)
            eng.stats_reset_torch()
            eng.fabrik_solve_device(xyz, angles, precision=self.precision)
            return eng, angles
        return self._ikine_pose(dest_poses, seed, weights, damping, tol, max_iter, as_array, return_iterations,
                                return_fk_error)


class AnnInverseKinematics(InverseKinematics):
    """Reaching inverse kinematics using the neural network (reference inverse.py:142-155)."""

    def __init__(self, dh_matrix, joints_distances, workspace_limits, device=None):
        super().__init__(dh_matrix, joints_distances, workspace_limits, device=device)
        self.ann = ANN(workspace_limits, dh_matrix, device=device)
        self.last_stats = None

    def load_model(self, model_name):
        """Load model weights + scalers (reference inverse.py:148-150)."""
        self.ann.load_model(model_name)

    def ikine(self, dest_points, as_array=False, out=None, return_fk_error=False):
        """Predict thetas using the neural network (limits checked first, inverse.py:154)."""
        arr = points_to_array(dest_points)
        if arr.shape[0] == 0:
            empty = np.zeros((0, 4), dtype=np.float32) if as_array else []
            return (empty, np.zeros(0, np.float32)) if return_fk_error else empty
        if out is not None:
            as_array = True
        res = self.ann.predict_with_stats(arr, out=out, return_fk_error=return_fk_error)
        angles, stats = res[0], res[1]
        self.last_stats = stats
        self._raise_from_stats(dest_points, stats)
        angles = angles if as_array else angles.tolist()
        return (angles, res[2]) if return_fk_error else angles

    def ikine_pose(self, dest_poses, weights=POSE_WEIGHTS, damping=POSE_DAMPING, tol=POSE_TOL, max_iter=POSE_MAX_ITER,
                   as_array=False, return_iterations=False, return_fk_error=False):
        """Joint angles that put the effector on each (4, 4) pose: the network's prediction for the pose's position
        column, widened to float64, then `refine_pose` from there, all on the GPU (one upload of the poses, one
        download of the angles).  Raises what `ikine` raises for those positions, then what `refine_pose` raises;
        returns as `refine_pose`."""
        import torch

        def seed(poses):
            eng = self.ann._ensure_uploaded()
            xyz = poses[:, :3, 3].contiguous()
            pred = torch.empty((xyz.shape[0], 4), dtype=torch.float32, device=xyz.device)
            eng.stats_reset_torch()
            eng.ann_solve_device(xyz, pred, mode=self.ann.mode)
            return eng, pred.double()
        return self._ikine_pose(dest_poses, seed, weights, damping, tol, max_iter, as_array, return_iterations,
                                return_fk_error)


_BASES = {"front": 0, "back": 2}
_ELBOWS = {1: 0, -1: 1}


def _branch(elbow, base="front"):
    """The branch index of ikb_analytic_ik_*: elbow 1 (theta3 >= 0) or -1 (theta3 <= 0), base 'front' (reaching
    toward the target) or 'back' (over the base)."""
    if elbow not in _ELBOWS:
        raise ValueError(f"elbow must be 1 (theta3 >= 0) or -1 (theta3 <= 0), got {elbow!r}")
    if base not in _BASES:
        raise ValueError(f"base must be 'front' or 'back', got {base!r}")
    return _BASES[base] + _ELBOWS[elbow]


class AnalyticInverseKinematics(InverseKinematics):
    """Closed-form inverse kinematics for arms with a turning base and three parallel joints (alpha_2..4 = 0,
    |cos alpha_1| <= 1e-12, a_2, a_3 > 0; the reference's arm is one): every solution branch, computed exactly
    rather than searched for.  A pose has two (one per elbow sign); a position with the tool axis' pitch above the
    horizontal (e.g. -pi/2: pointing down) has four: reaching toward the target or back over the base, times the elbow
    signs.  include/ikb200.h ikb_analytic_ik_* states the arithmetic.  Other DH tables raise RuntimeError on the
    first solve; `ikine_pose` of the other solvers serves them."""

    def __init__(self, dh_matrix, joints_distances, workspace_limits, device=None):
        super().__init__(dh_matrix, joints_distances, workspace_limits, device=device)
        self.last_stats = None

    def _solve(self, x, pitch, dest):
        angles, status, stats = self._engine().analytic_ik(x, pitch)
        self.last_stats = stats
        if stats.first_out_of_limits >= 0:
            raise self._limits_error(dest, stats.first_out_of_limits)
        return angles, status

    def ikine_branches(self, dest_points, pitch):
        """All four branches for (n, 3) points at `pitch` (one value or one per point): (angles (n, 4, 4) float64,
        ordered [front +, front -, back +, back -], status int32 (n,), bit b set when branch b does not reach -- the
        arm then points stretched or folded toward the wrist).  A point outside the workspace box raises
        OutOfRobotReachException with `ikine`'s message."""
        arr = points_to_array(dest_points)
        if arr.shape[0] == 0:
            return np.zeros((0, 4, 4)), np.zeros(0, np.int32)
        return self._solve(arr, np.asarray(pitch, dtype=np.float64), dest_points)

    def ikine(self, dest_points, pitch, elbow=1, base="front", as_array=False, return_status=False):
        """Joint angles [theta1..theta4] for every destination point with the tool axis at `pitch` above the
        horizontal: the branch with `elbow` 1 (theta3 >= 0) or -1 (theta3 <= 0), reaching toward the point
        (base='front') or back over the base (base='back').  Returns a list of rows, or an (n, 4) float64 array with
        `as_array`; `return_status` appends an int32 array, 1 where that branch does not reach (the angles then point
        the arm toward the point, stretched or folded).  Raises what `ikine_branches` raises."""
        b = _branch(elbow, base)
        angles, status = self.ikine_branches(dest_points, pitch)
        out = np.ascontiguousarray(angles[:, b])
        out = out if as_array else out.tolist()
        return (out, (status >> b) & 1) if return_status else out

    def ikine_device(self, points, pitch, out=None, status=None):
        """All four branches on CUDA tensors, enqueued on torch's current stream without a synchronisation: points
        (n, 3), pitch a tensor of the points' dtype with 1 or n elements, or a number; out (n, 4, 4) float32 or float64
        is allocated (float64) when None; status int32 (n,) or None.  Returns out.  The box guard sets
        first_out_of_limits of the engine's statistics (``stats_fetch_torch``) instead of raising."""
        import torch
        if not torch.is_tensor(pitch):
            pitch = torch.tensor([float(pitch)], dtype=points.dtype, device=points.device)
        if out is None:
            out = torch.empty((points.shape[0], 4, 4), dtype=torch.float64, device=points.device)
        self._engine().analytic_ik_device(points, pitch, out, status)
        return out

    def ikine_pose_branches(self, dest_poses):
        """Both branches for (n, 4, 4) poses: (angles (n, 2, 4) float64, ordered [theta3 >= 0, theta3 <= 0], status
        int32 (n,), bit b set when branch b does not reach).  theta1 comes from the pose's joint axis, so it is always
        on the side the pose reaches.  A pose that no angles produce is projected onto the arm's plane.  A position
        outside the workspace box raises OutOfRobotReachException with `ikine`'s message naming it."""
        poses = poses_to_array(dest_poses)
        if poses.shape[0] == 0:
            return np.zeros((0, 2, 4)), np.zeros(0, np.int32)
        return self._solve(poses, None, _PosePositions(poses))

    def ikine_pose_device(self, poses, out=None, status=None):
        """Both branches of (n, 4, 4) CUDA poses, enqueued on torch's current stream without a synchronisation; out
        (n, 2, 4) float32 or float64 is allocated (float64) when None; status int32 (n,) or None.  Returns out.  The
        box guard sets first_out_of_limits of the engine's statistics (``stats_fetch_torch``) instead of raising."""
        import torch
        if out is None:
            out = torch.empty((poses.shape[0], 2, 4), dtype=torch.float64, device=poses.device)
        self._engine().analytic_ik_device(poses, None, out, status)
        return out

    def ikine_pose(self, dest_poses, elbow=1, refine=True, weights=POSE_WEIGHTS, damping=POSE_DAMPING, tol=POSE_TOL,
                   max_iter=POSE_MAX_ITER, as_array=False, return_iterations=False, return_fk_error=False):
        """Joint angles that put the effector on each (4, 4) pose: the closed-form branch of `elbow` (1: theta3 >= 0,
        -1: theta3 <= 0), then `refine_pose` from there in place (refine=False: no steps, the closed form with its
        weighted error), all on the GPU (one upload of the poses, one download of the float64 angles).  Returns and
        raises as the other solvers' `ikine_pose`."""
        import torch
        b = _branch(elbow)

        def seed(poses):
            eng = self._engine()
            branches = torch.empty((poses.shape[0], 2, 4), dtype=torch.float64, device=poses.device)
            eng.stats_reset_torch()
            eng.analytic_ik_device(poses, None, branches)
            return eng, branches[:, b].contiguous()
        return self._ikine_pose(dest_poses, seed, weights, damping, tol, max_iter if refine else 0, as_array,
                                return_iterations, return_fk_error)

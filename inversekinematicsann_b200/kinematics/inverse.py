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
        """Upload the poses once, seed with `seed_on_device(xyz) -> (engine, float64 seeds)` on the position columns,
        raise what `ikine` raises, refine onto the poses in place and download once."""
        import torch
        poses = poses_to_array(dest_poses)
        n = poses.shape[0]
        if n == 0:
            return _empty_result(np.float64, as_array, return_iterations, return_fk_error)
        eng = self._engine()
        d_poses = torch.from_numpy(poses).to(torch.device("cuda", eng.device))
        solver, seed = seed_on_device(d_poses[:, :3, 3].contiguous())
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

        def seed(xyz):
            eng = self._engine()
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

        def seed(xyz):
            eng = self.ann._ensure_uploaded()
            pred = torch.empty((xyz.shape[0], 4), dtype=torch.float32, device=xyz.device)
            eng.stats_reset_torch()
            eng.ann_solve_device(xyz, pred, mode=self.ann.mode)
            return eng, pred.double()
        return self._ikine_pose(dest_poses, seed, weights, damping, tol, max_iter, as_array, return_iterations,
                                return_fk_error)

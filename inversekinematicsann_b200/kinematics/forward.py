"""DH forward kinematics -- API of reference kinematics/forward.py, computed by csrc/fk.cu.

``ForwardKinematics(dh_matrix).fkine(angles)`` returns ``(T_final, [T_1 .. T_4])`` as 4x4 NumPy
arrays exactly like the reference (forward.py:73-94); callers read the position as T[0:3, 3]
(cli.py:60, inverse.py:130).  ``fkine_positions`` is the batched form used for the
position-error check of both solvers.  ``fkine_batch`` is ``fkine`` for n angle sets, ``joint_positions`` gives
the joint origins of every set, and ``fkine_device`` keeps inputs and outputs in GPU memory.  ``jacobian``,
``jacobian_batch``, ``manipulability`` and ``jacobian_device`` give how the effector moves when the joints turn.
"""
import numpy as np

from ..robot.robot import OutOfRobotReachException
from ._shared import get_engine

_ANGLE_MSG = 'Forward Kinematics exception, robot joints angles limits are (-2pi, 2pi)'  # forward.py:24-25


class ForwardKinematics:
    """Planar robotic arm forward kinematics"""

    def __init__(self, dh_matrix, device=None):
        assert all(len(row) == len(dh_matrix[0]) for row in dh_matrix)
        self.dh_matrix = dh_matrix
        self.thetas, self.epsilons, self.ais, self.alphas = self.dh_matrix
        self.no_of_features = len(self.thetas)
        assert self.no_of_features >= 3
        if self.no_of_features != 4:
            # upstream's matrices are no_of_features x no_of_features and only work as homogeneous
            # transforms for 4 joints (SURVEY 3.4); the engine is built for exactly that case
            raise ValueError('the DH table must describe 4 joints')
        self._device = device

    def _engine(self):
        return get_engine(dh_matrix=self.dh_matrix, device=self._device)

    def fkine(self, angles):
        """All cumulative DH transforms for one set of joint angles -> (T_4, [T_1, T_2, T_3, T_4])."""
        self.thetas = angles  # upstream side effect (forward.py:77)
        chain, status = self._engine().fk_chain(angles)
        if status != 0:
            raise OutOfRobotReachException(_ANGLE_MSG)
        mats = [np.array(chain[i]) for i in range(4)]
        return mats[-1], mats

    def fkine_batch(self, angles):
        """fkine for (n, 4) angles -> (T[n,4,4], chain[n,4,4,4]) in the angles' dtype; T is a view of chain[:, 3]."""
        chain, stats = self._engine().fk_transforms(angles, "matrices")
        if stats.first_fk_angle_range >= 0:
            raise OutOfRobotReachException(_ANGLE_MSG)
        return chain[:, 3], chain

    def joint_positions(self, angles):
        """The four joint origins (column 3 of T_1..T_4) for (n, 4) angles -> (n, 4, 3) in the angles' dtype."""
        joints, stats = self._engine().fk_transforms(angles, "joints")
        if stats.first_fk_angle_range >= 0:
            raise OutOfRobotReachException(_ANGLE_MSG)
        return joints

    def fkine_device(self, angles, out=None, what="matrices"):
        """fkine_batch (what="matrices": out (n,4,4,4)) or joint_positions (what="joints": out (n,4,3)) on a CUDA
        tensor, enqueued on torch's current stream without a synchronisation; out is allocated when None.  An angle
        outside [-2pi, 2pi] sets first_fk_angle_range of the engine's statistics (``stats_fetch_torch``)."""
        import torch
        eng = self._engine()
        if out is None:
            tail = (4, 4, 4) if what == "matrices" else (4, 3)
            out = torch.empty((angles.shape[0],) + tail, dtype=angles.dtype, device=angles.device)
        eng.fk_transforms_device(angles, out, what)
        return out

    def fkine_positions(self, angles, targets=None):
        """Batched end-effector positions for (n, 4) angles; with `targets` also ||pos - target||."""
        pos, err, stats = self._engine().fk(angles, targets)
        if stats.first_fk_angle_range >= 0:
            raise OutOfRobotReachException(_ANGLE_MSG)
        return (pos, err) if targets is not None else pos

    def jacobian(self, angles):
        """The (6, 4) fp64 geometric Jacobian of one set of joint angles: rows 0-2 the linear part
        z_{i-1} x (p_4 - p_{i-1}), rows 3-5 the joint axis z_{i-1}, column i-1 for joint i.  The batch kernel at n = 1."""
        return self.jacobian_batch(np.asarray(angles, dtype=np.float64).reshape(1, 4))[0]

    def jacobian_batch(self, angles, what="geometric"):
        """jacobian for (n, 4) angles -> (n, 6, 4) (what="geometric") or the position rows only, (n, 3, 4)
        (what="position"), in the angles' dtype."""
        jac, _, stats = self._engine().jacobian(angles, what)
        if stats.first_fk_angle_range >= 0:
            raise OutOfRobotReachException(_ANGLE_MSG)
        return jac

    def manipulability(self, angles):
        """Yoshikawa manipulability sqrt(det(Jv Jv^T)) of the 3 x 4 position Jacobian for (n, 4) angles -> (n,) in the
        angles' dtype: 0 at a singular pose, such as the stretched arm."""
        _, w, stats = self._engine().jacobian(angles, None, manipulability=True)
        if stats.first_fk_angle_range >= 0:
            raise OutOfRobotReachException(_ANGLE_MSG)
        return w

    def jacobian_device(self, angles, out=None, what="geometric", manip_out=None):
        """jacobian_batch on a CUDA tensor, enqueued on torch's current stream without a synchronisation: out (n,6,4)
        or (n,3,4) by `what`, allocated when None (what=None: no Jacobian, out stays None); manip_out (n,), when given,
        receives the manipulability.  Returns out.  An angle outside [-2pi, 2pi] sets first_fk_angle_range of the
        engine's statistics (``stats_fetch_torch``)."""
        import torch
        eng = self._engine()
        if out is None and what is not None:
            tail = (6, 4) if what == "geometric" else (3, 4)
            out = torch.empty((angles.shape[0],) + tail, dtype=angles.dtype, device=angles.device)
        eng.jacobian_device(angles, out, what if what is not None else "geometric", manip_out)
        return out

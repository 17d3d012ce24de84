"""FABRIK solver -- API of reference kinematics/fabrik.py, computed by csrc/fabrik_chain.cu.

``Fabrik(joints_distances, err_margin, max_iter_num).calculate(init_positions, goal)`` keeps the
reference's signature and return type (fabrik.py:13,44-67: a list of ``Point``, one per joint) for
chains of any length J = len(joints_distances), 1..256.  The chain is solved on the GPU by the
chain kernel, which follows the reference's operation order in IEEE fp64; ``calculate_batch``
solves many goals in one call and ``calculate_device`` keeps inputs and outputs in GPU memory.
"""
import numpy as np

from .._native import IKB_CHAIN_MAX_POINTS
from ._shared import get_engine
from .point import Point


class Fabrik:
    """Forward And Backward Reaching Inverse Kinematics on a chain of len(joints_distances) points."""

    def __init__(self, joints_distances, err_margin=0.001, max_iter_num=100, device=None):
        self.joints_distances = joints_distances
        self.err_margin = err_margin
        self.max_iter_num = max_iter_num
        self._device = device

    def _engine(self):
        # link lengths, tolerance and iteration cap are arguments of every call: any engine of the device serves
        return get_engine(device=self._device)

    def _check_len(self, n_points):
        if n_points != len(self.joints_distances):
            raise ValueError('Input vectors should have equal lengths!')  # fabrik.py:46-48
        if not 1 <= n_points <= IKB_CHAIN_MAX_POINTS:
            raise ValueError(f'a chain needs 1..{IKB_CHAIN_MAX_POINTS} joints, got {n_points}')

    def calculate_batch(self, init_joints_positions, goal_effector_positions):
        """(J,3) or (n,J,3) initial chains, (n,3) goals -> (chains[n,J,3], iterations[n])."""
        init = np.asarray(init_joints_positions, dtype=np.float64)
        if init.ndim not in (2, 3) or init.shape[-1] != 3:
            raise ValueError(f'initial chains must have shape (J, 3) or (n, J, 3), got {init.shape}')
        self._check_len(init.shape[-2])
        chains, iters, stats = self._engine().fabrik_chain(self.joints_distances, self.err_margin, self.max_iter_num,
                                                           init, goal_effector_positions)
        if stats.first_zero_division >= 0:
            raise ZeroDivisionError('float division by zero')  # point.py:40 upstream
        return chains, iters

    def calculate(self, init_joints_positions, goal_effector_position):
        """Joint positions after FABRIK from `init_joints_positions` to the goal (fabrik.py:44-67)."""
        self._check_len(len(init_joints_positions))
        goal = Point(goal_effector_position)
        chains, _ = self.calculate_batch([list(p) for p in init_joints_positions], [list(goal)])
        return [Point(row.tolist()) for row in chains[0]]

    def calculate_device(self, init, goals, out=None, iters=None):
        """calculate_batch on float64 CUDA tensors, enqueued on torch's current stream without a synchronisation:
        init (J,3) or (n,J,3), goals (n,3) -> out (n,J,3) (allocated when None).  A zero-length segment leaves a
        non-finite chain and sets first_zero_division of the engine's statistics (``stats_fetch_torch``)."""
        import torch
        eng = self._engine()
        if init.dim() not in (2, 3):
            raise ValueError(f'initial chains must have shape (J, 3) or (n, J, 3), got {tuple(init.shape)}')
        self._check_len(init.shape[-2])
        if out is None:
            out = torch.empty((goals.shape[0], len(self.joints_distances), 3), dtype=torch.float64,
                              device=goals.device)
        eng.fabrik_chain_device(self.joints_distances, self.err_margin, self.max_iter_num, init, goals, out, iters)
        return out

"""bench.py --dump-outputs: what the last timed step computed, on inputs that are the same in every run, so that two
builds of the project can be compared output for output."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import conftest as C

BENCH = os.path.join(C.ROOT, "bench.py")


def test_dump_rows_are_a_fixed_sample():
    import bench
    np.testing.assert_array_equal(bench.dump_rows(10), np.arange(10))
    a, b = bench.dump_rows(10**8), bench.dump_rows(10**8)
    assert a.shape == (bench.DUMP_ROWS,) and np.array_equal(a, b)
    assert np.all(np.diff(a) > 0) and a[-1] < 10**8
    assert 2 * (bench.DUMP_ROWS * 4 * 4 + 128) <= 64 * 10**6   # both float32 [*, 4] .npy files stay within 64 MB


def test_steps_must_be_positive():
    p = subprocess.run([sys.executable, BENCH, "--steps", "0"], capture_output=True, text=True)
    assert p.returncode == 2 and "--steps" in p.stderr


@pytest.mark.gpu
def test_dump_outputs_hold_what_the_timed_path_computed(tmp_path):
    rows, ann_rows = 70_000, 4096
    p = subprocess.run([sys.executable, BENCH, "--steps", "2", "--warmup", "3", "--rows", str(rows),
                        "--ann-rows", str(ann_rows), "--ann-big-rows", "0", "--skip-cpu", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-4000:]
    line = json.loads([l for l in p.stdout.splitlines() if l.startswith("{")][-1])
    assert line["steps"] == 2
    fab, ann = np.load(tmp_path / "fabrik_angles.npy"), np.load(tmp_path / "ann_angles.npy")
    assert fab.dtype == np.float32 and fab.shape == (rows, 4)
    assert ann.dtype == np.float32 and ann.shape == (ann_rows, 4) and np.isfinite(ann).all()
    # the same solve in this process, on the bench's rank-0 input (device generator, seed 1234)
    import torch
    from inversekinematicsann_b200.kinematics.inverse import FabrikInverseKinematics
    from inversekinematicsann_b200.robot.position_generator import TrainingDataGenerator as Gen
    from inversekinematicsann_b200.robot.robot import SixDOFRobot as R
    xyz = Gen.cube_random_device(648.0 / rows, 6.0, 12.0, 9.0, start=(0.0, -6.0, -3.0), seed=1234,
                                 no_of_samples=rows, device=0)
    ik = FabrikInverseKinematics(R.dh_matrix, R.links_lengths, R.effector_workspace_limits, device=0)
    angles = torch.empty(rows, 4, device=xyz.device, dtype=torch.float32)
    ik._engine().fabrik_solve_device(xyz, angles)
    np.testing.assert_array_equal(fab, angles.cpu().numpy())
    # the ANN dump is the default mode's output for the bench's ANN input (seed 4321) and model
    from inversekinematicsann_b200.kinematics.inverse import AnnInverseKinematics
    ann_ik = AnnInverseKinematics(R.dh_matrix, R.links_lengths, R.effector_workspace_limits, device=0)
    ann_ik.load_model(os.path.join(C.ROOT, "models", "roboarm_b200_r01.h5"))
    axyz = Gen.random_distribution_device(ann_rows, R.effector_workspace_limits, 'normal', 0.5, seed=4321, device=0)
    aout = torch.empty(ann_rows, 4, device=axyz.device, dtype=torch.float32)
    ann_ik.ann._ensure_uploaded().ann_solve_device(axyz, aout, mode="fp16x3_ts")
    np.testing.assert_array_equal(ann, aout.cpu().numpy())

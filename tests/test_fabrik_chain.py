"""Fabrik.calculate on chains of J = 1..256 points (csrc/fabrik_chain.cu).

CPU: a literal Python transcription of the reference's point.py / fabrik.py loops equals the C restatement in
tests/chain_oracle.c bit for bit, and that restatement equals the pinned 4-point oracle at J = 4.
GPU: the chain kernel equals the C restatement bit for bit (chains, iteration counts, statistics) on both sides of the
register / local-memory split, whatever the row order, chunking or entry point."""
import ctypes
import math
import os
import subprocess

import numpy as np
import pytest

import conftest as C

HERE = os.path.dirname(os.path.abspath(__file__))
J_GPU = [1, 2, 3, 4, 5, 6, 8, 12, 16, 24, 32, 33, 64, 256]


# ---- the C restatement ---------------------------------------------------------------------------------------------
@pytest.fixture(scope="session")
def chain_lib(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("chain_oracle") / "libchain_oracle.so")
    subprocess.run(["gcc", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math", "-o", so,
                    os.path.join(HERE, "chain_oracle.c"), "-lm"], check=True, capture_output=True)
    lib = ctypes.CDLL(so)
    vp = ctypes.c_void_p
    lib.ico_fabrik_chain.restype = ctypes.c_int64
    lib.ico_fabrik_chain.argtypes = [ctypes.c_int, vp, ctypes.c_double, ctypes.c_int, vp, ctypes.c_int64, vp,
                                     ctypes.c_int64, vp, vp, ctypes.POINTER(ctypes.c_int64)]
    return lib


def oracle_chain(lib, links, tol, max_iter, init, goals):
    """-> (chains[n,J,3], iters[n], n_iter_capped, first_zero_division)"""
    links = np.ascontiguousarray(links, dtype=np.float64)
    J = links.shape[0]
    init = np.ascontiguousarray(init, dtype=np.float64)
    goals = np.ascontiguousarray(goals, dtype=np.float64).reshape(-1, 3)
    n = goals.shape[0]
    n_init = 1 if init.ndim == 2 else init.shape[0]
    out = np.empty((n, J, 3))
    iters = np.empty(n, dtype=np.int32)
    first = ctypes.c_int64(-1)
    capped = lib.ico_fabrik_chain(J, links.ctypes.data, float(tol), int(max_iter), init.ctypes.data, n_init,
                                  goals.ctypes.data, n, out.ctypes.data, iters.ctypes.data, ctypes.byref(first))
    return out, iters, int(capped), int(first.value)


# ---- a literal transcription of the reference (point.py:25-45, fabrik.py:19-67) ---------------------------------
class _P:
    def __init__(self, xyz):
        self.x, self.y, self.z = xyz

    def __iter__(self):
        return iter((self.x, self.y, self.z))


def _distance(a, b):
    # the reference squares with `** 2`, which goes through the C library's pow(): not always correctly rounded (about
    # 1 square in 1200 of standard-normal values differs from x * x in the last bit with glibc).  Every restatement
    # here -- the pinned oracle, the chain oracle, the kernels -- uses the correctly rounded product.
    dx, dy, dz = a.x - b.x, a.y - b.y, a.z - b.z
    return math.sqrt(dx * dx + dy * dy + dz * dz)


def _between(start, end, distance):
    ratio = distance / _distance(start, end)
    return _P([s + ratio * (e - s) for s, e in zip(start, end)])


def py_calculate(joints_distances, err_margin, max_iter_num, init, goal):
    def backward(points, goal):
        positions = [goal]
        for p, d in zip(reversed(points[:-1]), reversed(joints_distances[:-1])):
            positions.insert(0, _between(positions[0], p, d))
        return positions

    def forward(points, start):
        positions = [start]
        for p, d in zip(points[1:], joints_distances[1:]):
            positions.append(_between(positions[-1], p, d))
        return positions

    current = [_P(p) for p in init]
    goal = _P(goal)
    start = current[0]
    start_error, goal_error, step = 1, 1, 0
    while (start_error > err_margin or goal_error > err_margin) and max_iter_num > step:
        b = backward(current, goal)
        start_error = _distance(b[0], start)
        current = forward(b, start)
        goal_error = _distance(current[-1], goal)
        step += 1
    return np.array([list(p) for p in current]), step


def random_case(rng, J, n, per_row, unit=False, radius=1.25):
    """Links, initial chains (per row or one straight chain) and goals uniform in a ball of radius * reach about S."""
    links = np.ones(J) if unit else rng.uniform(0.5, 2.0, J)
    reach = float(links[1:].sum()) if J > 1 else 1.0
    if per_row:
        init = rng.standard_normal((n, J, 3)).cumsum(axis=1)
        S = init[:, 0]
    else:
        init = np.zeros((J, 3))
        init[:, 2] = np.concatenate([[0.0], np.cumsum(links[1:])])
        S = np.zeros((n, 3))
    u = rng.standard_normal((n, 3))
    u /= np.linalg.norm(u, axis=1, keepdims=True)
    goals = S + u * (reach * radius * rng.uniform(0, 1, (n, 1)) ** (1 / 3))
    return links, init, goals


# ---- CPU ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("J", [1, 2, 3, 4, 5, 6, 8, 13])
def test_python_transcription_equals_chain_oracle(chain_lib, J):
    rng = np.random.default_rng(100 + J)
    for per_row in (False, True):
        links, init, goals = random_case(rng, J, 6, per_row, radius=1.4)  # reachable and unreachable goals
        for tol in (1e-3, 0.0):
            for max_iter in (0, 1, 100):
                got, iters, _, first = oracle_chain(chain_lib, links, tol, max_iter, init, goals)
                assert first == -1
                for r in range(goals.shape[0]):
                    want, k = py_calculate(list(links), tol, max_iter, init[r] if per_row else init, goals[r])
                    assert k == iters[r]
                    assert np.array_equal(got[r], want), (J, per_row, tol, max_iter, r)


def test_chain_oracle_at_four_points_equals_the_pinned_oracle(chain_lib):
    from oracle import c_oracle
    rng = np.random.default_rng(7)
    links, init, goals = random_case(rng, 4, 40, True, radius=1.3)
    for tol, max_iter in ((1e-3, 100), (0.0, 7), (1e-3, 0)):
        got, iters, _, _ = oracle_chain(chain_lib, links, tol, max_iter, init, goals)
        for r in range(goals.shape[0]):
            st, want, k = c_oracle.fabrik_calculate(init[r], goals[r], links=links, tol=tol, max_iter=max_iter)
            assert st == 0 and k == iters[r] and np.array_equal(got[r], want)


def test_argument_validation_without_gpu():
    from inversekinematicsann_b200 import _native
    from inversekinematicsann_b200.engine import IkEngine
    from inversekinematicsann_b200.kinematics.fabrik import Fabrik
    with pytest.raises(ValueError, match="Input vectors should have equal lengths!"):
        Fabrik([1.0] * 5).calculate([[0, 0, 0]] * 4, [1, 2, 3])
    with pytest.raises(ValueError, match="Input vectors should have equal lengths!"):
        Fabrik([1.0] * 5).calculate_batch(np.zeros((3, 6, 3)), np.zeros((3, 3)))
    with pytest.raises(ValueError):
        Fabrik([]).calculate([], [1, 2, 3])
    with pytest.raises(ValueError):
        Fabrik([1.0] * 257).calculate([[0, 0, 0]] * 257, [1, 2, 3])
    for bad in ([], [1.0] * 257, [[1.0, 2.0]]):
        with pytest.raises(ValueError):
            IkEngine._chain_links(bad)
    assert IkEngine._chain_links([1, 2]).dtype == np.float64
    lib = _native.load()
    buf = np.zeros(3)
    for fn in (lib.ikb_fabrik_chain_host, lib.ikb_fabrik_chain_device):
        assert fn(None, 4, buf.ctypes.data, 1e-3, 100, buf.ctypes.data, 1, buf.ctypes.data, 1, buf.ctypes.data,
                  None, None) == _native.IKB_ERR_INVALID


@pytest.mark.reference
def test_live_reference_fabrik_on_other_lengths(chain_lib):
    """The reference's Fabrik itself on J = 2, 3, 6: its loops take any length (fabrik.py:19-42)."""
    from oracle import ref_import
    if not ref_import.available():
        pytest.skip("reference tree not present")
    ref = ref_import.load()
    rng = np.random.default_rng(3)
    for J in (2, 3, 6):
        links, init, goals = random_case(rng, J, 5, True)
        got, iters, _, _ = oracle_chain(chain_lib, links, 1e-3, 100, init, goals)
        for r in range(goals.shape[0]):
            f = ref.fabrik.Fabrik(list(links), 1e-3, 100)
            pts = f.calculate([ref.point.Point(list(p)) for p in init[r]], ref.point.Point(list(goals[r])))
            assert np.array_equal(np.array([[p.x, p.y, p.z] for p in pts]), got[r])


# ---- GPU ------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def eng():
    from inversekinematicsann_b200.kinematics._shared import get_engine
    return get_engine()


def _rows_for(J):
    return 4000 if J <= 8 else (1500 if J <= 33 else 300)


@pytest.mark.gpu
@pytest.mark.parametrize("J", J_GPU)
@pytest.mark.parametrize("per_row", [False, True], ids=["n_init1", "n_init_n"])
def test_gpu_bit_exact(eng, chain_lib, J, per_row):
    rng = np.random.default_rng(J * 7 + per_row)
    n = _rows_for(J)
    links, init, goals = random_case(rng, J, n, per_row)
    if J > 1:  # goals within +-1e-3 of full reach
        S = init[:, 0] if per_row else np.zeros((n, 3))
        u = rng.standard_normal((n // 4, 3))
        u /= np.linalg.norm(u, axis=1, keepdims=True)
        goals[: n // 4] = S[: n // 4] + u * (links[1:].sum() + rng.uniform(-1e-3, 1e-3, (n // 4, 1)))
    want, want_it, want_capped, _ = oracle_chain(chain_lib, links, 1e-3, 100, init, goals)
    got, it, st = eng.fabrik_chain(links, 1e-3, 100, init, goals)
    np.testing.assert_array_equal(got, want)
    np.testing.assert_array_equal(it, want_it)
    assert st.n_solved == n and st.sum_iterations == int(want_it.sum())
    assert st.n_iter_capped == want_capped and st.first_zero_division == -1


@pytest.mark.gpu
@pytest.mark.parametrize("n", [0, 1, 31, 33, 1000])
@pytest.mark.parametrize("J", [4, 40])
def test_gpu_row_permutation(eng, J, n):
    rng = np.random.default_rng(n + J)
    links, init, goals = random_case(rng, J, n, True)
    a, ia, sa = eng.fabrik_chain(links, 0.0 if n % 2 else 1e-3, 50, init, goals)
    perm = rng.permutation(n)
    b, ib, sb = eng.fabrik_chain(links, 0.0 if n % 2 else 1e-3, 50, init[perm], goals[perm])
    assert a.shape == (n, J, 3)
    np.testing.assert_array_equal(b, a[perm])
    np.testing.assert_array_equal(ib, ia[perm])
    assert (sa.n_solved, sa.sum_iterations, sa.n_iter_capped) == (sb.n_solved, sb.sum_iterations, sb.n_iter_capped)


@pytest.mark.gpu
@pytest.mark.parametrize("tol,max_iter", [(0.0, 3), (1e-3, 0), (1.0, 100)])
def test_gpu_tolerance_and_cap_edges(eng, chain_lib, tol, max_iter):
    rng = np.random.default_rng(11)
    links, init, goals = random_case(rng, 6, 3000, True)
    want, want_it, _, _ = oracle_chain(chain_lib, links, tol, max_iter, init, goals)
    got, it, _ = eng.fabrik_chain(links, tol, max_iter, init, goals)
    np.testing.assert_array_equal(got, want)
    np.testing.assert_array_equal(it, want_it)
    if max_iter == 0 or tol >= 1.0:
        np.testing.assert_array_equal(got, init)


def _big_case(rng, J=256, n=50_000):
    # > 1 host chunk: a chunk holds 4 * 2^22 / (3 J) rows of the slot buffers (21 845 at J = 256)
    return random_case(rng, J, n, True)


@pytest.mark.gpu
def test_gpu_zero_division_lowest_global_row(eng, chain_lib):
    from inversekinematicsann_b200.kinematics.fabrik import Fabrik
    rng = np.random.default_rng(5)
    links, init, goals = _big_case(rng)
    for r in (45_000, 30_001):  # the goal on P[J-2]: the first backward step divides by 0
        goals[r] = init[r, -2]
    want, want_it, _, first = oracle_chain(chain_lib, links, 0.0, 3, init, goals)
    got, it, st = eng.fabrik_chain(links, 0.0, 3, init, goals)
    assert first == 30_001 and st.first_zero_division == 30_001
    np.testing.assert_array_equal(got, want)
    np.testing.assert_array_equal(it, want_it)
    assert not np.isfinite(got[30_001, 1:]).all() and np.isfinite(got[:30_001]).all()
    f = Fabrik(list(links), 0.0, 3)
    with pytest.raises(ZeroDivisionError, match="float division by zero"):
        f.calculate(init[30_001].tolist(), goals[30_001].tolist())


@pytest.mark.gpu
def test_gpu_host_chunks_equal_device_path_on_a_side_stream(eng, chain_lib):
    import torch
    rng = np.random.default_rng(6)
    links, init, goals = _big_case(rng)
    host, it_h, st_h = eng.fabrik_chain(links, 0.0, 3, init, goals)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        d_init = torch.from_numpy(init).cuda()
        d_goals = torch.from_numpy(goals).cuda()
        out = torch.empty((goals.shape[0], 256, 3), dtype=torch.float64, device="cuda")
        iters = torch.empty(goals.shape[0], dtype=torch.int32, device="cuda")
        eng.stats_reset_torch()
        eng.fabrik_chain_device(links, 0.0, 3, d_init, d_goals, out, iters)
        st_d = eng.stats_fetch_torch()
    s.synchronize()
    np.testing.assert_array_equal(out.cpu().numpy(), host)
    np.testing.assert_array_equal(iters.cpu().numpy(), it_h)
    assert (st_d.n_solved, st_d.sum_iterations, st_d.n_iter_capped) == (st_h.n_solved, st_h.sum_iterations,
                                                                         st_h.n_iter_capped)
    want, _, _, _ = oracle_chain(chain_lib, links, 0.0, 3, init[:500], goals[:500])
    np.testing.assert_array_equal(host[:500], want)


@pytest.mark.gpu
def test_gpu_fabrik_six_points(chain_lib):
    from inversekinematicsann_b200.kinematics.fabrik import Fabrik
    from inversekinematicsann_b200.kinematics.point import Point
    init = [[0.0, 0.0, 1.5 * j] for j in range(6)]
    got = Fabrik([1.5] * 6).calculate(init, [2.0, 1.0, 4.0])
    assert len(got) == 6 and all(isinstance(p, Point) for p in got)
    want, _, _, _ = oracle_chain(chain_lib, [1.5] * 6, 1e-3, 100, np.array(init), [2.0, 1.0, 4.0])
    np.testing.assert_array_equal(np.array(got), want[0])
    # batch and device forms
    import torch
    f = Fabrik([1.5] * 6)
    goals = np.array([[2.0, 1.0, 4.0], [0.5, -1.0, 3.0]])
    chains, _ = f.calculate_batch(init, goals)
    np.testing.assert_array_equal(chains[0], want[0])
    dev = f.calculate_device(torch.tensor(init, dtype=torch.float64, device="cuda"),
                             torch.tensor(goals, device="cuda"))
    np.testing.assert_array_equal(dev.cpu().numpy(), chains)


@pytest.mark.gpu
def test_gpu_four_point_wrapper_equals_chain(eng):
    from inversekinematicsann_b200.robot.robot import SixDOFRobot
    rng = np.random.default_rng(9)
    _, init, goals = random_case(rng, 4, 2000, True)
    a, ia, sa = eng.fabrik_calculate(init, goals)
    b, ib, sb = eng.fabrik_chain(SixDOFRobot.links_lengths, 1e-3, 100, init, goals)  # the engine's configuration
    np.testing.assert_array_equal(a, b)
    np.testing.assert_array_equal(ia, ib)
    assert (sa.n_solved, sa.sum_iterations, sa.n_iter_capped) == (sb.n_solved, sb.sum_iterations, sb.n_iter_capped)


@pytest.mark.gpu
def test_gpu_device_arguments_rejected_before_launch(eng):
    import torch
    J, n = 5, 8
    links = np.ones(J)
    ok = dict(init=torch.zeros(J, 3, dtype=torch.float64, device="cuda"),
              goals=torch.zeros(n, 3, dtype=torch.float64, device="cuda"),
              out=torch.empty(n, J, 3, dtype=torch.float64, device="cuda"))
    bad = [(TypeError, "goals", torch.zeros(n, 3, dtype=torch.float64)),            # host tensor
           (ValueError, "goals", torch.zeros(n, 3, dtype=torch.float32, device="cuda")),
           (ValueError, "init", torch.zeros(J + 1, 3, dtype=torch.float64, device="cuda")),
           (ValueError, "init", torch.zeros(J, 3, dtype=torch.float32, device="cuda")),
           (ValueError, "out", torch.empty(n, J, 4, dtype=torch.float64, device="cuda")),
           (ValueError, "out", torch.empty(J, n, 3, dtype=torch.float64, device="cuda").transpose(0, 1)),
           (TypeError, "init", np.zeros((J, 3)))]
    before = eng.launch_count
    for exc, name, value in bad:
        kw = dict(ok, **{name: value})
        with pytest.raises(exc):
            eng.fabrik_chain_device(links, 1e-3, 100, kw["init"], kw["goals"], kw["out"])
    with pytest.raises(ValueError):
        eng.fabrik_chain_device(np.ones(300), 1e-3, 100, ok["init"], ok["goals"], ok["out"])
    with pytest.raises(ValueError):
        eng.fabrik_chain_device(links, 1e-3, 100, ok["init"], ok["goals"], ok["out"],
                                torch.empty(n, dtype=torch.int64, device="cuda"))
    with pytest.raises(ValueError):
        eng.fabrik_chain(links, 1e-3, 100, np.zeros((3, J, 3)), np.zeros((n, 3)))
    assert eng.launch_count == before

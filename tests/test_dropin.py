"""The zero-edit drop-in (INTEGRATION.md section 1): the reference's own callers on top of dropin/.

CPU: with dropin/ ahead of the reference tree every `kinematics.*` / `robot.*` import of cli.py, rpc_broker.py and
the reference's tests resolves to the shims while the reference's own `tests`, `plot`, `cli`, `rpc_broker` stay its
own, and `cli.CLI()` constructs.  GPU: the reference's unit suites, cli.py and the broker callback run unmodified
(tools/run_reference_suite.py).  Both run the reference's own code, which is not part of this repository, so they need
a checkout of it (IK_REFERENCE_ROOT, or a .refscratch/ copy in the repository root) and skip without one; the log of
one such run is profiles/r02_dropin_suite.log.  test_plain_pythonpath_is_not_enough needs only the reference's package
layout and builds a stand-in tree for it."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _reference_root():
    for cand in (os.environ.get("IK_REFERENCE_ROOT", ""), "/root/reference", os.path.join(ROOT, ".refscratch")):
        if cand and os.path.isfile(os.path.join(cand, "cli.py")):
            return cand
    return None


def _run(stage):
    ref = _reference_root()
    if ref is None:
        pytest.skip("no checkout of the reference available")
    env = dict(os.environ, IK_REFERENCE_ROOT=ref)
    p = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "run_reference_suite.py"), "--stage", stage],
                       env=env, capture_output=True, text=True, timeout=900)
    assert p.returncode == 0 and "ALL GREEN" in p.stdout, p.stdout[-4000:] + p.stderr[-2000:]
    return p.stdout


def test_reference_imports_resolve_to_the_dropin():
    out = _run("resolve")
    assert "ok  kinematics.inverse" in out and "ok  cli" in out and "LAUNCH" in out


def test_plain_pythonpath_is_not_enough(tmp_path):
    """Why INTEGRATION.md prescribes the launcher (or PYTHONSAFEPATH): `python cli.py` puts the script directory at
    sys.path[0], ahead of PYTHONPATH, so the reference's own packages would win.  Only the reference's package layout
    matters here, so a stand-in tree with its `kinematics` package and a `cli.py` takes its place."""
    ref = str(tmp_path)
    os.makedirs(os.path.join(ref, "kinematics"))
    for name in ("cli.py", os.path.join("kinematics", "__init__.py"), os.path.join("kinematics", "point.py")):
        open(os.path.join(ref, name), "w").close()
    env = dict(os.environ, PYTHONPATH=os.path.join(ROOT, "dropin"), PYTHONDONTWRITEBYTECODE="1")
    env.pop("PYTHONSAFEPATH", None)
    probe = "import sys; sys.path.insert(0, sys.argv[1]); import kinematics.point as m; print(m.__file__)"
    # emulate `python <ref>/script.py`: the script directory goes to sys.path[0]
    p = subprocess.run([sys.executable, "-c", probe, ref], env=env, capture_output=True, text=True, cwd=ref)
    assert os.path.realpath(p.stdout.strip()).startswith(os.path.realpath(ref))


@pytest.mark.gpu
def test_reference_suites_cli_and_broker_run_on_the_engine():
    out = _run("suites,cli,broker")
    assert "SUITE inverse_fabrik: run=1 failures=0 errors=0" in out

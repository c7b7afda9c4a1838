"""``gossipy_b200.compat``: experiment scripts written for the reference (``from gossipy ...``) run UNMODIFIED on this
framework."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# scripts written against the original gossipy's API; GOSSIPY_REFERENCE=<checkout of the original> runs its own instead
SCRIPTS = os.environ.get("GOSSIPY_REFERENCE") or os.path.join(ROOT, "tests", "compat_scripts")


def _run(args, timeout=900):
    env = dict(os.environ, OMP_NUM_THREADS="2", PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""))
    out = subprocess.run([sys.executable, "-m", "gossipy_b200.compat"] + args, capture_output=True, text=True,
                         timeout=timeout, env=env, cwd=ROOT)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-3000:]
    return out.stdout + out.stderr


def test_install_aliases_every_module_of_the_reference_layout():
    code = ("import gossipy_b200.compat as c; c.install(); "
            "import gossipy, gossipy.core, gossipy.node, gossipy.simul, gossipy.flow_control, gossipy.utils, gossipy.data, "
            "gossipy.data.handler, gossipy.model, gossipy.model.handler, gossipy.model.nn, gossipy.model.sampling; "
            "from gossipy.simul import GossipSimulator; import gossipy_b200.simul as s; assert GossipSimulator is s.GossipSimulator; "
            "from gossipy import set_seed, GlobalSettings, CACHE; "
            "c.uninstall(); import sys; assert 'gossipy' not in sys.modules; print('ok')")
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=ROOT, timeout=300)
    assert out.returncode == 0 and "ok" in out.stdout, out.stderr[-2000:]


@pytest.mark.parametrize("script,extra", [
    ("main_hegedus_2021.py", []),                                       # tokenized, partitioned models, Python loop
    ("main_hegedus_2021.py", ["--engine", "native", "--native-utility", "1"]),   # same script on the C++ scheduler + executor
    ("main_ormandi_2013.py", ["--engine", "native"]),                   # 1 617 Pegasos nodes: the banked engine
    ("main_all2all.py", []),
])
def test_reference_scripts_run_unmodified(script, extra):
    out = _run(["--synthetic", "--max-rounds", "2"] + extra + [os.path.join(SCRIPTS, script)])
    assert "Sent messages" in out and "accuracy" in out

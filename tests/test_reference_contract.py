"""The reference's own tests of the path as the drop-in contract (SURVEY section 4 item 1): tests/test_denovo3D_solver.py
and tests/test_denovo3D_pipeline.py of jianglab/helicon, UNMODIFIED (copied by oracle/build_ref.py into the git-ignored
oracle/_ref/reference_tests/, they travel to the GPU box with the snapshot), run in a subprocess with helicon_b200 mounted
at ``helicon.webApps.denovo3D.*`` (tests/alias_plugin.py)."""
import os
import subprocess
import sys

import pytest

from tests.helpers import ROOT

REF_TESTS = os.path.join(ROOT, "oracle", "_ref", "reference_tests")


def test_alias_plugin_mounts_the_module_paths():
    code = ("import tests.alias_plugin, helicon.webApps.denovo3D.solver_linear_regression as s, helicon_b200."
            "solver_linear_regression as g, helicon; assert s is g and callable(helicon.get_cylindrical_mask); print('ok')")
    out = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True)
    assert out.returncode == 0 and "ok" in out.stdout, out.stderr[-2000:]


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["test_denovo3D_solver.py", "test_denovo3D_pipeline.py"])
def test_reference_test_file_passes_against_helicon_b200(name):
    path = os.path.join(REF_TESTS, name)
    if not os.path.isfile(path):
        pytest.skip("oracle/_ref/reference_tests absent: copy tests/test_denovo3D_solver.py and "
                    "tests/test_denovo3D_pipeline.py of jianglab/helicon there (oracle/build_ref.py does it from a checkout)")
    out = subprocess.run([sys.executable, "-m", "pytest", "-q", "-x", "-p", "tests.alias_plugin", "-p", "no:cacheprovider",
                          "--rootdir", REF_TESTS, path], cwd=ROOT, capture_output=True, text=True, timeout=1500)
    tail = out.stdout[-3000:] + out.stderr[-1500:]
    print(tail)
    assert out.returncode == 0, tail

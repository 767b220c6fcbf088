"""Where a checkout of the reference is at hand ($PGW4ERA5_REFERENCE), the committed golden fixtures must be
exactly what the UNMODIFIED reference produces today: regenerate them and compare array by array.  The reference
is not part of this repository; without it the fixtures are all there is (skipped)."""
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle.golden import load as load_golden

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("PGW4ERA5_REFERENCE", "")
pytestmark = pytest.mark.skipif(not os.path.isfile(os.path.join(REF, "functions.py")),
                                reason="PGW4ERA5_REFERENCE does not name a checkout of the reference")


@pytest.mark.parametrize("script,fixture", [("make_golden.py", "reference_functions.npz"),
                                            ("make_golden_glue.py", "reference_glue.npz")])
def test_fixture_is_what_the_reference_returns(tmp_path, script, fixture):
    out = str(tmp_path / fixture)
    # a fresh interpreter: the scripts install stand-ins for xarray / pyvista / pyproj in sys.modules
    code = ("import sys; sys.path.insert(0, %r); sys.path.insert(0, %r); import %s as m; m.main(%r)"
            % (ROOT, os.path.join(ROOT, "oracle"), script[:-3], out))
    r = subprocess.run([sys.executable, "-W", "ignore", "-c", code], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    new, old = load_golden(out), load_golden(os.path.join(ROOT, "tests", "golden", fixture))
    assert sorted(new) == sorted(old)
    for k in old:
        assert new[k].dtype == old[k].dtype and new[k].shape == old[k].shape, k
        assert np.array_equal(new[k], old[k], equal_nan=(old[k].dtype.kind == "f")), k

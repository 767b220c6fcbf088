"""step_03 in latitude bands on the GPU: the command line's ``--latitude_bands`` under torchrun with one rank gives
the same bytes as the single-GPU command line (both column-kernel flavours), the band checks of
tests/multigpu_step03_bands.py at one rank, and a band of the delta climatology that stays resident under a
memory limit that makes the whole set stream."""
import os
import subprocess
import sys
from datetime import datetime, timedelta

import numpy as np
import pytest
import torch

from cases import make_case
from test_cli_gpu import _write_deltas, _write_era
from pgw4era5_b200 import settings, synthetic as S

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _env(**kw):
    env = dict(os.environ)
    env["PYTHONPATH"] = ROOT + (os.pathsep + env["PYTHONPATH"] if env.get("PYTHONPATH") else "")
    for k, v in kw.items():
        if v is None:
            env.pop(k, None)
        else:
            env[k] = v
    return env


def _run(cmd, env):
    p = subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, (cmd, p.stdout[-3000:], p.stderr[-5000:])
    return p.stdout


TORCHRUN = [sys.executable, "-m", "torch.distributed.run", "--standalone", "--nproc-per-node", "1"]


@pytest.mark.parametrize("column_path", [None, "generic"])
def test_one_band_cli_equals_the_cli(tmp_path, column_path):
    inp, dd = tmp_path / "in", tmp_path / "deltas"
    inp.mkdir(); dd.mkdir()
    era0, deltas = make_case(12, 20, 71)
    _write_deltas(str(dd), deltas, era0["lat"], era0["lon"])
    whens = [datetime(2006, 8, 2, 0) + timedelta(hours=6 * i) for i in range(3)]
    for i, w in enumerate(whens):
        _write_era(str(inp / settings.era5_file_name_base.format(w)),
                   S.make_era5(12, 20, 710 + i, lat=era0["lat"], lon=era0["lon"], orog_seed=71), w)
    args = lambda out: ["-i", str(inp), "-o", str(tmp_path / out), "-d", str(dd), "-f", "2006080200",
                        "-l", "2006080212", "-H", "6", "-t"]
    env = _env(PGW_COLUMN_PATH=column_path)
    _run([sys.executable, "-m", "pgw4era5_b200.step_03_apply_to_era"] + args("whole"), env)
    _run(TORCHRUN + ["-m", "pgw4era5_b200.step_03_apply_to_era"] + args("band") + ["--latitude_bands"], env)
    for w in whens:
        name = settings.era5_file_name_base.format(w)
        assert (tmp_path / "band" / name).read_bytes() == (tmp_path / "whole" / name).read_bytes(), name


def test_band_script_at_one_rank():
    out = _run(TORCHRUN + [os.path.join(ROOT, "tests", "multigpu_step03_bands.py")], _env())
    assert "all checks passed on 1 rank(s)" in out, out


def test_band_delta_set_stays_resident_where_the_whole_set_streams(tmp_path):
    from pgw4era5_b200 import deltastream
    from pgw4era5_b200 import step_03_apply_to_era as S3
    ny, nx = 14, 16
    era = S.make_era5(ny, nx, 72)
    deltas = S.make_deltas(era, 72, ntime=366)
    stamps = np.datetime64("2000-01-01T12:00", "ns") + np.arange(366) * np.timedelta64(86400 * 10 ** 9, "ns")
    for d in deltas.values():
        d["time"] = stamps
    dd = tmp_path / "deltas"
    dd.mkdir()
    _write_deltas(str(dd), deltas, era["lat"], era["lon"])
    need = deltastream.resident_bytes(deltastream.read_3d_headers(str(dd)))
    limit = need // 2 + 1
    assert S3.load_delta_set(str(dd), "cuda", max_resident_bytes=limit).streamed
    whole = S3.load_delta_set(str(dd), "cuda", max_resident_bytes=1 << 40)
    for r0, r1 in [(0, 7), (7, 14)]:
        band = S3.load_delta_set(str(dd), "cuda", max_resident_bytes=limit, rows=(r0, r1))
        assert not getattr(band, "streamed", False) and band.shape2d == (r1 - r0, nx)
        for name, v in whole.vars.items():
            assert torch.equal(band.vars[name]["data"].contiguous().view(torch.int32),
                               v["data"][..., r0:r1, :].contiguous().view(torch.int32)), name
        torch.testing.assert_close(band.ts_clim, whole.ts_clim[r0:r1], rtol=0, atol=0)
    with pytest.raises(ValueError, match="ranks or more would fit"):
        S3.load_delta_set(str(dd), "cuda", max_resident_bytes=need // 3 + 1, rows=(0, 7))

"""GCM-grid deltas without a GPU: the argument checks of pgw_regrid_pack_d4_f32, which return before any CUDA
call, and the refusals of step_03 --gcm_grid_deltas, which come before any delta is read."""
import ctypes as C
from datetime import datetime

import pytest

from pgw4era5_b200 import _native as N
from pgw4era5_b200 import step_03_apply_to_era as S3

P = C.c_void_p(4096)          # a 16-byte aligned address the checks never dereference


def _call(src=P, dst=P, pm=P, nlev=3, ny_s=12, nx_s=24, ny_t=20, nx_t=40, r0=0, r1=20, scratch=None):
    return N.lib.pgw_regrid_pack_d4_f32(src, dst, pm, nlev, ny_s, nx_s, ny_t, nx_t, r0, r1, P, P, P, P, P, P,
                                        scratch, None)


@pytest.mark.parametrize("bad", [
    dict(src=None), dict(dst=None), dict(pm=None), dict(nlev=0), dict(ny_s=0), dict(nx_s=0), dict(ny_t=0),
    dict(nx_t=0), dict(r0=-1), dict(r1=21), dict(r0=5, r1=5), dict(r0=6, r1=5),
    dict(dst=C.c_void_p(4100)),                                            # float4 stores need 16-byte alignment
    dict(nx_s=N.REGRID_PACK_MAX_NX_S + 1),                                 # the unfused branch needs the scratch
    dict(nx_s=N.REGRID_PACK_MAX_NX_S + 1, scratch=C.c_void_p(4104)),
])
def test_regrid_pack_rejects_bad_arguments(bad):
    assert _call(**bad) == N.PGW_E_INVALID


def _argv(tmp_path, *extra):
    return ["-i", str(tmp_path), "-o", str(tmp_path / "out"), "-d", str(tmp_path), "--gcm_grid_deltas",
            "-f", "2006080200", "-l", "2006080200"] + list(extra)


@pytest.fixture
def no_delta_set(monkeypatch):
    def built(*a, **k):
        raise AssertionError("a delta set was built")
    monkeypatch.setattr(S3, "load_gcm_grid_delta_set", built)
    monkeypatch.setattr(S3, "load_delta_set", built)


def test_cli_refuses_latitude_bands(tmp_path, no_delta_set):
    with pytest.raises(ValueError, match="--gcm_grid_deltas does not run with --latitude_bands"):
        S3.main(_argv(tmp_path, "--latitude_bands"))
    assert not (tmp_path / "out").exists()


def test_cli_refuses_interpolate_time(tmp_path, no_delta_set):
    with pytest.raises(ValueError, match="interpolate_time"):
        S3.main(_argv(tmp_path, "-D", "interpolate_time"))
    assert not (tmp_path / "out").exists()


def test_file_api_refusals(tmp_path, no_delta_set):
    steps = [dict(inp_era_file_path=str(tmp_path / "a.nc"), out_era_file_path=str(tmp_path / "b.nc"),
                  era_step_dt=datetime(2006, 8, 2))]
    with pytest.raises(ValueError, match="--latitude_bands"):
        S3.pgw_for_era5_files(steps, str(tmp_path), True, band=S3.Band(None, None), gcm_grid_deltas=True)
    with pytest.raises(ValueError, match="interpolate_time"):
        S3.pgw_for_era5_files(steps, str(tmp_path), True, debug_mode="interpolate_time", gcm_grid_deltas=True)
    with pytest.raises(ValueError, match="interpolate_time"):
        S3.debug_interpolate_time(gcm_grid_deltas=True, ignore_top_pressure_error=True, **steps[0],
                                  delta_input_dir=str(tmp_path))

"""Deltas on the GCM grid regridded on the device (gcmdeltas.GcmGridDeltaSet, pgw_regrid_pack_d4_f32) against
step_02 regridding followed by a resident DeltaSet: the fused kernel bit for bit against regrid_arrays and
pgw_pack_d4_f32, the engine's outputs bit for bit, and the output files of step_03 byte for byte."""
import ctypes as C
import os
from datetime import datetime

import numpy as np
import pytest
import torch

from cases import make_case
from test_delta_stream_gpu import (DATES, OUT, SETTINGS, _bits, _engine, _pipeline_all, _run, _settings, _snap,
                                   _submit_all, assert_same)
from pgw4era5_b200 import _native as N
from pgw4era5_b200 import functions as F
from pgw4era5_b200 import ncio, settings, synthetic as S
from pgw4era5_b200.engine import DeltaSet, VARS_2D, VARS_3D
from pgw4era5_b200.gcmdeltas import OCEAN_VARS, GcmGridDeltaSet

pytestmark = pytest.mark.gpu

DAY = np.timedelta64(86400 * 10 ** 9, "ns")
GL_LAT, GL_LON = np.linspace(-90.0, 90.0, 73), np.arange(144) * 2.5


def _p(t):
    return C.c_void_p(t.data_ptr() if t is not None else 0)


def _st():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _fields(K, lat, lon, seed, nan=True):
    """[4, K, ny_s, nx_s] float32 on the device; with ``nan``, scattered NaN, a NaN stretch of a row, and the whole
    first row of one field NaN (its pole mean is NaN)."""
    rng = np.random.default_rng(seed)
    ny, nx = len(lat), len(lon)
    x = (rng.normal(size=(4, K, ny, nx)) * 3 + 280).astype(np.float32)
    if nan:
        x[rng.uniform(size=x.shape) < 0.02] = np.nan
        x[1, 0, ny // 2, : nx // 3] = np.nan
        x[2, K - 1, 0, :] = np.nan
        x[3, 0, ny - 1, :] = np.nan
    return torch.from_numpy(x).cuda()


def _fused(src, lat, lon, tlat, tlon, rows=None, scratch=True):
    tb = F.regrid_tables(lat, lon, tlat, tlon)
    ti = lambda a: torch.as_tensor(np.ascontiguousarray(a), device="cuda", dtype=torch.int32)
    tf = lambda a: torch.as_tensor(np.ascontiguousarray(a), device="cuda", dtype=torch.float64)
    _, K, ny_s, nx_s = src.shape
    r0, r1 = (0, len(tlat)) if rows is None else rows
    pm = torch.empty((4 * K, 2), device="cuda", dtype=torch.float32)
    N.check(N.lib.pgw_zonal_mean_f32(_p(src), _p(pm), 4 * K, ny_s, nx_s, _st()), "pgw_zonal_mean_f32")
    n = K * (r1 - r0) * len(tlon)
    out = torch.full((n, 4), -1, device="cuda", dtype=torch.int32)
    sc = torch.empty(4 * ((n + 3) // 4 * 4), device="cuda", dtype=torch.float32) if scratch else None
    # the tables stay referenced until the kernel has run (a temporary would return its block to the allocator)
    tabs = [ti(tb["j0"]), ti(tb["j1"]), tf(tb["wy"]), ti(tb["i0"]), ti(tb["i1"]), tf(tb["wx"])]
    rc = N.lib.pgw_regrid_pack_d4_f32(_p(src), _p(out), _p(pm), K, ny_s, nx_s, len(tlat), len(tlon), r0, r1,
                                      *[_p(t) for t in tabs], _p(sc), _st())
    torch.cuda.synchronize()
    return rc, out


def _unfused(src, lat, lon, tlat, tlon, rows=None):
    """regrid_arrays on each variable, then pgw_pack_d4_f32."""
    parts = [F.regrid_arrays(src[v], lat, lon, tlat, tlon, rows=rows).contiguous() for v in range(4)]
    n = parts[0].numel()
    out = torch.full((n, 4), -2, device="cuda", dtype=torch.int32)
    N.check(N.lib.pgw_pack_d4_f32(*[_p(t) for t in parts], _p(out), n, 0, _st()), "pgw_pack_d4_f32")
    return out


KERNEL_CASES = {
    # global GCM grid (192 x 384 like MPI-ESM1-2-HR, fewer levels) onto a 2.5 degree global target
    "global": (np.linspace(-89.28, 89.28, 192), np.arange(384) * 0.9375, GL_LAT, GL_LON, None, 3),
    # regional ERA5 subset, longitudes west of 0 served by the periodic source, nx_t not a multiple of 4
    "regional": (np.linspace(-88.5, 88.5, 60), np.arange(96) * 3.75, np.linspace(30.0, 80.0, 51),
                 np.linspace(-20.0, 50.0, 71), None, 4),
    # source latitudes north to south (no pole rows then: the median step is negative), only target rows [7, 40)
    "descending_rows": (np.linspace(88.5, -88.5, 60), np.arange(96) * 3.75, np.linspace(-80.0, 80.0, 65), GL_LON,
                        (7, 40), 2),
    # rows wider than the fused kernel takes: regridded into the scratch and packed
    "wide_fallback": (np.linspace(20.0, 85.0, 14), np.arange(1600) * 0.225, np.linspace(30.0, 80.0, 21),
                      np.linspace(-20.0, 50.0, 36), (3, 17), 2),
}


@pytest.mark.parametrize("case", list(KERNEL_CASES))
def test_regrid_pack_matches_regrid_then_pack(case):
    lat, lon, tlat, tlon, rows, K = KERNEL_CASES[case]
    assert (len(lon) > N.REGRID_PACK_MAX_NX_S) == (case == "wide_fallback")
    src = _fields(K, lat, lon, seed=len(case))
    rc, got = _fused(src, lat, lon, tlat, tlon, rows)
    assert rc == N.PGW_OK
    want = _unfused(src, lat, lon, tlat, tlon, rows)
    assert torch.isnan(got.view(torch.float32)).any()              # NaN made it through (and the pole row's)
    assert torch.equal(got.cpu(), want.cpu())


# ------------------------------------------------------------------------------------------------ the delta set
GCM_LAT, GCM_LON = np.linspace(-88.5, 88.5, 12), np.arange(24) * 15.0


def _ocean_grid(lat, lon):
    """Curvilinear 2-D coordinates around the regular grid (as an ocean model's)."""
    glat, glon = np.meshgrid(lat, lon, indexing="ij")
    return np.clip(glat + 0.8 * np.sin(np.radians(glon) * 2), -89.0, 89.5), np.mod(glon + 1.5 * np.cos(np.radians(glat) * 3), 360.0)


def gcm_daily_case(ny, nx, seed=5):
    """An EU-region ERA5 case on (ny, nx) and a daily (leap year 2000) climatology on a global 12 x 24 GCM grid,
    tos / siconc on a curvilinear version of it, in the dict form GcmGridDeltaSet takes."""
    era, _ = make_case(ny, nx, seed)
    gera = S.make_era5(len(GCM_LAT), len(GCM_LON), seed, lat=GCM_LAT, lon=GCM_LON)
    deltas = S.make_deltas(gera, seed, ntime=366)
    stamps = np.datetime64("2000-01-01T12:00", "ns") + np.arange(366) * DAY
    olat, olon = _ocean_grid(GCM_LAT, GCM_LON)
    for name, d in deltas.items():
        d["time"] = stamps
        d["data"] = d["data"].numpy()
        d["lat"], d["lon"] = (olat, olon) if name in OCEAN_VARS else (GCM_LAT, GCM_LON)
    return era, deltas


def regridded(era, deltas):
    """What step_02 regridding writes for ``deltas`` (float64 for tos / siconc), as DeltaSet's dict form."""
    land = S.to_numpy(era)["FR_LAND"][0]
    out = {}
    for name, d in deltas.items():
        if name in OCEAN_VARS:
            data = F.nan_ignoring_interp_arrays(land, era["lat"], era["lon"], d["data"], d["lat"], d["lon"],
                                                settings.nan_interp_kernel_radius, settings.nan_interp_sharpness)
        else:
            data = F.regrid_arrays(d["data"], d["lat"], d["lon"], era["lat"], era["lon"])
        out[name] = dict(time=d["time"], plev=d["plev"], data=data)
    return out


def _gcm_set(era, deltas, slots=4):
    return GcmGridDeltaSet(deltas, era["lat"], era["lon"], S.to_numpy(era)["FR_LAND"][0], slots=slots)


@pytest.mark.parametrize("grid", [(8, 16), (7, 13)], ids=["tma", "cp_async"])
@pytest.mark.parametrize("slots", [2, 4])
@pytest.mark.parametrize("setting", list(SETTINGS))
def test_submit_matches_resident(grid, slots, setting):
    era, deltas = gcm_daily_case(*grid)
    names = OUT + (("p_ref",) if setting == "p_ref_inp=None" else ())
    with _settings(**SETTINGS[setting]):
        want = _submit_all(_engine(era, DeltaSet(regridded(era, deltas))), era, DATES)
        ds = _gcm_set(era, deltas, slots)
        got = _submit_all(_engine(era, ds), era, DATES)
    for g, w in zip(got, want):
        assert_same(g, w, names)
    # 9 days of stamps (27 Feb .. 2 Mar without 29 Feb, 30 Dec .. 1 Jan): each loaded once
    assert ds.rings["d4"].loads == ds.rings["zg"].loads == 9


def test_stamps_and_2d_deltas_match_step02():
    era, deltas = gcm_daily_case(8, 16)
    ref = DeltaSet(regridded(era, deltas))
    ds = _gcm_set(era, deltas, slots=2)
    assert ds.streamed and ds.device_bytes() > 0
    for name in VARS_2D:
        assert torch.equal(_bits(ds.stamp(name, 59)), _bits(ref.stamp(name, 59))), name
    assert torch.isnan(ds.stamp("tos", 0)).any()                   # land and GCM land stay NaN
    for name in VARS_3D:
        for i in (0, 58, 59, 364, -1):
            assert torch.equal(_bits(ds.stamp(name, i)), _bits(ref.stamp(name, i))), (name, i)
            ds.hold()                                               # a ring of 2 slots: release the stamp


def test_host_pipeline_matches_resident():
    era, deltas = gcm_daily_case(8, 16)
    want = _pipeline_all(DeltaSet(regridded(era, deltas)), era, 8, 16)
    got = _pipeline_all(_gcm_set(era, deltas, slots=2), era, 8, 16)
    assert len(got) == len(want) == len(DATES)
    for g, w in zip(got, want):
        for name in OUT:
            assert torch.equal(_bits(g[name]), _bits(w[name])), name
        assert g["n_iter"] == w["n_iter"]


@pytest.mark.parametrize("setting", [dict(i_reinterp=1), dict(i_reinterp=1, p_ref_inp=None)])
def test_staged_apply_matches_resident(setting):
    era, deltas = gcm_daily_case(7, 13)
    dates = [datetime(2000, 2, 28, 18), datetime(2000, 3, 1, 12), datetime(2000, 12, 31, 21)]
    dev = {k: (v.cuda() if isinstance(v, torch.Tensor) else v) for k, v in era.items()}
    with _settings(**setting):
        want = [_snap(_engine(era, DeltaSet(regridded(era, deltas))).apply(dev, d, ignore_top_pressure_error=True))
                for d in dates]
        eng = _engine(era, _gcm_set(era, deltas, slots=2))
        got = [_snap(eng.apply(dev, d, ignore_top_pressure_error=True)) for d in dates]
    names = OUT + (("p_ref",) if "p_ref_inp" in setting else ())
    for g, w in zip(got, want):
        assert_same(g, w, names)


def test_gcm_grid_must_cover_the_era5_domain():
    era, deltas = gcm_daily_case(8, 16)
    for name in ("ta", "hur", "ua", "va"):
        deltas[name]["lat"] = deltas[name]["lat"] * 0.5               # reaches 44 N, ERA5 80 N
    with pytest.raises(ValueError, match="ERA5 dataset extends further North or South than GCM dataset"):
        _gcm_set(era, deltas)


# ------------------------------------------------------------------------------------------- the command line
def _write_gcm_files(ddir, deltas):
    """The GCM-grid delta files step_02 regridding reads: every variable as HIST and SCEN-HIST."""
    for name, v in deltas.items():
        var = "ps" if name == "ps_hist" else name
        ds = ncio.Dataset()
        ds["time"] = ncio.encode_time(v["time"], "days since 1850-01-01 00:00:00")
        if name in OCEAN_VARS:
            ds["latitude"] = ncio.Variable(("j", "i"), v["lat"]); ds["longitude"] = ncio.Variable(("j", "i"), v["lon"])
            ds[var] = ncio.Variable(("time", "j", "i"), v["data"])
        else:
            ds["lat"] = ncio.Variable(("lat",), v["lat"]); ds["lon"] = ncio.Variable(("lon",), v["lon"])
            if v["plev"] is not None:
                ds["plev"] = ncio.Variable(("plev",), v["plev"])
                ds[var] = ncio.Variable(("time", "plev", "lat", "lon"), v["data"])
            else:
                ds[var] = ncio.Variable(("time", "lat", "lon"), v["data"])
        for base in settings.file_name_bases.values():
            ds.to_netcdf(os.path.join(ddir, base.format(var)))


def test_cli_gcm_grid_deltas_match_step02_regridding(tmp_path, monkeypatch):
    from test_cli_gpu import _write_era
    from pgw4era5_b200 import step_02_preproc_deltas as S2
    from pgw4era5_b200 import step_03_apply_to_era as S3
    era, deltas = gcm_daily_case(10, 24)
    inp, gdir, rdir = tmp_path / "in", tmp_path / "gcm", tmp_path / "regridded"
    inp.mkdir(); gdir.mkdir()
    dates = _run(datetime(2000, 2, 28, 6), datetime(2000, 3, 1, 18), hours=6)
    for when in dates:
        _write_era(str(inp / settings.era5_file_name_base.format(when)), era, when)
    # -D interpolate_full writes the hur delta in the shape of the file's RELHUM
    inpf = tmp_path / "in_full"
    inpf.mkdir()
    for when in dates[3:6]:
        name = settings.era5_file_name_base.format(when)
        e = ncio.open_dataset(str(inp / name))
        e["RELHUM"] = ncio.Variable(e["T"].dims, np.zeros_like(e["T"].data))
        e.to_netcdf(str(inpf / name))
    _write_gcm_files(str(gdir), deltas)
    first = str(inp / settings.era5_file_name_base.format(dates[0]))
    argv = lambda d, out, *extra: ["-i", str(inp), "-o", str(tmp_path / out), "-d", str(d), "-f",
                                   dates[0].strftime("%Y%m%d%H"), "-l", dates[-1].strftime("%Y%m%d%H"), "-H", "6",
                                   "-t"] + list(extra)
    argv_full = lambda d, out, *extra: ["-i", str(inpf), "-o", str(tmp_path / out), "-d", str(d), "-f",
                                        dates[3].strftime("%Y%m%d%H"), "-l", dates[5].strftime("%Y%m%d%H"), "-H",
                                        "6", "-t", "-D", "interpolate_full"] + list(extra)
    with _settings(i_debug=0):
        monkeypatch.setattr(S3, "_ENGINES", {})
        S2.main(["regridding", "-i", str(gdir), "-o", str(rdir), "-e", first])
        runs = [("a1", rdir), ("b1", gdir, "--gcm_grid_deltas"), ("a2", rdir, "-p", "2"),
                ("b2", gdir, "--gcm_grid_deltas", "-p", "2")]
        for out, d, *extra in runs:
            S3.main(argv(d, out, *extra))
        S3.main(argv_full(rdir, "af"))
        S3.main(argv_full(gdir, "bf", "--gcm_grid_deltas"))
    assert any(getattr(e.deltas, "grids", None) for e in S3._ENGINES.values())
    for a, b in (("a1", "b1"), ("a2", "b2"), ("af", "bf")):
        names = sorted(os.listdir(tmp_path / a))
        assert names == sorted(os.listdir(tmp_path / b)) and len(names) >= 3
        for name in names:
            assert (tmp_path / a / name).read_bytes() == (tmp_path / b / name).read_bytes(), (a, b, name)
    assert len(os.listdir(tmp_path / "a1")) == len(dates)
    assert len(os.listdir(tmp_path / "af")) == 7 * 3                  # interpolate_full writes 7 deltas per file

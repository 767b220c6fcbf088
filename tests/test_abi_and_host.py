"""CPU-side checks: the C-ABI library loads and exports every symbol the header declares;
host logic (calendar brackets, regrid tables, partitioning, NetCDF shim) against the oracle."""
import os
import re
import warnings
from datetime import datetime

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "pgw_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(pgw_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    import ctypes
    from pgw4era5_b200 import _native as N
    lib = ctypes.CDLL(N.LIB_PATH)
    declared = _declared_symbols()
    assert len(declared) >= 25
    for name in declared:
        assert hasattr(lib, name), "libpgw_b200.so does not export %s" % name
    # and the Python binding covers all of them
    assert set(declared) <= set(N.EXPORTED) | {"pgw_version", "pgw_last_error"}
    assert N.lib.pgw_version().startswith(b"pgw_b200")
    assert N.lib.pgw_sizeof_timestep_args() == ctypes.sizeof(N.TimestepArgs)
    # the header's ABI number is what the library reports and what the binding expects
    import re
    hdr = open(os.path.join(os.path.dirname(__file__), "..", "include", "pgw_b200.h")).read()
    ver = int(re.search(r"#define PGW_B200_ABI_VERSION (\d+)", hdr).group(1))
    assert N.lib.pgw_abi_version() == ver == N.ABI_VERSION
    assert ("abi %d" % ver).encode() in N.lib.pgw_version()


def test_invalid_arguments_are_rejected_without_a_gpu():
    from pgw4era5_b200 import _native as N
    assert N.lib.pgw_time_mean_f32(None, 12, None, 10, None) == N.PGW_E_INVALID
    assert N.lib.pgw_interp_logp_f32(None, None, None, None, 1, 2, 3, 4, 0, 0, 2, None, None) == N.PGW_E_INVALID
    assert N.lib.pgw_smooth_harmonic_f32(None, None, 365, 10, None) == N.PGW_E_INVALID
    assert N.lib.pgw_timestep(None, None) == N.PGW_E_INVALID


def test_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from pgw4era5_b200 import functions as F
    with pytest.raises(RuntimeError, match="no CPU path"):
        F.specific_to_relative_humidity(np.ones(3), np.ones(3), np.ones(3))


@pytest.mark.parametrize("when", [datetime(2006, 8, 2, 6), datetime(2006, 1, 1, 0), datetime(2006, 12, 31, 18),
                                  datetime(2006, 3, 16, 12), datetime(2008, 2, 29, 6), datetime(2007, 1, 16, 12)])
def test_time_bracket_matches_oracle(when):
    from oracle import pgw_oracle as O
    from pgw4era5_b200 import synthetic as S, timeinterp as TI
    stamps = S.monthly_stamps()
    b = TI.bracket(stamps[TI.drop_leap_day(stamps)], when)
    keep, ib, ia, x_hi, x_new = O.delta_time_bracket(stamps, when)
    assert (b.ind_before, b.ind_after) == (ib, ia)
    if ib != ia:
        assert (b.x_hi, b.x_new) == (x_hi, x_new)
    else:
        assert b.exact and b.x_new == 0.0


def test_leap_day_dropped_from_daily_series():
    from oracle import pgw_oracle as O
    from pgw4era5_b200 import timeinterp as TI
    days = np.datetime64("2000-01-01T12", "ns") + np.arange(366) * np.timedelta64(86400 * 10 ** 9, "ns")
    keep = TI.drop_leap_day(days)
    assert len(keep) == 365 and 59 not in keep
    assert keep == O.delta_time_bracket(days, datetime(2003, 3, 1, 0))[0]
    b = TI.bracket(days[keep], datetime(2003, 2, 28, 18))
    k2, ib, ia, x_hi, x_new = O.delta_time_bracket(days, datetime(2003, 2, 28, 18))
    assert (b.ind_before, b.ind_after, b.x_hi, b.x_new) == (ib, ia, x_hi, x_new)


def _emulate_gather(data, tb):
    # zonal_mean_kernel: mean of the valid points of the first / last row (NaN if none), rounded to float32
    with np.errstate(all="ignore"), warnings.catch_warnings():
        warnings.simplefilter("ignore", RuntimeWarning)
        pm0 = np.nanmean(data[..., 0, :], -1, dtype=np.float64).astype(np.float32).astype(np.float64)
        pm1 = np.nanmean(data[..., -1, :], -1, dtype=np.float64).astype(np.float32).astype(np.float64)

    def at(j, i):
        out = np.empty(data.shape[:-2] + (len(j), len(i)))
        for a, jj in enumerate(j):
            for b, ii in enumerate(i):
                out[..., a, b] = pm0 if jj == -1 else (pm1 if jj == -2 else data[..., jj, ii])
        return out
    a0, a1 = at(tb["j0"], tb["i0"]), at(tb["j1"], tb["i0"])
    b0, b1 = at(tb["j0"], tb["i1"]), at(tb["j1"], tb["i1"])
    wy, wx = tb["wy"][:, None], tb["wx"][None, :]
    a = (a1 - a0) * wy + a0
    b = (b1 - b0) * wy + b0
    return (b - a) * wx + a


GRID_CASES = [
    # global 10 degree GCM -> coarse "ERA5" incl. poles, 0..360 both
    (np.linspace(-85, 85, 18), np.arange(0.0, 360, 10.0), np.linspace(-90, 90, 25), np.arange(0, 360, 7.5)),
    # GCM on -180..180, target 0..360: periodic wrap to the east
    (np.linspace(-85, 85, 18), np.arange(-180.0, 180, 10.0), np.linspace(-60, 60, 13), np.arange(0, 360, 7.5)),
    # GCM on 0..360, target -180..180: periodic wrap to the west
    (np.linspace(-85, 85, 18), np.arange(0.0, 360, 10.0), np.linspace(-60, 60, 13), np.arange(-180, 180, 7.5)),
    # regional, descending source latitude
    (np.linspace(85, 20, 14), np.arange(-30.0, 61, 5.0), np.linspace(30, 80, 11), np.linspace(-20, 50, 15)),
]


@pytest.mark.parametrize("case", range(len(GRID_CASES)))
def test_regrid_tables_match_oracle(case):
    from oracle import pgw_oracle as O
    from pgw4era5_b200 import functions as F
    lat, lon, tlat, tlon = GRID_CASES[case]
    rng = np.random.default_rng(case)
    data = rng.normal(size=(2, len(lat), len(lon))).astype(np.float32)
    ref = O.regrid_lat_lon(data, lat, lon, tlat, tlon)
    got = _emulate_gather(data.astype(np.float64), F.regrid_tables(lat, lon, tlat, tlon))
    assert not np.isnan(ref).any()
    np.testing.assert_allclose(got, ref, rtol=0, atol=2e-7)


def test_regrid_pole_rows_skip_nan():
    """The pole rows are `north[var].mean(dim=[lon])` (functions.py:833-842): an xarray mean, which skips NaN
    for float data.  A partly missing first / last source row gives the mean of its valid points, so the target
    rows between the pole and that row stay finite wherever the row is; an all-NaN row gives NaN."""
    from oracle import pgw_oracle as O
    from oracle import xrlite as xr
    from pgw4era5_b200 import functions as F
    lat, lon = np.linspace(-85, 85, 18), np.arange(0.0, 360, 10.0)
    tlat, tlon = np.linspace(-90, 90, 73), np.arange(0, 360, 7.5)
    rng = np.random.default_rng(4)
    data = rng.normal(size=(3, len(lat), len(lon))).astype(np.float32)
    data[0, 0, 5:9] = np.nan                       # partly missing southernmost row
    data[1, -1, ::9] = np.nan                      # partly missing northernmost row
    data[2, 0, :] = np.nan                         # whole southernmost row missing
    ref = O.regrid_lat_lon(data, lat, lon, tlat, tlon)
    got = _emulate_gather(data.astype(np.float64), F.regrid_tables(lat, lon, tlat, tlon))
    np.testing.assert_array_equal(np.isnan(got), np.isnan(ref))
    np.testing.assert_allclose(got, ref, rtol=0, atol=2e-7, equal_nan=True)
    # target rows -87.5 and 87.5 lie between a pole row and the partly missing source row: finite where that row is
    assert 0 < np.isnan(ref[0, 1]).sum() < len(tlon) // 2 and 0 < np.isnan(ref[1, -2]).sum() < len(tlon) // 2
    # an all-NaN row: NaN up to the next source row (-75, bracketed with row 0), finite from there on
    assert np.isnan(ref[2, :7]).all() and np.isfinite(ref[2, 7:]).all()
    # the pole value itself is xrlite's DataArray.mean over lon (xarray semantics restated)
    da = xr.DataArray(data[0, :1].astype(np.float64), dims=("lat", "lon"), coords={"lat": lat[:1], "lon": lon})
    pole = float(da.mean(dim=["lon"]).values[0])
    assert np.isfinite(pole) and abs(ref[0, 0, 0] - pole) < 1e-12


def test_regrid_bounds_errors():
    from pgw4era5_b200 import functions as F
    lat, lon = np.linspace(20, 60, 9), np.arange(0.0, 41, 5.0)
    with pytest.raises(ValueError, match="North or South"):
        F.regrid_tables(lat, lon, np.linspace(10, 50, 5), np.linspace(5, 35, 4))
    with pytest.raises(ValueError, match="East or West"):
        F.regrid_tables(lat, lon, np.linspace(25, 50, 5), np.linspace(5, 75, 4))
    # the reference's quirk: a descending-latitude global GCM grid gets no pole rows (dlat < 0)
    with pytest.raises(ValueError, match="North or South"):
        F.regrid_tables(np.linspace(85, -85, 18), np.arange(0.0, 360, 10), np.linspace(-90, 90, 7), np.arange(0, 360, 30.))


def test_partitioning():
    from pgw4era5_b200 import parallel as P
    bands = P.split_rows(721, 8)
    assert bands[0] == (0, 90) and bands[-1] == (630, 721)
    assert sum(b - a for a, b in bands) == 721
    assert all(bands[i][1] == bands[i + 1][0] for i in range(7))
    seen = sorted(sum((P.timesteps_for_rank(124, r, 8) for r in range(8)), []))
    assert seen == list(range(124))
    assert P.decide_n_iter([270.0, 40.0, 5.9, 0.87, 0.139], 0.15) == 5
    assert P.decide_n_iter([270.0, 40.0], 0.15) == 0
    assert P.decide_n_iter([float("nan")], 0.15) == 1      # NaN > thresh is False: loop ends (step_03:189)


def test_netcdf_roundtrip(tmp_path):
    from pgw4era5_b200 import ncio
    ds = ncio.Dataset()
    ds["time"] = ncio.Variable(("time",), np.array([1.5]), {"units": "hours since 2006-08-02 00:00:00"})
    ds["lat"] = ncio.Variable(("lat",), np.linspace(30, 32, 3))
    ds["lon"] = ncio.Variable(("lon",), np.linspace(5, 8, 4))
    ds["PS"] = ncio.Variable(("time", "lat", "lon"), np.arange(12, dtype=np.float32).reshape(1, 3, 4), {"units": "Pa"})
    path = str(tmp_path / "x.nc")
    ds.to_netcdf(path)
    back = ncio.open_dataset(path)
    assert back["PS"].dims == ("time", "lat", "lon") and back["PS"].data.dtype == np.float32
    np.testing.assert_array_equal(back["PS"].data, ds["PS"].data)
    assert back["PS"].attrs["units"] == "Pa"
    t = ncio.decode_time(back["time"])
    assert t[0] == np.datetime64("2006-08-02T01:30:00", "ns")
    noleap = ncio.Variable(("time",), np.array([59.0, 365.0]), {"units": "days since 2001-01-01", "calendar": "noleap"})
    assert list(ncio.decode_time(noleap)) == [np.datetime64("2001-03-01", "ns"), np.datetime64("2002-01-01", "ns")]


def test_settings_surface():
    from pgw4era5_b200 import settings, constants
    assert (constants.CON_RD, constants.CON_G, constants.CON_MW_MD) == (287.05, 9.80665, 0.622)
    assert settings.p_ref_inp == 30000 and settings.adj_factor == 0.95
    assert settings.thresh_phi_ref_max_error == 0.15 and settings.max_n_iter == 20 and settings.i_reinterp == 0
    assert settings.var_name_map["hus"] == "QV" and settings.era5_file_name_base.format(datetime(2006, 8, 2, 6)) == \
        "cas20060802060000.nc"
    from pgw4era5_b200.step_03_apply_to_era import build_parser
    a = build_parser().parse_args(["-i", "a", "-o", "b", "-d", "c", "-t", "-p", "2", "-H", "6"])
    assert a.ignore_top_pressure_error and a.n_par == 2 and a.hour_inc_step == 6 and a.first_era_step == "2006080200"


def test_numa_binding_helpers():
    """parallel.bind_to_gpu_numa: cpulist parsing; without a GPU / exposed topology nothing changes."""
    import os
    from pgw4era5_b200.parallel import _parse_cpulist, bind_to_gpu_numa
    assert _parse_cpulist("0-3,8,10-11\n") == {0, 1, 2, 3, 8, 10, 11} and _parse_cpulist("") == set()
    before = os.sched_getaffinity(0)
    import torch
    if not torch.cuda.is_available():
        assert bind_to_gpu_numa(0) is None and os.sched_getaffinity(0) == before


def test_decode_time_calendars():
    """CF calendars the way the reference ends up with them after to_datetimeindex (functions.py:203-221): the
    calendar date is kept, nothing is shifted; dates the standard calendar lacks and unknown calendars raise."""
    from pgw4era5_b200 import ncio, timeinterp
    V = ncio.Variable
    # a 360_day monthly delta file (HadGEM / UKESM style): mid-month stamps of model year 2000
    t360 = np.array([150 * 360 + 30 * m + 15.5 for m in range(12)])
    got = ncio.decode_time(V(("time",), t360, {"units": "days since 1850-01-01", "calendar": "360_day"}))
    want = np.array(["2000-%02d-16T12:00:00" % (m + 1) for m in range(12)], dtype="datetime64[ns]")
    assert np.array_equal(got, want)
    # ... which brackets an ERA5 date exactly like a standard-calendar file with the same stamps
    from datetime import datetime
    b = timeinterp.bracket(got, datetime(2006, 8, 2, 6))
    assert (b.ind_before, b.ind_after) == (6, 7)
    # decoded as proleptic Gregorian (what the code did before) these stamps would drift ~5 days per year
    greg = ncio.decode_time(V(("time",), t360, {"units": "days since 1850-01-01"}))
    assert abs((greg[0] - want[0]) / np.timedelta64(1, "D")) > 700
    # noleap across years, all_leap, julian
    got = ncio.decode_time(V(("time",), np.array([59.5, 365.0 + 59.5]),
                             {"units": "days since 2001-01-01", "calendar": "noleap"}))
    assert np.array_equal(got, np.array(["2001-03-01T12", "2002-03-01T12"], dtype="datetime64[ns]"))
    got = ncio.decode_time(V(("time",), np.array([60.0, 366.0 + 60.0]),
                             {"units": "days since 2000-01-01", "calendar": "366_day"}))
    assert np.array_equal(got, np.array(["2000-03-01", "2001-03-01"], dtype="datetime64[ns]"))
    # 1900-02-29 exists in the julian calendar only
    with pytest.raises(ValueError, match="standard calendar"):
        ncio.decode_time(V(("time",), np.array([365.0 * 3 + 59.0]),
                           {"units": "days since 1897-01-01", "calendar": "julian"}))
    with pytest.raises(ValueError, match="standard calendar"):          # 30 February
        ncio.decode_time(V(("time",), np.array([150 * 360 + 59.0]), {"units": "days since 1850-01-01",
                                                                     "calendar": "360_day"}))
    with pytest.raises(ValueError, match="unsupported calendar"):
        ncio.decode_time(V(("time",), np.array([1.0]), {"units": "days since 1850-01-01", "calendar": "lunar"}))
    # negative offsets
    got = ncio.decode_time(V(("time",), np.array([-1.0]), {"units": "days since 2001-01-01", "calendar": "360_day"}))
    assert got[0] == np.datetime64("2000-12-30")


def test_error_bits_of_iterations_the_reference_never_ran_are_ignored(monkeypatch):
    """The kernel runs k_spec iterations for every column, the reference stops after N.  PGW_ERR_PREF_BELOW_SFC /
    PGW_ERR_PS_BOUND that first fired in an iteration >= N (status.first_k) did not happen in the reference:
    no error, no rerun.  Host logic of PGWEngine._complete on a hand-made status block (no GPU needed)."""
    import types
    from pgw4era5_b200 import _native as N
    from pgw4era5_b200 import engine as E

    def run(err, first_k, n_iter, converged=1, k_spec=8):
        st = N.TimestepStatus()
        st.err = err
        st.first_k[0], st.first_k[1] = first_k
        st.result.n_iter, st.result.converged, st.result.rewritten = n_iter, converged, 0
        st.stats[0], st.stats[1] = 500.0, 100.0
        eng = object.__new__(E.PGWEngine)
        eng.deltas = types.SimpleNamespace(plev=np.array([100000.0, 100.0]))
        eng.stats = dict(timesteps=0, rewrites=0, reruns=0, launches=0)
        eng._n_hist, eng.k_pred, eng.ps_bound = [], 8, 110000.0
        eng.submit = lambda *a, **k: (_ for _ in ()).throw(AssertionError("rerun"))
        import contextlib
        p = types.SimpleNamespace(snapshot=lambda: st, out={}, ctx=dict(
            ignore_top=True, k_spec=k_spec, k_max=19, file_name="f", stream=None, era=None, when=None, slot=0,
            direct=False))
        E.torch.cuda.stream = lambda s: contextlib.nullcontext()
        return E.PGWEngine._complete(eng, p)

    big = N.INT32_MAX
    from pgw4era5_b200 import settings
    monkeypatch.setattr(settings, "i_debug", 0)
    monkeypatch.setattr(E.torch.cuda, "stream", E.torch.cuda.stream)      # restored after the test
    assert run(0, (big, big), 6)["n_iter"] == 6
    # fired only in the speculative iterations 6, 7 (0-based) of k_spec = 8 while the reference stopped after 6
    assert run(N.ERR_PREF_BELOW_SFC, (6, big), 6)["n_iter"] == 6
    assert run(N.ERR_PS_BOUND, (big, 7), 6)["n_iter"] == 6
    # fired in an iteration the reference did run
    with pytest.raises(ValueError, match="below the surface"):
        run(N.ERR_PREF_BELOW_SFC, (5, big), 6)
    with pytest.raises(AssertionError, match="rerun"):
        run(N.ERR_PS_BOUND, (big, 2), 6)
    # not converged: every one of the k_spec iterations counts
    with pytest.raises(ValueError, match="below the surface"):
        run(N.ERR_PREF_BELOW_SFC, (7, big), 0, converged=0)

"""
TEST INFRASTRUCTURE ONLY -- generates tests/golden/reference_glue.npz by running the UNMODIFIED
reference code -- functions.py and step_03_apply_to_era.py of the PGW4ERA5 checkout in
$PGW4ERA5_REFERENCE, including the xarray-bound
functions (integ_geopot, load_delta, load_delta_interp, vert_interp_delta, interp_logp_4d,
regrid_lat_lon, filter_data and the whole of pgw_for_era5) -- on small seeded cases.

xarray is absent from the build container; ``oracle/xrlite.py`` (a restatement of xarray's published
semantics for exactly the calls the reference makes) is installed as ``sys.modules['xarray']`` for
this script only, pyvista/pyproj are empty stand-ins (never touched on this path).  The reference
is not part of this repository, hence the inputs AND the reference's outputs are committed as a
fixture (written by oracle/golden.py); ``tests/test_oracle_glue_golden.py`` pins the oracle against
it and ``tests/test_timestep_gpu.py`` the CUDA path.

    PGW4ERA5_REFERENCE=/path/to/PGW4ERA5 python oracle/make_golden_glue.py
"""
import contextlib
import io
import os
import re
import sys
import tempfile
import types
from datetime import datetime

import numpy as np
from scipy.io import netcdf_file

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
REF = os.environ.get("PGW4ERA5_REFERENCE", "")
OUT = os.path.join(ROOT, "tests", "golden", "reference_glue.npz")
sys.path.insert(0, ROOT)
from oracle import golden  # noqa: E402


def import_reference():
    if not os.path.isfile(os.path.join(REF, "functions.py")):
        raise SystemExit("set PGW4ERA5_REFERENCE to the directory of a PGW4ERA5 checkout")
    from oracle import xrlite
    sys.modules["xarray"] = xrlite
    for name, attrs in (("pyvista", ("PolyData",)), ("pyproj", ("Geod",))):
        mod = types.ModuleType(name)
        for a in attrs:
            setattr(mod, a, object)
        sys.modules[name] = mod
    sys.path.insert(0, REF)
    import functions            # noqa: the reference's functions.py
    import step_03_apply_to_era  # noqa: the reference's step_03
    return xrlite, functions, step_03_apply_to_era


# ----------------------------------------------------------------------------- file writers
def _nc(path, dims, variables):
    """variables: name -> (dims, data, attrs)"""
    with netcdf_file(path, "w", version=2) as f:
        for d, n in dims.items():
            f.createDimension(d, n)
        for name, (vd, data, attrs) in variables.items():
            data = np.asarray(data)
            v = f.createVariable(name, "f" if data.dtype == np.float32 else "d", vd)
            v[:] = data
            for k, a in attrs.items():
                setattr(v, k, a)


def write_era(path, era, when, with_akm=False, ps_f64=False):
    hours = (np.datetime64(when, "ns") - np.datetime64("2006-08-01T00", "ns")) / np.timedelta64(1, "h")
    L = era["T"].shape[1]
    ny, nx = era["PS"].shape[-2:]
    v = {"time": (("time",), np.array([float(hours)]), {"units": "hours since 2006-08-01 00:00:00"}),
         "lat": (("lat",), era["lat"], {}), "lon": (("lon",), era["lon"], {}),
         "level": (("level",), np.arange(1, L + 1, dtype=np.float64), {}),
         "level1": (("level1",), np.arange(1, L + 2, dtype=np.float64), {}),
         "soil1": (("soil1",), era["soil1"], {}),
         "ak": (("level1",), era["ak"], {}), "bk": (("level1",), era["bk"], {})}
    if with_akm:
        v["akm"] = (("level",), era["akm"], {})
        v["bkm"] = (("level",), era["bkm"], {})
    for name in ("PS", "FIS", "FR_LAND", "FR_SEA_ICE", "T_SKIN"):
        v[name] = (("time", "lat", "lon"), era[name], {})
    if ps_f64:          # the same (float32-representable) values stored as double
        v["PS"] = (("time", "lat", "lon"), era["PS"].astype(np.float64), {})
        v["FIS"] = (("time", "lat", "lon"), era["FIS"].astype(np.float64), {})
    v["T_SO"] = (("time", "soil1", "lat", "lon"), era["T_SO"], {})
    for name in ("T", "QV", "U", "V"):
        v[name] = (("time", "level", "lat", "lon"), era[name], {})
    _nc(path, dict(time=1, lat=ny, lon=nx, level=L, level1=L + 1, soil1=len(era["soil1"])), v)


def write_delta(path, var, d, lat, lon):
    days = (d["time"] - np.datetime64("1850-01-01T00", "ns")) / np.timedelta64(1, "D")
    v = {"time": (("time",), days.astype(np.float64), {"units": "days since 1850-01-01 00:00:00", "calendar": "standard"}),
         "lat": (("lat",), lat, {}), "lon": (("lon",), lon, {})}
    dims = dict(time=len(days), lat=len(lat), lon=len(lon))
    if d["plev"] is not None:
        dims["plev"] = len(d["plev"])
        v["plev"] = (("plev",), d["plev"], {})
        v[var] = (("time", "plev", "lat", "lon"), d["data"], {})
    else:
        v[var] = (("time", "lat", "lon"), d["data"], {})
    _nc(path, dims, v)


def write_deltas(ddir, deltas, lat, lon, F):
    for name, d in deltas.items():
        var, base = ("ps", F.file_name_bases["HIST"]) if name == "ps_hist" else (name, F.file_name_bases["SCEN-HIST"])
        write_delta(os.path.join(ddir, base.format(var)), var, d, lat, lon)


def read_nc(path):
    out = {}
    with netcdf_file(path, "r", mmap=False) as f:
        for k, v in f.variables.items():
            a = np.array(v.data, copy=True)
            out[k] = a.astype(a.dtype.newbyteorder("="))
    return out


def capture(fn, *a, **kw):
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        r = fn(*a, **kw)
    return r, buf.getvalue()


def main(out=OUT):
    import warnings
    warnings.filterwarnings("ignore", message="no explicit representation of timezones")
    warnings.filterwarnings("ignore", category=DeprecationWarning)
    xr, F, S3 = import_reference()
    from pgw4era5_b200 import synthetic as S
    g = {}
    rng = np.random.default_rng(20261018)

    # ---------------------------------------------------------------- humidity with the alpha blend (functions.py:91-125)
    ta = xr.DataArray(np.array([200., 250.16, 250.17, 260., 273.15, 273.16, 273.17, 300.]).reshape(1, 8, 1, 1),
                      dims=("time", "level", "lat", "lon"))
    pa = xr.DataArray(np.linspace(2e3, 1e5, 8).reshape(1, 8, 1, 1), dims=("time", "level", "lat", "lon"))
    hus = xr.DataArray(np.geomspace(3e-6, 2e-2, 8).reshape(1, 8, 1, 1), dims=("time", "level", "lat", "lon"))
    g["hum_ta"], g["hum_pa"], g["hum_hus"] = ta.values, pa.values, hus.values
    g["hum_esat"] = F.saturation_vapor_pressure_water_and_ice(pa, ta).values
    hur = F.specific_to_relative_humidity(hus, pa, ta)
    g["hum_hur"] = hur.values
    g["hum_back"] = F.relative_to_specific_humidity(hur, pa, ta).values

    # ---------------------------------------------------------------- integ_geopot (functions.py:128-189)
    nl, ny, nx = 24, 3, 4
    ak, bk = S.hybrid_coefficients(nl)
    ps = rng.uniform(6.0e4, 1.04e5, (1, ny, nx))
    dims4 = ("time", "level1", "lat", "lon")
    co = dict(time=np.array([30.0]), lat=np.arange(ny, dtype=float), lon=np.arange(nx, dtype=float))
    level1 = xr.DataArray(np.arange(1, nl + 2, dtype=float), dims=("level1",), coords={"level1": np.arange(1, nl + 2, dtype=float)})
    pa_hl = xr.DataArray(ak[None, :, None, None] + ps[:, None] * bk[None, :, None, None], dims=dims4,
                         coords=dict(co, level1=np.arange(1, nl + 2, dtype=float)))
    co_f = dict(co, level=np.arange(1, nl + 1, dtype=float))
    t3 = xr.DataArray(rng.uniform(210., 300., (1, nl, ny, nx)), dims=("time", "level", "lat", "lon"), coords=co_f)
    q3 = xr.DataArray(rng.uniform(1e-6, 1.5e-2, (1, nl, ny, nx)), dims=("time", "level", "lat", "lon"), coords=co_f)
    zgs = xr.DataArray(rng.uniform(0., 3.0e4, (1, ny, nx)), dims=("time", "lat", "lon"), coords=co)
    g["ig_ak"], g["ig_bk"], g["ig_ps"] = ak, bk, ps
    g["ig_ta"], g["ig_hus"], g["ig_zgs"] = t3.values, q3.values, zgs.values
    for tag, p_ref in (("30000", 30000), ("50000", 50000.0)):
        g["ig_phi_" + tag] = F.integ_geopot(pa_hl, zgs, t3, q3, level1["level1"], p_ref).values
    pref_col = xr.DataArray(rng.choice([20000., 30000., 40000., 50000.], size=(1, ny, nx)), dims=("time", "lat", "lon"), coords=co)
    g["ig_pref_col"] = pref_col.values
    g["ig_phi_col"] = F.integ_geopot(pa_hl, zgs, t3, q3, level1["level1"], pref_col).values
    try:
        F.integ_geopot(pa_hl, zgs, t3, q3, level1["level1"], 104500.0)
        g["ig_below_sfc_raises"] = np.array(0)
    except ValueError as e:
        g["ig_below_sfc_raises"] = np.array(1)
        g["ig_below_sfc_msg"] = np.array(str(e))

    # ---------------------------------------------------------------- the per-timestep path on files
    when = datetime(2006, 8, 2, 6)
    ny, nx = 5, 6
    lat, lon = np.linspace(40.0, 70.0, ny), np.linspace(-10.0, 15.0, nx)
    era = S.to_numpy(S.make_era5(ny, nx, 77, lat=lat, lon=lon))
    deltas = S.to_numpy(S.make_deltas(S.make_era5(ny, nx, 77, lat=lat, lon=lon), 77))
    for k in ("ak", "bk", "soil1", "lat", "lon", "PS", "FIS", "T", "QV", "U", "V", "FR_LAND", "FR_SEA_ICE", "T_SKIN", "T_SO"):
        g["case_era_" + k] = era[k]
    for k, d in deltas.items():
        g["case_delta_" + k] = d["data"]
    g["case_delta_time"] = deltas["ta"]["time"].astype("datetime64[ns]").astype(np.int64)
    g["case_delta_plev"] = deltas["ta"]["plev"]
    g["case_when"] = np.array(when.isoformat())

    with tempfile.TemporaryDirectory() as tmp:
        ddir = os.path.join(tmp, "deltas")
        os.makedirs(ddir)
        inp = os.path.join(tmp, "era_in.nc")
        write_era(inp, era, when)
        write_deltas(ddir, deltas, lat, lon, F)
        era_ds = xr.open_dataset(inp, decode_cf=False)
        era_time = era_ds["time"]

        # ---- load_delta (functions.py:195-303): inside the year, both wraps, exact hit, no target
        dates = [datetime(2006, 8, 2, 6), datetime(2006, 1, 3, 0), datetime(2006, 12, 30, 18),
                 datetime(2006, 3, 16, 12), datetime(2008, 2, 29, 12)]
        g["ld_dates"] = np.array([d.isoformat() for d in dates])
        for i, d in enumerate(dates):
            r, _ = capture(F.load_delta, ddir, "ta", era_time, d)
            assert r.dims == ("time", "plev", "lat", "lon")
            g["ld_ta_%d" % i] = r.values
            r, _ = capture(F.load_delta, ddir, "tos", era_time, d)
            g["ld_tos_%d" % i] = r.values
        g["ld_ts_full"] = F.load_delta(ddir, "ts", era_time, None).values
        g["ld_ts_clim"] = F.load_delta(ddir, "ts", era_time, None).mean(dim=["time"]).values

        # ---- a DAILY delta series of a leap year (366 stamps): 29 February is dropped (:223-230), the other
        # stamps are moved to the target's year (:235-238); dates next to the gap and at both year ends
        ddir2 = os.path.join(tmp, "daily")
        os.makedirs(ddir2)
        stamps = np.datetime64("2000-01-01T12", "ns") + np.arange(366) * np.timedelta64(86400 * 10 ** 9, "ns")
        daily = (np.arange(366, dtype=np.float32)[:, None, None] + rng.normal(size=(366, 2, 3)).astype(np.float32))
        write_delta(os.path.join(ddir2, F.file_name_bases["SCEN-HIST"].format("tas")), "tas",
                    dict(time=stamps, plev=None, data=daily), np.arange(2.0), np.arange(3.0))
        ddates = [datetime(2006, 2, 28, 12), datetime(2006, 2, 28, 18), datetime(2006, 3, 1, 0), datetime(2006, 3, 1, 12),
                  datetime(2006, 1, 1, 0), datetime(2006, 12, 31, 18), datetime(2008, 2, 29, 6), datetime(2006, 7, 4, 3)]
        g["ldd_stamps"] = stamps.astype(np.int64)
        g["ldd_data"] = daily
        g["ldd_dates"] = np.array([d.isoformat() for d in ddates])
        for i, d in enumerate(ddates):
            r, _ = capture(F.load_delta, ddir2, "tas", era_time, d)
            g["ldd_out_%d" % i] = r.values
        g["ldd_full_len"] = np.array(F.load_delta(ddir2, "tas", era_time, None).shape[0])

        # ---- model-level pressure, vert_interp_delta / load_delta_interp (functions.py:306-431)
        akm = 0.5 * (era["ak"][1:] + era["ak"][:-1])
        bkm = 0.5 * (era["bk"][1:] + era["bk"][:-1])
        akm_da = xr.DataArray(akm, dims=("level",), coords={"level": era_ds["level"].values})
        bkm_da = xr.DataArray(bkm, dims=("level",), coords={"level": era_ds["level"].values})
        pa_era = (akm_da + era_ds["PS"] * bkm_da).transpose("time", "level", "lat", "lon")
        g["vi_pa_era"] = pa_era.values
        for var in ("ta", "hur", "ua", "va"):
            r, _ = capture(F.load_delta_interp, ddir, var, pa_era, era_time, when, True)
            assert r.dims == ("time", "level", "lat", "lon")
            g["vi_" + var] = r.values
        d_ta, _ = capture(F.load_delta, ddir, "ta", era_time, when)
        g["vi_ta_nosfc"] = F.vert_interp_delta(d_ta, pa_era, None, None, True).values
        try:
            F.vert_interp_delta(d_ta, pa_era, None, None, False)
            g["vi_top_raises"] = np.array(0)
        except ValueError:
            g["vi_top_raises"] = np.array(1)

        # ---- interp_logp_4d with linear extrapolation (functions.py:434-477)
        src_P = xr.DataArray(np.sort(rng.uniform(5e3, 9e4, (1, 6, ny, nx)), axis=1), dims=("time", "plev", "lat", "lon"))
        var_s = xr.DataArray(rng.normal(size=(1, 6, ny, nx)), dims=("time", "plev", "lat", "lon"))
        g["il_src_P"], g["il_var"] = src_P.values, var_s.values
        for mode in ("linear", "constant", "nan"):
            g["il_out_" + mode] = F.interp_logp_4d(var_s, src_P, pa_era, extrapolate=mode).values

        # ---- pgw_for_era5 (step_03_apply_to_era.py:44-381), three settings
        def run(tag, with_akm=False, ps_f64=False, **settings):
            old = {k: getattr(S3, k) for k in settings}
            for k, v in settings.items():
                setattr(S3, k, v)
            try:
                fin = os.path.join(tmp, "in_%s.nc" % tag)
                fout = os.path.join(tmp, "out_%s.nc" % tag)
                write_era(fin, era, when, with_akm, ps_f64)
                _, log = capture(S3.pgw_for_era5, fin, fout, ddir, when, True, None)
            finally:
                for k, v in old.items():
                    setattr(S3, k, v)
            errs = [float(m) for m in re.findall(r"### iteration \d+, phi max error: ([0-9.eE+-]+|nan)", log)]
            res = read_nc(fout)
            assert "RELHUM" not in res
            g["pgw_%s_n_iter" % tag] = np.array(len(errs))
            g["pgw_%s_errs" % tag] = np.array(errs)
            for k in ("PS", "T", "QV", "U", "V", "T_SKIN", "T_SO", "FR_SEA_ICE"):
                g["pgw_%s_%s" % (tag, k)] = res[k]
            print(tag, "iterations", len(errs), "last max error", errs[-1], "PS dtype", res["PS"].dtype, "T dtype", res["T"].dtype)

        # The reference inherits the dtypes of the ERA5 file in two places: ``delta_ps += adj_ps``
        # (step_03:194, xarray's in-place operators keep the dtype of zeros_like(PS)) and
        # ``phi_hl = zgs.expand_dims(...).copy()`` (functions.py:141, the half-level geopotential is stored
        # in the dtype of FIS).  With float32 PS/FIS -- what real ERA5 files hold -- the surface pressure of
        # every iteration is rounded to float32 (ulp 0.0078 Pa) and the geopotential sum is rounded to
        # float32 on every level (ulp 0.0078 m2/s2 at 300 hPa): its max error plateaus near 1e-2 m2/s2, so a
        # threshold of 1e-3 never converges.  With PS/FIS stored as double (same values) it is float64
        # throughout.  Both are recorded.
        run("default")
        run("akm", with_akm=True)
        run("default64", ps_f64=True)
        run("tight64", ps_f64=True, thresh_phi_ref_max_error=1e-3)
        run("pref_none64", ps_f64=True, p_ref_inp=None)
        run("reinterp64", ps_f64=True, i_reinterp=1)
        try:
            run("tight32", thresh_phi_ref_max_error=1e-3)
            g["pgw_tight32_raises"] = np.array(0)
        except ValueError as e:
            g["pgw_tight32_raises"] = np.array(1)
            print("tight32:", str(e)[:60])

    # ---------------------------------------------------------------- regrid_lat_lon (functions.py:748-898)
    with tempfile.TemporaryDirectory() as tmp:
        def gcm_file(path, glat, glon, data):
            _nc(path, dict(time=data.shape[0], plev=data.shape[1], lat=len(glat), lon=len(glon)),
                {"time": (("time",), np.arange(data.shape[0], dtype=np.float64) + 0.5,
                          {"units": "days since 2001-01-01 00:00:00", "calendar": "standard"}),
                 "plev": (("plev",), np.array([85000., 50000.])[:data.shape[1]], {}),
                 "lat": (("lat",), glat, {}), "lon": (("lon",), glon, {}),
                 "ta": (("time", "plev", "lat", "lon"), data, {})})

        def era_grid(path, tlat, tlon):
            _nc(path, dict(lat=len(tlat), lon=len(tlon)), {"lat": (("lat",), tlat, {}), "lon": (("lon",), tlon, {}),
                                                           "FIS": (("lat", "lon"), np.zeros((len(tlat), len(tlon)), np.float32), {})})
        cases = {
            # global 10 degree GCM grid, target reaches both poles (pole rows = zonal means) and wraps in longitude
            "glob": (np.linspace(-85., 85., 18), np.arange(5., 360., 10.), np.linspace(-90., 90., 37), np.arange(0., 360., 5.)),
            # latitudes stored north -> south (flipped by the reference), target inside
            "desc": (np.linspace(85., -85., 18), np.arange(5., 360., 10.), np.linspace(-60., 60., 25), np.arange(0., 360., 5.)),
            # target in -180..180 longitudes on a 0..360 GCM grid (periodic padding below)
            "west": (np.linspace(-85., 85., 18), np.arange(5., 360., 10.), np.linspace(30., 70., 9), np.linspace(-20., 40., 13)),
            # regional GCM grid (not periodic)
            "regio": (np.linspace(20., 80., 13), np.linspace(-30., 60., 19), np.linspace(30., 70., 9), np.linspace(-20., 40., 13)),
        }
        for tag, (glat, glon, tlat, tlon) in cases.items():
            data = rng.normal(size=(2, 2, len(glat), len(glon))).astype(np.float32)
            gcm_file(os.path.join(tmp, "g.nc"), glat, glon, data)
            era_grid(os.path.join(tmp, "e.nc"), tlat, tlon)
            ds_gcm, ds_era = xr.open_dataset(os.path.join(tmp, "g.nc")), xr.open_dataset(os.path.join(tmp, "e.nc"))
            r, _ = capture(F.regrid_lat_lon, ds_gcm, ds_era, "ta")
            assert r["ta"].dims == ("time", "plev", "lat", "lon")
            for k, v in (("glat", glat), ("glon", glon), ("tlat", tlat), ("tlon", tlon), ("in", data), ("out", r["ta"].values)):
                g["rg_%s_%s" % (tag, k)] = v
        # north -> south latitudes AND a target that reaches the poles: dlat_gcm is taken before the flip
        # (functions.py:776) and is negative, so no pole rows are added and the bounds check raises
        glat, glon = np.linspace(85., -85., 18), np.arange(5., 360., 10.)
        gcm_file(os.path.join(tmp, "gd.nc"), glat, glon, rng.normal(size=(1, 1, 18, 36)).astype(np.float32))
        era_grid(os.path.join(tmp, "ed.nc"), np.linspace(-90., 90., 37), np.arange(0., 360., 5.))
        try:
            capture(F.regrid_lat_lon, xr.open_dataset(os.path.join(tmp, "gd.nc")), xr.open_dataset(os.path.join(tmp, "ed.nc")), "ta")
            g["rg_desc_poles_raises"] = np.array(0)
        except ValueError:
            g["rg_desc_poles_raises"] = np.array(1)
        # a target outside a regional GCM grid raises (functions.py:845-856)
        era_grid(os.path.join(tmp, "e2.nc"), np.linspace(10., 70., 9), np.linspace(-20., 40., 13))
        try:
            capture(F.regrid_lat_lon, xr.open_dataset(os.path.join(tmp, "g.nc")), xr.open_dataset(os.path.join(tmp, "e2.nc")), "ta")
            g["rg_oob_raises"] = np.array(0)
        except ValueError:
            g["rg_oob_raises"] = np.array(1)

        # ------------------------------------------------------------ filter_data (functions.py:606-675)
        t = np.arange(1, 366)[:, None, None, None]
        raw = (1.0 + np.cos(2 * np.pi * t / 365) + 0.3 * rng.normal(size=(365, 2, 3, 4))).astype(np.float32)
        raw[:, 1, 2, 3] = np.nan
        raw[100, 0, 0, 0] = np.nan
        _nc(os.path.join(tmp, "raw.nc"), dict(time=365, plev=2, lat=3, lon=4),
            {"time": (("time",), np.arange(365, dtype=np.float64) + 0.5, {"units": "days since 2001-01-01 00:00:00", "calendar": "standard"}),
             "plev": (("plev",), np.array([85000., 50000.]), {}), "lat": (("lat",), np.arange(3.), {}), "lon": (("lon",), np.arange(4.), {}),
             "ta": (("time", "plev", "lat", "lon"), raw, {})})
        capture(F.filter_data, os.path.join(tmp, "raw.nc"), "ta", os.path.join(tmp, "smooth.nc"))
        g["fd_in"] = raw
        g["fd_out"] = read_nc(os.path.join(tmp, "smooth.nc"))["ta"]

    golden.save(out, g)
    print("wrote", out, len(g), "arrays", os.path.getsize(out), "bytes")


if __name__ == "__main__":
    main()

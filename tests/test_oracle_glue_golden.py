"""
The oracle against the UNMODIFIED reference executed in the build container, including its
xarray-bound functions and the whole of ``pgw_for_era5`` (tests/golden/reference_glue.npz, written by
oracle/make_golden_glue.py: the reference's functions.py and step_03_apply_to_era.py run over
oracle/xrlite.py, a restatement of the xarray semantics they rely on).  Tolerances are float64
round-off unless a comment says what else is in them.
"""
import os
from datetime import datetime

import numpy as np
import pytest

from oracle import pgw_oracle as O
from oracle.golden import load as load_golden

G = load_golden(os.path.join(os.path.dirname(__file__), "golden", "reference_glue.npz"))


def md(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    assert a.shape == b.shape, (a.shape, b.shape)
    assert np.array_equal(np.isnan(a), np.isnan(b)), "NaN pattern differs"
    return float(np.nanmax(np.abs(a - b))) if a.size else 0.0


def golden_case():
    """The inputs of the per-timestep goldens (5 x 6 columns, 137 levels, plev19 monthly deltas)."""
    era = {k[len("case_era_"):]: G[k] for k in G if k.startswith("case_era_")}
    times = G["case_delta_time"].astype("datetime64[ns]")
    deltas = {}
    for k in G:
        if k.startswith("case_delta_") and k not in ("case_delta_time", "case_delta_plev"):
            d = G[k]
            deltas[k[len("case_delta_"):]] = dict(time=times, data=d, plev=G["case_delta_plev"] if d.ndim == 4 else None)
    return era, deltas, datetime.fromisoformat(str(G["case_when"]))


def test_humidity_with_alpha_blend():
    """functions.py:91-125 on temperatures at and around both blend limits."""
    assert md(O.saturation_vapor_pressure_water_and_ice(G["hum_pa"], G["hum_ta"]), G["hum_esat"]) == 0.0
    hur = O.specific_to_relative_humidity(G["hum_hus"], G["hum_pa"], G["hum_ta"])
    assert md(hur, G["hum_hur"]) == 0.0
    assert md(O.relative_to_specific_humidity(hur, G["hum_pa"], G["hum_ta"]), G["hum_back"]) == 0.0


def test_integ_geopot():
    """functions.py:128-189 with a scalar and a per-column p_ref, and the all-NaN error path."""
    ak, bk, ps = G["ig_ak"], G["ig_bk"], G["ig_ps"]
    pa_hl = ak[None, :, None, None] + ps[:, None] * bk[None, :, None, None]
    for tag, p_ref in (("30000", 30000), ("50000", 50000.0), ("col", G["ig_pref_col"])):
        assert md(O.integ_geopot(pa_hl, G["ig_zgs"], G["ig_ta"], G["ig_hus"], p_ref), G["ig_phi_" + tag]) <= 1e-10
    assert int(G["ig_below_sfc_raises"]) == 1 and "below the surface" in str(G["ig_below_sfc_msg"])
    with pytest.raises(ValueError, match="below the surface"):
        O.integ_geopot(pa_hl, G["ig_zgs"], G["ig_ta"], G["ig_hus"], 104500.0)


def test_load_delta_calendar_logic():
    """functions.py:195-303: inside the year, both periodic wraps, an exact hit, a leap-day target."""
    era, deltas, _ = golden_case()
    for i, stamp in enumerate(G["ld_dates"]):
        d = datetime.fromisoformat(str(stamp))
        # the reference interpolates the float32 file values with scipy (difference taken in float32)
        assert md(O.load_delta(deltas["ta"], d), G["ld_ta_%d" % i]) <= 1e-6
        assert md(O.load_delta(deltas["tos"], d), G["ld_tos_%d" % i]) <= 1e-6
    assert md(O.load_delta(deltas["ts"], None), G["ld_ts_full"]) == 0.0
    # annual mean: float32 mean in the reference (:134-136)
    assert md(O.load_delta(deltas["ts"], None).mean(axis=0), G["ld_ts_clim"]) <= 2e-6


def test_vert_interp_delta_and_interp_logp_4d():
    """functions.py:306-477: surface-node replacement, axis flip, top check, all extrapolation modes."""
    era, deltas, when = golden_case()
    pa_era = G["vi_pa_era"]
    for var in ("ta", "hur", "ua", "va"):
        d = O.load_delta(deltas[var], when)
        sfc = (O.load_delta(deltas[var + "s"], when), O.load_delta(deltas["ps_hist"], when)) if var in ("ta", "hur") else (None, None)
        assert md(O.vert_interp_delta(d, deltas[var]["plev"], pa_era, sfc[0], sfc[1], True), G["vi_" + var]) <= 1e-6
    d = O.load_delta(deltas["ta"], when)
    assert md(O.vert_interp_delta(d, deltas["ta"]["plev"], pa_era, None, None, True), G["vi_ta_nosfc"]) <= 1e-6
    assert int(G["vi_top_raises"]) == 1
    with pytest.raises(ValueError, match="top pressure"):
        O.vert_interp_delta(d, deltas["ta"]["plev"], pa_era, None, None, False)
    for mode in ("linear", "constant", "nan"):
        assert md(O.interp_logp_4d(G["il_var"], G["il_src_P"], pa_era, mode), G["il_out_" + mode]) == 0.0


# what the reference writes as float32 (in-place updates of float32 file fields): half an ulp
F32_OUT = dict(T_SKIN=2e-5, T_SO=2e-5, FR_SEA_ICE=1e-7)


@pytest.mark.parametrize("tag,kw", [
    ("default", {}), ("akm", {}), ("default64", {}), ("tight64", dict(thresh_phi_ref_max_error=1e-3)),
    ("pref_none64", dict(p_ref_inp=None)), ("reinterp64", dict(i_reinterp=1))])
def test_pgw_for_era5_whole_path(tag, kw):
    """step_03_apply_to_era.py:44-381 end to end, dtype propagation of the file included:
    ``default``/``akm`` = all fields float32 as in a real ERA5 file, ``*64`` = PS and FIS stored as double."""
    era, deltas, when = golden_case()
    if tag.endswith("64"):
        era["PS"], era["FIS"] = era["PS"].astype(np.float64), era["FIS"].astype(np.float64)
    if tag == "akm":
        era["akm"], era["bkm"] = 0.5 * (era["ak"][1:] + era["ak"][:-1]), 0.5 * (era["bk"][1:] + era["bk"][:-1])
    r = O.pgw_for_era5(era, deltas, when, ignore_top_pressure_error=True, emulate_file_dtypes=True, **kw)
    assert r["n_iter"] == int(G["pgw_%s_n_iter" % tag])
    # the max geopotential error of every iteration, as printed by the reference
    np.testing.assert_allclose(r["phi_max_errors"], G["pgw_%s_errs" % tag], rtol=0, atol=1e-9)
    tol = dict(PS=1e-9, T=1e-9, QV=1e-13, U=1e-9, V=1e-9, **F32_OUT)
    if tag == "reinterp64":
        tol.update(U=5e-6, V=5e-6)     # the reference hands the float32 U, V to its numba kernel (difference in float32)
    for k, t in tol.items():
        assert md(r[k], G["pgw_%s_%s" % (tag, k)]) <= t, (k, md(r[k], G["pgw_%s_%s" % (tag, k)]))
    assert G["pgw_%s_PS" % tag].dtype == (np.float64 if tag.endswith("64") else np.float32)


def test_float32_files_cannot_meet_a_tight_threshold():
    """With float32 PS/FIS the reference rounds ps_pgw and the half-level geopotential to float32 in every
    iteration; its max error plateaus near 1e-2 m2/s2 and thresh 1e-3 ends in 'did not converge'."""
    assert int(G["pgw_tight32_raises"]) == 1
    era, deltas, when = golden_case()
    with pytest.raises(ValueError, match="did not converge"):
        O.pgw_for_era5(era, deltas, when, ignore_top_pressure_error=True, emulate_file_dtypes=True,
                       thresh_phi_ref_max_error=1e-3)
    # the exact-arithmetic model of the same inputs converges
    assert O.pgw_for_era5(era, deltas, when, ignore_top_pressure_error=True, thresh_phi_ref_max_error=1e-3)["n_iter"] == 8


def test_default_oracle_close_to_reference_on_float32_files():
    """The float64-PS/FIS model used by the GPU parity tests vs the reference on all-float32 files: the
    difference is the reference's own float32 rounding noise (ps ~3e-2 Pa), the iteration count agrees."""
    era, deltas, when = golden_case()
    r = O.pgw_for_era5(era, deltas, when, ignore_top_pressure_error=True)
    assert r["n_iter"] == int(G["pgw_default_n_iter"])
    assert md(r["PS"], G["pgw_default_PS"]) <= 5e-2
    assert md(r["T"], G["pgw_default_T"]) <= 1e-9 and md(r["QV"], G["pgw_default_QV"]) <= 1e-7
    assert np.max(np.abs(np.array(r["phi_max_errors"]) - G["pgw_default_errs"])) <= 3e-2


def test_regrid_lat_lon():
    """functions.py:748-898: pole rows, periodic padding for -180..180 targets, flipped latitudes, errors."""
    for tag in ("glob", "desc", "west", "regio"):
        r = O.regrid_lat_lon(G["rg_%s_in" % tag], G["rg_%s_glat" % tag], G["rg_%s_glon" % tag],
                             G["rg_%s_tlat" % tag], G["rg_%s_tlon" % tag])
        # pole rows: zonal mean of float32 values taken in float32 by the reference
        assert md(r, G["rg_%s_out" % tag]) <= (1e-7 if tag == "glob" else 1e-12), tag
    assert int(G["rg_oob_raises"]) == 1 and int(G["rg_desc_poles_raises"]) == 1
    with pytest.raises(ValueError, match="North or South"):
        O.regrid_lat_lon(G["rg_regio_in"], G["rg_regio_glat"], G["rg_regio_glon"], np.linspace(10., 70., 9), G["rg_regio_tlon"])
    # latitudes stored north -> south and a target that reaches the poles: dlat is taken before the flip
    with pytest.raises(ValueError, match="North or South"):
        O.regrid_lat_lon(np.zeros((1, 18, 36)), np.linspace(85., -85., 18), np.arange(5., 360., 10.),
                         np.linspace(-90., 90., 37), np.arange(0., 360., 5.))


def test_filter_data():
    """functions.py:606-675 (the result is written back into the float32 array of the file)."""
    assert md(O.filter_data(G["fd_in"]), G["fd_out"]) <= 5e-7


def test_daily_series_with_leap_day():
    """load_delta on a 366-stamp daily series (functions.py:223-292): 29 February dropped, dates right next to
    the gap, both year wraps, a leap-day target -- the oracle and the product's host-side bracket logic
    (pgw4era5_b200/timeinterp.py, whose blend runs on the GPU) against the executed reference."""
    from pgw4era5_b200 import timeinterp as TI
    stamps = G["ldd_stamps"].astype("datetime64[ns]")
    data = G["ldd_data"]
    assert int(G["ldd_full_len"]) == 365
    kept = TI.drop_leap_day(stamps)
    assert len(kept) == 365 and 59 not in kept
    delta = dict(time=stamps, data=data, plev=None)
    for i, stamp in enumerate(G["ldd_dates"]):
        when = datetime.fromisoformat(str(stamp))
        want = G["ldd_out_%d" % i]
        assert md(O.load_delta(delta, when), want) <= 1e-4, stamp
        b = TI.bracket(stamps[kept], when)
        lo, hi = data[kept][b.ind_before].astype(np.float64), data[kept][b.ind_after].astype(np.float64)
        got = lo if b.exact else (hi - lo) / b.x_hi * b.x_new + lo
        assert md(got[None], want) <= 1e-4, stamp
    # 28 Feb 18:00 lies between 28 Feb 12:00 and 1 Mar 12:00: a quarter of the way across the dropped day
    b = TI.bracket(stamps[kept], datetime(2006, 2, 28, 18))
    assert (b.ind_before, b.ind_after) == (58, 59) and abs(b.x_new / b.x_hi - 0.25) < 1e-12

"""Parity of the stand-alone operators (functions.py drop-in, through the C ABI) against the
golden vectors of the reference and against the fp64 oracle."""
import numpy as np
import pytest

from oracle import pgw_oracle as O
from oracle.golden import load as load_golden

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def F():
    from pgw4era5_b200 import functions
    return functions


@pytest.mark.parametrize("mode", ["linear", "constant", "nan"])
def test_interp_extrap_1d_golden(F, golden, mode):
    out = F.interp_extrap_1d(golden["ie1_src_x"], golden["ie1_src_y"], golden["ie1_targ_x"], mode)
    np.testing.assert_allclose(out, golden["ie1_out_" + mode], rtol=0, atol=1e-14, equal_nan=True)


def test_interp_extrap_1d_off(F, golden):
    out = F.interp_extrap_1d(golden["ie1_src_x"], golden["ie1_src_y"], golden["ie1_targ_inner"], "off")
    np.testing.assert_allclose(out, golden["ie1_out_off_inner"], rtol=0, atol=1e-14)
    with pytest.raises(ValueError, match="Extrapolation deactivated"):
        F.interp_extrap_1d(golden["ie1_src_x"], golden["ie1_src_y"], golden["ie1_targ_x"], "off")


@pytest.mark.parametrize("mode", ["linear", "constant", "nan"])
def test_interp_1d_for_timelatlon_golden(F, golden, mode):
    sp, tp, val = golden["i4_src_p"], golden["i4_targ_p"], golden["i4_val"]
    out = np.zeros_like(tp)
    F.interp_1d_for_timelatlon(val, sp, tp, out, tp.shape[0], tp.shape[2], tp.shape[3], mode)
    ref = golden["i4_out_" + mode]
    np.testing.assert_array_equal(np.isnan(out), np.isnan(ref))
    np.testing.assert_allclose(out, ref, rtol=0, atol=1e-13, equal_nan=True)      # float64, same formula


def test_interp_errors(F, golden):
    sp, tp, val = golden["i4_src_p"], golden["i4_targ_p"], golden["i4_val"]
    out = np.zeros_like(tp)
    with pytest.raises(ValueError, match="Source pressure"):
        F.interp_1d_for_timelatlon(val, np.ascontiguousarray(sp[:, ::-1]), tp, out, 2, 5, 6, "constant")
    with pytest.raises(ValueError, match="Target pressure"):
        F.interp_1d_for_timelatlon(val, sp, np.ascontiguousarray(tp[:, ::-1]), out, 2, 5, 6, "constant")
    with pytest.raises(ValueError, match="Invalid input"):
        F.interp_logp_4d(val, np.exp(sp), np.exp(tp), extrapolate="bogus")
    with pytest.raises(ValueError, match="Lat dimension"):
        F.interp_logp_4d(val, np.exp(sp), np.exp(tp)[:, :, :4], extrapolate="constant")


@pytest.mark.parametrize("dtype,tol", [(np.float64, 1e-12), (np.float32, 1e-4)])
def test_interp_logp_4d_vs_oracle(F, dtype, tol):
    from pgw4era5_b200 import synthetic as S
    rng = np.random.default_rng(5)
    nt, ks, kt, ny, nx = 1, 19, 137, 9, 33
    # source: plev19 jittered per column; target: hybrid model levels for random surface pressures
    sp = np.sort(S.PLEV19[None, :, None, None] * rng.uniform(0.97, 1.03, (nt, ks, ny, nx)), axis=1)
    ak, bk = S.hybrid_coefficients()
    akm, bkm = 0.5 * (ak[1:] + ak[:-1]), 0.5 * (bk[1:] + bk[:-1])
    tp = akm[None, :, None, None] + rng.uniform(6e4, 1.05e5, (nt, 1, ny, nx)) * bkm[None, :, None, None]
    val = rng.normal(size=(nt, ks, ny, nx))
    ref = O.interp_logp_4d(val.astype(dtype), sp.astype(dtype), tp.astype(dtype), "constant")
    out = F.interp_logp_4d(val.astype(dtype), sp.astype(dtype), tp.astype(dtype), "constant")
    assert out.dtype == dtype
    np.testing.assert_allclose(out, ref, rtol=0, atol=tol)
    # 1-D pressure-level table shared by all columns
    plev = np.sort(rng.uniform(100., 1.0e5, ks))
    ref1 = O.interp_logp_4d(val, np.broadcast_to(plev[None, :, None, None], val.shape).copy(), tp, "linear")
    out1 = F.interp_logp_4d(val, plev, tp, "linear")
    np.testing.assert_allclose(out1, ref1, rtol=0, atol=1e-11)


def test_humidity_golden_and_oracle(F, golden):
    hus, pa, ta = golden["hum_hus"], golden["hum_pa"], golden["hum_ta"]
    np.testing.assert_allclose(F.specific_humidity_to_vapor_pressure(hus, pa), golden["hum_e"], rtol=1e-15)
    np.testing.assert_allclose(F.vapor_pressure_to_specific_humidity(golden["hum_e"], pa), golden["hum_q"], rtol=1e-15)
    np.testing.assert_allclose(F.saturation_vapor_pressure_water_or_ice(pa, ta, True), golden["hum_esw"], rtol=1e-14)
    np.testing.assert_allclose(F.saturation_vapor_pressure_water_or_ice(pa, ta, False), golden["hum_esi"], rtol=1e-14)
    ta2 = np.concatenate([ta, [250.16, 273.16, 260.0, np.nan]])
    np.testing.assert_allclose(F.saturation_vapor_pressure_water_and_ice(None, ta2),
                               O.saturation_vapor_pressure_water_and_ice(None, ta2), rtol=1e-14, equal_nan=True)
    rh = O.specific_to_relative_humidity(hus, pa, ta)
    np.testing.assert_allclose(F.specific_to_relative_humidity(hus, pa, ta), rh, rtol=1e-13)
    np.testing.assert_allclose(F.relative_to_specific_humidity(rh, pa, ta), hus, rtol=1e-12)
    f32 = F.specific_to_relative_humidity(hus.astype(np.float32), pa.astype(np.float32), ta.astype(np.float32))
    assert f32.dtype == np.float32
    np.testing.assert_allclose(f32, rh, rtol=2e-5)


def test_integ_geopot_vs_oracle(F):
    from pgw4era5_b200 import synthetic as S
    era = S.to_numpy(S.make_era5(6, 20, 31))
    ak, bk = era["ak"], era["bk"]
    pa_hl = ak[None, :, None, None] + era["PS"].astype(np.float64)[:, None] * bk[None, :, None, None]
    fis, T64, Q64 = era["FIS"].astype(np.float64), era["T"].astype(np.float64), era["QV"].astype(np.float64)
    pref = np.where(era["PS"] > 90000, 50000.0, 30000.0)
    for p_ref in (30000.0, pref):
        # all float64, and float32 T/QV with float64 pressures (Rd * Tv in float32, like numpy in the reference)
        np.testing.assert_allclose(F.integ_geopot(pa_hl, fis, T64, Q64, None, p_ref),
                                   O.integ_geopot(pa_hl, fis, T64, Q64, p_ref), rtol=0, atol=1e-8)
        np.testing.assert_allclose(F.integ_geopot(pa_hl, fis, era["T"], era["QV"], None, p_ref),
                                   O.integ_geopot(pa_hl, fis, era["T"], era["QV"], p_ref), rtol=0, atol=1e-8)
    d = np.abs(O.integ_geopot(pa_hl, fis, era["T"], era["QV"], 30000.0) - O.integ_geopot(pa_hl, fis, T64, Q64, 30000.0))
    assert 1e-5 < d.max() < 2e-2                      # the two really differ
    with pytest.raises(ValueError, match="below the surface"):
        F.integ_geopot(pa_hl, fis, T64, Q64, None, 120000.0)


def test_integ_geopot_vs_executed_reference(F):
    """functions.py:128-189 run unmodified over oracle/xrlite.py (tests/golden/reference_glue.npz)."""
    import os
    G = load_golden(os.path.join(os.path.dirname(__file__), "golden", "reference_glue.npz"))
    ak, bk, ps = G["ig_ak"], G["ig_bk"], G["ig_ps"]
    pa_hl = ak[None, :, None, None] + ps[:, None] * bk[None, :, None, None]
    for tag, p_ref in (("30000", 30000), ("50000", 50000.0), ("col", G["ig_pref_col"])):
        out = F.integ_geopot(pa_hl, G["ig_zgs"], G["ig_ta"], G["ig_hus"], None, p_ref)
        np.testing.assert_allclose(out, G["ig_phi_" + tag], rtol=0, atol=1e-8)


def test_integrate_tos_golden(F, golden):
    out = F.integrate_tos(golden["it_tos"], golden["it_ts"], golden["it_land"], golden["it_ice"])
    np.testing.assert_allclose(out, golden["it_out"], rtol=0, atol=1e-15)
    small = F.integrate_tos(np.array([[1., np.nan]]), np.array([[2., 3.]]), np.array([[.2, .5]]), np.array([[.1, 0.]]))
    np.testing.assert_allclose(small, [[1.3, 3.0]], rtol=0, atol=1e-15)


def test_replace_delta_sfc_golden(F, golden):
    plev = golden["rds_plev"]
    delta = np.arange(19.)
    for i, ph in enumerate(golden["rds_ps_hist"]):
        P, D = F.replace_delta_sfc(plev, ph, delta, 99.0)
        np.testing.assert_array_equal(P, golden["rds_P_%d" % i])
        np.testing.assert_array_equal(D, golden["rds_D_%d" % i])
    for bad in (50.0, 100.0, np.nan):
        with pytest.raises(ValueError):
            F.replace_delta_sfc(plev, bad, delta, 99.0)


def test_vert_interp_delta_vs_oracle(F):
    from pgw4era5_b200 import synthetic as S
    from cases import make_case, ERA_DATE
    era, deltas = make_case(7, 21, 41)
    e, d = S.to_numpy(era), S.to_numpy(deltas)
    pa = e["akm"][None, :, None, None] + e["PS"].astype(np.float64)[:, None] * e["bkm"][None, :, None, None]
    ta = O.load_delta(d["ta"], ERA_DATE); tas = O.load_delta(d["tas"], ERA_DATE); psh = O.load_delta(d["ps_hist"], ERA_DATE)
    ref = O.vert_interp_delta(ta, d["ta"]["plev"], pa, tas, psh, True)
    out = F.vert_interp_delta(ta, pa, tas, psh, True, plev=d["ta"]["plev"])
    np.testing.assert_allclose(out, ref, rtol=0, atol=1e-11)
    ref2 = O.vert_interp_delta(ta, d["ta"]["plev"], pa, None, None, True)
    np.testing.assert_allclose(F.vert_interp_delta(ta, pa, None, None, True, plev=d["ta"]["plev"]), ref2, rtol=0, atol=1e-11)
    with pytest.raises(ValueError, match="top pressure"):
        F.vert_interp_delta(ta, pa, tas, psh, False, plev=d["ta"]["plev"])


def test_smoothing_vs_oracle_and_golden(F, golden):
    np.testing.assert_allclose(F.harmonic_ac_analysis(golden["hac_in"]), golden["hac_out"], rtol=0, atol=2e-6)
    rng = np.random.default_rng(8)
    x = (rng.normal(size=(365, 3, 5, 7)) + 3.0).astype(np.float32)
    x[:, 1, 2, 3] = np.nan
    x[17, 0, 0, 0] = np.nan
    ref = O.filter_data_fast(x)
    out = F.smooth_annual_cycle(x)
    assert out.dtype == np.float32
    np.testing.assert_array_equal(np.isnan(out), np.isnan(ref))
    np.testing.assert_allclose(out, ref, rtol=0, atol=2e-6, equal_nan=True)
    x12 = rng.normal(size=(12, 4, 6)).astype(np.float32)
    np.testing.assert_allclose(F.smooth_annual_cycle(x12), O.filter_data(x12), rtol=0, atol=2e-6)


@pytest.mark.parametrize("case", range(4))
def test_regrid_vs_oracle(F, case):
    from test_abi_and_host import GRID_CASES
    lat, lon, tlat, tlon = GRID_CASES[case]
    rng = np.random.default_rng(10 + case)
    data = rng.normal(size=(3, 2, len(lat), len(lon))).astype(np.float32)
    ref = O.regrid_lat_lon(data, lat, lon, tlat, tlon)
    out = F.regrid_arrays(data, lat, lon, tlat, tlon)
    assert out.shape == ref.shape and out.dtype == np.float32
    np.testing.assert_allclose(out, ref, rtol=0, atol=5e-7)


def test_regrid_identity_and_pole_rows(F):
    lat, lon = np.linspace(-88, 88, 45), np.arange(0.0, 360, 4.0)
    rng = np.random.default_rng(12)
    data = rng.normal(size=(2, len(lat), len(lon))).astype(np.float32)
    same = F.regrid_arrays(data, lat, lon, lat, lon)
    np.testing.assert_allclose(same, data, rtol=0, atol=1e-6)                      # identical grids -> identity
    poles = F.regrid_arrays(data, lat, lon, np.array([-90.0, 90.0]), lon)
    np.testing.assert_allclose(poles[:, 0], np.repeat(data[:, 0].mean(-1, keepdims=True), len(lon), -1), atol=1e-6)
    np.testing.assert_allclose(poles[:, 1], np.repeat(data[:, -1].mean(-1, keepdims=True), len(lon), -1), atol=1e-6)


def test_byteswap32():
    """pgw_byteswap32: the big-endian float32 words of a NetCDF-3 file, swapped in place on the device."""
    import ctypes as C
    import torch
    from pgw4era5_b200 import _native as N
    rng = np.random.default_rng(11)
    for n in (1, 3, 4, 1023, 4096 + 5):
        x = rng.normal(size=n).astype(np.float32)
        d = torch.from_numpy(x.astype(">f4").view(np.float32).copy()).cuda()
        N.check(N.lib.pgw_byteswap32(C.c_void_p(d.data_ptr()), n, C.c_void_p(torch.cuda.current_stream().cuda_stream)),
                "pgw_byteswap32")
        np.testing.assert_array_equal(d.cpu().numpy(), x)


def _regrid_with(path, F, *args, **kw):
    import os
    old = os.environ.get("PGW_REGRID_PATH")
    if path:
        os.environ["PGW_REGRID_PATH"] = path
    try:
        return F.regrid_arrays(*args, **kw)
    finally:
        if old is None:
            os.environ.pop("PGW_REGRID_PATH", None)
        else:
            os.environ["PGW_REGRID_PATH"] = old


@pytest.mark.parametrize("case", ["era_quarter", "flipped_irregular", "odd_nx", "many_source_rows"])
def test_regrid_walk_kernel_bit_identical_and_banded(F, case):
    """The walking kernel (source rows staged per chunk of target rows, three-column pattern) against the older
    row and generic kernels -- same expressions, bit-identical -- and against the oracle; target-latitude bands
    (SURVEY 8e row 3) concatenate to the whole field bit for bit, for band edges that cut chunks and row pairs."""
    rng = np.random.default_rng(31)
    if case == "era_quarter":               # 1 degree -> 0.25 degree incl. both poles: the regular 4:1 pattern
        lat, lon = np.linspace(-89.5, 89.5, 180), 0.5 + np.arange(360)
        tlat, tlon = np.linspace(-90, 90, 721), 0.25 * np.arange(1440)
        lead = (3,)
    elif case == "flipped_irregular":       # north-to-south source, irregular longitudes: no three-column pattern
        lat = np.linspace(80, -80, 41)
        lon = np.sort(rng.uniform(0, 360, 97))
        tlat, tlon = np.linspace(-75, 75, 61), np.linspace(lon[0] + 0.1, lon[-1] - 0.1, 200)
        lead = (2, 3)
    elif case == "odd_nx":                  # target width not a multiple of 4: scalar stores
        lat, lon = np.linspace(-60, 60, 25), np.linspace(0, 100, 41)
        tlat, tlon = np.linspace(-50, 50, 33), np.linspace(5, 95, 123)
        lead = (4,)
    else:                                   # finer source than target: a chunk spans more source rows than are staged
        lat, lon = np.linspace(-80, 80, 321), np.linspace(0, 357, 120)
        tlat, tlon = np.linspace(-70, 70, 29), np.linspace(1, 350, 64)
        lead = (2,)
    data = rng.normal(size=lead + (len(lat), len(lon))).astype(np.float32)
    walk = _regrid_with(None, F, data, lat, lon, tlat, tlon)
    rows = _regrid_with("rows", F, data, lat, lon, tlat, tlon)
    gen = _regrid_with("generic", F, data, lat, lon, tlat, tlon)
    np.testing.assert_array_equal(walk, gen)
    np.testing.assert_array_equal(rows, gen)
    ref = O.regrid_lat_lon(data, lat, lon, tlat, tlon)
    np.testing.assert_allclose(walk, ref, rtol=0, atol=5e-7)
    ny_t = len(tlat)
    for bounds in ([0, 7, 8, 21, ny_t], [0, ny_t // 3, ny_t - 1, ny_t]):
        parts = [F.regrid_arrays(data, lat, lon, tlat, tlon, rows=(a, b)) for a, b in zip(bounds[:-1], bounds[1:])]
        np.testing.assert_array_equal(np.concatenate(parts, axis=-2), walk)
    with pytest.raises(ValueError):
        F.regrid_arrays(data, lat, lon, tlat, tlon, rows=(5, ny_t + 1))

"""Parity of the fused CUDA timestep (through the C ABI) against the fp64 oracle."""
import numpy as np
import pytest
import torch

from cases import ERA_DATE, TOL, compare, make_case, run_oracle

pytestmark = pytest.mark.gpu


def _engine(era, deltas):
    from pgw4era5_b200.engine import DeltaSet, PGWEngine
    ds = DeltaSet(deltas, device="cuda")
    return PGWEngine(era["ak"], era["bk"], ds, soil1=era["soil1"])


def _dev(era):
    return {k: (v.cuda() if isinstance(v, torch.Tensor) else v) for k, v in era.items()}


@pytest.mark.parametrize("ny,nx,seed", [(24, 40, 1), (33, 129, 2), (7, 31, 3)])
def test_timestep_matches_oracle(ny, nx, seed):
    era, deltas = make_case(ny, nx, seed)
    ref = run_oracle(era, deltas)
    eng = _engine(era, deltas)
    res = eng.apply(_dev(era), ERA_DATE, ignore_top_pressure_error=True)
    assert res["n_iter"] == ref["n_iter"]
    np.testing.assert_allclose(res["phi_max_errors"], ref["phi_max_errors"], rtol=0, atol=1e-3)
    errs = compare(res, ref)
    for name, e in errs.items():
        assert e <= TOL[name], (name, e, errs)


@pytest.mark.parametrize("k_spec", [3, 5, 9, 19])
def test_speculation_paths_agree(k_spec):
    """rerun (k_spec too small), exact hit and rewrite (k_spec too large) give the same fields."""
    era, deltas = make_case(24, 40, 1)
    ref = run_oracle(era, deltas)
    eng = _engine(era, deltas)
    res = eng.apply(_dev(era), ERA_DATE, ignore_top_pressure_error=True, k_spec=k_spec)
    assert res["n_iter"] == ref["n_iter"]
    errs = compare(res, ref)
    for name, e in errs.items():
        assert e <= TOL[name], (name, e, errs)


def _apply(era, deltas, when=ERA_DATE, ignore_top=True, **kw):
    eng = _engine(era, deltas)
    return eng.apply(_dev(era), when, ignore_top_pressure_error=ignore_top, **kw), eng


def _check(res, ref):
    assert res["n_iter"] == ref["n_iter"], (res["phi_max_errors"], ref["phi_max_errors"])
    errs = compare(res, ref)
    for name, e in errs.items():
        assert e <= TOL[name], (name, e, errs)
    return errs


def test_config1_european_domain():
    """BASELINE configs[0]: 201x281 European subdomain, 137 levels, plev19, one timestep."""
    era, deltas = make_case(201, 281, 1)
    ref = run_oracle(era, deltas)
    res, _ = _apply(era, deltas)
    _check(res, ref)
    # iteration-count margin of this seed: |E_N - thresh| must dwarf the fp32 storage noise
    assert abs(ref["phi_max_errors"][-1] - 0.15) > 1e-3 * 0.15


def test_config5_plev37_tight_threshold():
    """BASELINE configs[4] (small grid): 37 pressure levels and thresh 1e-3 -> ~10 iterations."""
    from pgw4era5_b200 import settings, synthetic as S
    era, deltas = make_case(19, 47, 5, plev=S.PLEV37, region="GL")
    ref = run_oracle(era, deltas, thresh_phi_ref_max_error=1e-3)
    old = settings.thresh_phi_ref_max_error
    settings.thresh_phi_ref_max_error = 1e-3
    try:
        res, _ = _apply(era, deltas)
    finally:
        settings.thresh_phi_ref_max_error = old
    assert ref["n_iter"] >= 8
    _check(res, ref)


@pytest.mark.parametrize("when", ["2006-03-16T12", "2006-01-01T00", "2006-12-31T18", "2008-02-29T06"])
def test_time_interpolation_cases(when):
    """exact hit on a delta stamp, the two year wraps, and a leap day (functions.py:242-292)."""
    from datetime import datetime
    when = datetime.fromisoformat(when)
    era, deltas = make_case(9, 33, 7)
    ref = run_oracle(era, deltas, when=when)
    res, _ = _apply(era, deltas, when=when)
    _check(res, ref)


def test_zero_deltas_identity():
    era, deltas = make_case(12, 40, 21)
    for v in deltas.values():
        v["data"].zero_()
    deltas["ps_hist"]["data"] += era["PS"]
    res, _ = _apply(era, deltas)
    assert res["n_iter"] == 1
    for name in ("T", "U", "V", "PS", "T_SKIN", "T_SO"):
        assert torch.equal(res[name].cpu().reshape(-1), era[name].reshape(-1)), name
    assert float(res["delta_ps"].abs().max()) == 0.0
    q = res["QV"].cpu().reshape(-1).double(); q0 = era["QV"].reshape(-1).double()
    assert float(((q - q0).abs() / q0).max()) < 5e-6                    # rh -> q round trip in fp32


def test_nan_handling_matches_oracle():
    """NaN sea ice over land and NaN tos pass through exactly like the reference
    (np.clip keeps NaN, integrate_tos masks them, step_03:103-125)."""
    era, deltas = make_case(10, 36, 9, region="GL")
    assert torch.isnan(era["FR_SEA_ICE"]).any() and torch.isnan(deltas["tos"]["data"]).any()
    ref = run_oracle(era, deltas)
    res, _ = _apply(era, deltas)
    _check(res, ref)


def test_errors_match_reference():
    from pgw4era5_b200 import settings
    era, deltas = make_case(8, 33, 23)
    with pytest.raises(ValueError, match="top pressure"):                  # functions.py:417-425
        _apply(era, deltas, ignore_top=False)
    old = settings.max_n_iter
    settings.max_n_iter = 3
    try:
        with pytest.raises(ValueError, match="did not converge"):           # step_03:315-319
            _apply(era, deltas)
    finally:
        settings.max_n_iter = old
    old = settings.p_ref_inp
    settings.p_ref_inp = 100000
    try:
        with pytest.raises(ValueError, match="below the surface"):          # functions.py:162-165
            _apply(era, deltas)
    finally:
        settings.p_ref_inp = old
    bad = {k: dict(v) for k, v in deltas.items()}
    bad["ps_hist"] = dict(deltas["ps_hist"], data=deltas["ps_hist"]["data"] * 0 + 50.0)
    with pytest.raises(ValueError):                                         # functions.py:360-361
        _apply(era, bad)
    old = settings.p_ref_inp
    settings.p_ref_inp = 31000
    try:
        with pytest.raises(KeyError):                                       # .sel(plev=p_ref), step_03:294
            _apply(era, deltas)
    finally:
        settings.p_ref_inp = old


def test_ps_bound_rerun():
    """A stash sized for a too small ps bound is detected on the device and the step is rerun."""
    era, deltas = make_case(8, 33, 2)
    ref = run_oracle(era, deltas)
    from pgw4era5_b200.engine import DeltaSet, PGWEngine
    eng = PGWEngine(era["ak"], era["bk"], DeltaSet(deltas, device="cuda"), soil1=era["soil1"], ps_bound=60000.0)
    res = eng.apply(_dev(era), ERA_DATE, ignore_top_pressure_error=True)
    assert eng.stats["reruns"] >= 1 and eng.ps_bound > 100000
    _check(res, ref)


def test_global_size_properties():
    """BASELINE configs[1] at full size (721x1440x137): properties that need no oracle run.
    (a) zero deltas: one iteration, T/U/V/PS bit-identical; (b) the fused pass agrees with the
    stand-alone operators on a latitude band; (c) result is independent of k_spec."""
    from pgw4era5_b200 import synthetic as S
    from pgw4era5_b200.engine import DeltaSet, PGWEngine
    ny, nx = 721, 1440
    era = S.make_era5(ny, nx, 2, device="cuda", orog_seed=2)
    deltas = S.make_deltas(era, 2, device="cuda")
    eng = PGWEngine(era["ak"], era["bk"], DeltaSet(deltas, device="cuda"), soil1=era["soil1"])
    r1 = eng.apply(era, ERA_DATE, ignore_top_pressure_error=True)
    n1 = r1["n_iter"]
    ps1, q1 = r1["PS"].clone(), r1["QV"].clone()
    r2 = eng.apply(era, ERA_DATE, ignore_top_pressure_error=True, k_spec=n1 + 3)      # rewrite path
    assert r2["n_iter"] == n1
    assert float((r2["PS"] - ps1).abs().max()) <= 1e-2
    assert float((r2["QV"] - q1).abs().max()) <= 1e-7
    assert 4 <= n1 <= 10 and r1["phi_max_errors"][-1] <= 0.15 < r1["phi_max_errors"][-2]
    # band check against the oracle (rows 300..303)
    band = slice(300, 304)
    sub = {k: (v[..., band, :].cpu() if isinstance(v, torch.Tensor) and v.dim() >= 3 else v) for k, v in era.items()}
    subd = {k: dict(v, data=v["data"][..., band, :].cpu()) for k, v in deltas.items()}
    ref = run_oracle(sub, subd)
    for name, tol in (("T", 1e-4), ("U", 1e-4), ("V", 1e-4)):
        g = r1[name][..., band, :].cpu().numpy().astype(np.float64)
        assert np.max(np.abs(g - ref[name])) <= tol, name
    # zero deltas
    for v in deltas.values():
        v["data"].zero_()
    deltas["ps_hist"]["data"] += era["PS"]
    eng0 = PGWEngine(era["ak"], era["bk"], DeltaSet(deltas, device="cuda"), soil1=era["soil1"])
    r0 = eng0.apply(era, ERA_DATE, ignore_top_pressure_error=True)
    assert r0["n_iter"] == 1
    for name in ("T", "U", "V", "PS"):
        assert torch.equal(r0[name].reshape(-1), era[name].reshape(-1)), name


def _uses_tma(eng, era):
    """Which flavour of the column kernel pgw_timestep() picked for the last submit."""
    import ctypes as C
    from pgw4era5_b200 import _native as N
    p = eng.submit(_dev(era), ERA_DATE, ignore_top_pressure_error=True)
    flag = N.lib.pgw_timestep_uses_tma(C.byref(p.args))
    p.result()
    return flag


@pytest.mark.parametrize("ny,nx,seed", [(24, 40, 1), (16, 64, 11), (12, 44, 7)])
def test_tma_and_generic_flavours_agree(ny, nx, seed, monkeypatch):
    """ncol % 4 == 0 -> TMA flavour (incl. a partial last CTA); PGW_COLUMN_PATH=generic forces the
    per-thread cp.async flavour.  Same arithmetic up to fma contraction (and one more parked
    level), so the fields agree to rounding, and both must match the oracle."""
    era, deltas = make_case(ny, nx, seed)
    ref = run_oracle(era, deltas)
    eng = _engine(era, deltas)
    monkeypatch.delenv("PGW_COLUMN_PATH", raising=False)
    assert _uses_tma(eng, era) == 1
    res_t = eng.apply(_dev(era), ERA_DATE, ignore_top_pressure_error=True)
    monkeypatch.setenv("PGW_COLUMN_PATH", "generic")
    assert _uses_tma(eng, era) == 0
    res_g = eng.apply(_dev(era), ERA_DATE, ignore_top_pressure_error=True)
    _check(res_t, ref)
    _check(res_g, ref)
    assert res_t["n_iter"] == res_g["n_iter"]
    for name in ("T", "U", "V", "T_SKIN", "T_SO", "FR_SEA_ICE"):
        assert torch.equal(res_t[name].view(torch.int32), res_g[name].view(torch.int32)), name
    assert float((res_t["PS"] - res_g["PS"]).abs().max()) <= 1e-5 * 1e5 * 2 ** -23 * 4     # few fp32 ulps of ps
    assert float((res_t["QV"] - res_g["QV"]).abs().max()) <= 1e-9
    # the TMA flavour sums the layers below p_ref through a polynomial in dps (truncation + fp32 humidity
    # coefficients: a few 1e-7 m2/s2), the cp.async flavour integrates every level in every iteration
    np.testing.assert_allclose(res_t["phi_max_errors"], res_g["phi_max_errors"], rtol=0, atol=5e-6)


def test_odd_ncol_takes_generic_flavour():
    era, deltas = make_case(7, 31, 3)
    eng = _engine(era, deltas)
    assert _uses_tma(eng, era) == 0


@pytest.mark.parametrize("i_reinterp,p_ref_inp", [(1, 30000), (0, None), (1, None)])
def test_staged_path_variants(i_reinterp, p_ref_inp):
    """SURVEY 8f rank 2: i_reinterp = 1 and p_ref_inp = None run through the staged path
    (pgw4era5_b200/staged.py) and match the oracle's restatement of step_03:202-251,:330-343."""
    from pgw4era5_b200 import settings
    era, deltas = make_case(12, 20, 4)
    ref = run_oracle(era, deltas, i_reinterp=i_reinterp, p_ref_inp=p_ref_inp)
    old = settings.i_reinterp, settings.p_ref_inp
    settings.i_reinterp, settings.p_ref_inp = i_reinterp, p_ref_inp
    try:
        res, _ = _apply(era, deltas)
    finally:
        settings.i_reinterp, settings.p_ref_inp = old
    np.testing.assert_allclose(res["phi_max_errors"], ref["phi_max_errors"], rtol=0, atol=1e-3)
    _check(res, ref)
    if p_ref_inp is None:
        np.testing.assert_array_equal(res["p_ref"].cpu().numpy(), ref["p_ref"])


def test_staged_path_equals_fused_for_default_settings():
    """The staged path run with the default settings (forced) agrees with the fused kernel."""
    from pgw4era5_b200 import staged
    era, deltas = make_case(12, 20, 4)
    eng = _engine(era, deltas)
    res_f = eng.apply(_dev(era), ERA_DATE, ignore_top_pressure_error=True)
    fused = {k: v.clone() for k, v in res_f.items() if isinstance(v, torch.Tensor)}
    res_s = staged.apply_staged(eng, _dev(era), ERA_DATE, ignore_top_pressure_error=True)
    assert res_s["n_iter"] == res_f["n_iter"]
    for name in ("PS", "T", "QV", "U", "V", "T_SKIN", "T_SO", "FR_SEA_ICE"):
        assert float((res_s[name] - fused[name]).abs().nan_to_num().max()) <= TOL[name], name


def _flat_case(ny, nx, seed, zscale):
    """A case with the orography scaled down (so that a high p_ref stays above the ground)."""
    from pgw4era5_b200.constants import CON_RD
    era, deltas = make_case(ny, nx, seed)
    era["FIS"] = era["FIS"] * zscale
    era["PS"] = (101325.0 * torch.exp(-era["FIS"].double() / (CON_RD * 270.0))).float()
    deltas["ps_hist"]["data"] = era["PS"].expand_as(deltas["ps_hist"]["data"]).clone() * 1.002
    return era, deltas


@pytest.mark.parametrize("p_ref", [85000, 50000, 10000])
def test_polynomial_fixed_point_other_reference_pressures(p_ref):
    """TMA flavour (ncol % 4 == 0): p_ref two layers above the ground (almost no layer in the polynomial,
    l* + 1 == the lowest level for some columns), mid troposphere, and 100 hPa (91 parked levels: the
    stash no longer allows 3 CTAs/SM) against the oracle."""
    from pgw4era5_b200 import settings
    era, deltas = _flat_case(12, 24, 31, 0.05)
    ref = run_oracle(era, deltas, p_ref_inp=p_ref)
    old = settings.p_ref_inp
    settings.p_ref_inp = p_ref
    try:
        res, eng = _apply(era, deltas)
        assert _uses_tma(eng, era) == 1
    finally:
        settings.p_ref_inp = old
    np.testing.assert_allclose(res["phi_max_errors"], ref["phi_max_errors"], rtol=0, atol=1e-3)
    _check(res, ref)


def test_polynomial_fixed_point_large_ps_change_falls_back():
    """zg deltas ten times larger: |dps| reaches several thousand Pa, beyond the range of the polynomial
    (0.012 ps), so warps integrate all parked levels directly; results still match the oracle."""
    era, deltas = make_case(12, 24, 33)
    deltas["zg"]["data"] = deltas["zg"]["data"] * 10.0
    ref = run_oracle(era, deltas)
    assert float(np.abs(ref["deltas"]["ps"]).max()) > 0.012 * 101325
    res, eng = _apply(era, deltas)
    assert _uses_tma(eng, era) == 1
    np.testing.assert_allclose(res["phi_max_errors"], ref["phi_max_errors"], rtol=0, atol=1e-3)
    _check(res, ref)


# ---------------------------------------------------------------------------------------------
# against the UNMODIFIED reference executed in the build container (tests/golden/reference_glue.npz,
# oracle/make_golden_glue.py): step_03's pgw_for_era5 from NetCDF in to NetCDF out
# ---------------------------------------------------------------------------------------------
def _golden_case():
    import os
    from datetime import datetime
    from oracle.golden import load as load_golden
    G = load_golden(os.path.join(os.path.dirname(__file__), "golden", "reference_glue.npz"))
    era = {}
    for k in G:
        if k.startswith("case_era_"):
            v = G[k]
            era[k[len("case_era_"):]] = torch.from_numpy(v) if v.dtype == np.float32 else v
    era["akm"], era["bkm"] = 0.5 * (era["ak"][1:] + era["ak"][:-1]), 0.5 * (era["bk"][1:] + era["bk"][:-1])
    times = G["case_delta_time"].astype("datetime64[ns]")
    deltas = {}
    for k in G:
        if k.startswith("case_delta_") and k not in ("case_delta_time", "case_delta_plev"):
            d = G[k]
            deltas[k[len("case_delta_"):]] = dict(time=times, data=torch.from_numpy(d),
                                                  plev=G["case_delta_plev"] if d.ndim == 4 else None)
    return G, era, deltas, datetime.fromisoformat(str(G["case_when"]))


def _vs_reference(G, tag, res, tol):
    out = {}
    for name, t in tol.items():
        g = res[name].detach().cpu().numpy().astype(np.float64).reshape(-1)
        r = G["pgw_%s_%s" % (tag, name)].astype(np.float64).reshape(-1)
        assert np.array_equal(np.isnan(g), np.isnan(r)), name
        out[name] = float(np.nanmax(np.abs(g - r)))
        assert out[name] <= t, (tag, name, out)
    return out


@pytest.mark.parametrize("flavour", ["auto", "generic"])
def test_fused_pass_matches_executed_reference(flavour, monkeypatch):
    """north_star tolerances (ta 1e-4 K, ps 1e-2 Pa, hus 1e-7, same iteration count) against what the
    reference itself wrote for PS/FIS stored as double; with all-float32 files the reference's own
    float32 rounding of ps_pgw and of the half-level geopotential (see oracle/make_golden_glue.py) adds
    up to ~3e-2 Pa of noise to ITS ps, which bounds the agreement there."""
    if flavour == "generic":
        monkeypatch.setenv("PGW_COLUMN_PATH", "generic")
    from pgw4era5_b200 import settings
    G, era, deltas, when = _golden_case()
    res, _ = _apply(era, deltas, when=when)
    assert res["n_iter"] == int(G["pgw_default64_n_iter"]) == int(G["pgw_default_n_iter"])
    np.testing.assert_allclose(res["phi_max_errors"], G["pgw_default64_errs"], rtol=0, atol=1e-3)
    tol = dict(TOL)
    tol.pop("delta_ps")
    _vs_reference(G, "default64", res, tol)
    _vs_reference(G, "default", res, dict(tol, PS=5e-2))
    old = settings.thresh_phi_ref_max_error
    settings.thresh_phi_ref_max_error = 1e-3
    try:
        res, _ = _apply(era, deltas, when=when)
    finally:
        settings.thresh_phi_ref_max_error = old
    assert res["n_iter"] == int(G["pgw_tight64_n_iter"]) == 8
    np.testing.assert_allclose(res["phi_max_errors"], G["pgw_tight64_errs"], rtol=0, atol=1e-3)
    _vs_reference(G, "tight64", res, tol)


def test_tma_flavour_matches_executed_reference():
    """The golden case has 30 columns, too few (and not a multiple of four) for the TMA flavour: tile it 32 times
    along the longitude (columns are independent, the stopping rule is a maximum) and compare every tile with
    what the reference wrote."""
    G, era, deltas, when = _golden_case()
    rep = 32
    tile = lambda t: t.repeat(*([1] * (t.dim() - 1)), rep).contiguous()
    era_t = {k: (tile(v) if isinstance(v, torch.Tensor) else v) for k, v in era.items()}
    era_t["lon"] = np.arange(len(era["lon"]) * rep, dtype=np.float64)
    deltas_t = {k: dict(v, data=tile(v["data"])) for k, v in deltas.items()}
    eng = _engine(era_t, deltas_t)
    res = eng.apply(_dev(era_t), when, ignore_top_pressure_error=True)
    assert _uses_tma(eng, era_t) == 1
    assert res["n_iter"] == int(G["pgw_default64_n_iter"])
    np.testing.assert_allclose(res["phi_max_errors"], G["pgw_default64_errs"], rtol=0, atol=1e-3)
    nx = len(era["lon"])
    tol = dict(TOL)
    tol.pop("delta_ps")
    for name, t in tol.items():
        g = res[name].detach().cpu().numpy().astype(np.float64)
        r = G["pgw_default64_%s" % name].astype(np.float64).reshape(g.shape[:-1] + (nx,))
        for k in (0, 13, rep - 1):
            part = g[..., k * nx:(k + 1) * nx]
            assert np.array_equal(np.isnan(part), np.isnan(r)), name
            assert np.nanmax(np.abs(part - r)) <= t, (name, k, float(np.nanmax(np.abs(part - r))))


@pytest.mark.parametrize("tag,name,value", [("pref_none64", "p_ref_inp", None), ("reinterp64", "i_reinterp", 1)])
def test_staged_path_matches_executed_reference(tag, name, value):
    """The non-default settings (step_03:202-251, :330-343) through pgw4era5_b200.staged."""
    from pgw4era5_b200 import settings
    G, era, deltas, when = _golden_case()
    old = getattr(settings, name)
    setattr(settings, name, value)
    try:
        res, _ = _apply(era, deltas, when=when)
    finally:
        setattr(settings, name, old)
    assert res["n_iter"] == int(G["pgw_%s_n_iter" % tag])
    np.testing.assert_allclose(res["phi_max_errors"], G["pgw_%s_errs" % tag], rtol=0, atol=1e-3)
    tol = dict(TOL)
    tol.pop("delta_ps")
    _vs_reference(G, tag, res, tol)


def test_no_soil_levels_and_many_soil_levels():
    """Edge cases of the soil block (step_03:139-146): a file without soil levels, and the maximum the ABI carries
    (PGW_MAX_SOIL = 16)."""
    from pgw4era5_b200 import _native as N
    era, deltas = make_case(9, 32, 41)
    ref_T_SKIN = run_oracle(era, deltas)["T_SKIN"]
    for nsoil in (0, N.PGW_MAX_SOIL):
        e = dict(era)
        e["soil1"] = np.linspace(0.01, 3.0, nsoil)
        e["T_SO"] = era["T_SO"][:, :1].repeat(1, max(nsoil, 1), 1, 1)[:, :nsoil].contiguous() - \
            0.1 * torch.arange(nsoil, dtype=torch.float32).reshape(1, nsoil, 1, 1)
        ref = run_oracle(e, deltas)
        res, _ = _apply(e, deltas)
        assert tuple(res["T_SO"].shape[:2]) == (1, nsoil)
        _check(res, ref)
        np.testing.assert_array_equal(ref["T_SKIN"], ref_T_SKIN)         # the soil block does not touch the rest
    with pytest.raises(ValueError, match="soil"):
        e = dict(era)
        e["soil1"] = np.linspace(0.01, 3.0, N.PGW_MAX_SOIL + 1)
        _engine(e, deltas)

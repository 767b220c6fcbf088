"""
The fused column kernel on model-level tables other than L137, and the instances the L137 cases never launch.

On the synthetic L137 table every layer the iteration can touch is thin enough for the ln series (FAST) at every
p_ref the other tests use, so they launch only the FAST instances, always with 137 levels.  Here:

- level tables x p_ref: L12 (a short column the pair ring nearly holds), L31, L60, L91, L160 (kTmaMaxLev), L161
  (one level too many: the cp.async flavour on a grid that is otherwise TMA-eligible), at p_ref down to 1 hPa
  (140 parked levels: the 512-column tensor-memory stash).  Each runs the TMA flavour and PGW_COLUMN_PATH=generic
  against the oracle and against each other.
- `<false, 137, 56>`: L137 with one thick layer in the stash (exact log, the L137 instance), once at the top of the
  stash (s just above the series' range) and once a layer spanning 25 below p_ref (s = 0.36).
- the per-column p_ref, the re-interpolation (with its replay for iteration N) and the reference-dtype instances
  on a coarse table (exact log) and on L137 (FAST).
- the 512-column stash on a grid of two waves, and next to a 128-column plan on another stream.
- ascending delta axes, pinned to the result of the descending file in every path.

Every case asserts the plan it means to run (pgw_timestep_plan_info): a case that misses its instance is broken.
"""
from contextlib import contextmanager

import numpy as np
import pytest
import torch

from cases import ERA_DATE, TOL, compare, run_oracle
from pgw4era5_b200 import synthetic as S

pytestmark = pytest.mark.gpu

THRESH = 0.15
SEED = 1
NY, NX = 12, 32                        # 384 columns: TMA-eligible, 3 CTAs
FIELDS = ("PS", "delta_ps", "T", "QV", "U", "V", "T_SKIN", "T_SO", "FR_SEA_ICE")
K_THICK = 82                           # the thick layer of thick_layer_table (the top layer of the L137 stash)


def thick_layer_table():
    """L137 with half levels K_THICK+1 and K_THICK+2 moved to 98 % and 99 % of the way to K_THICK+3: layer K_THICK
    spans about three layers, s = (pb-pt)/(pb+pt) = 0.069 at ps = 110000 Pa and > 0.06 (the exact-log branch of
    ln_ratio) at the surface pressures of the case.  The stash top (half level 82 is the first at or below 300 hPa
    for ps = 110000 Pa) and hence 137 levels with 56 parked ones are unchanged."""
    ak, bk = S.hybrid_coefficients(137)
    k = K_THICK
    for j, w in ((k + 1, 0.98), (k + 2, 0.99)):
        ak[j] = (1.0 - w) * ak[k] + w * ak[k + 3]
        bk[j] = (1.0 - w) * bk[k] + w * bk[k + 3]
    return ak, bk


def wide_layer_table():
    """L137 with half levels 91..114 moved to 99 % and more of the way to half level 115: layer 90 spans 25 layers,
    s = 0.36 at ps = 95000 Pa, below p_ref for every column.  Where the exact log matters: the ln series there is off
    by ~2 s^9 / 9 = 2e-5, ~1.5 m2/s2 of geopotential.  137 levels with 56 parked ones, like thick_layer_table."""
    ak, bk = S.hybrid_coefficients(137)
    k, m = 90, 25
    a0, b0, a1, b1 = ak[k], bk[k], ak[k + m], bk[k + m]
    for i in range(1, m):
        w = 0.99 + 0.01 * i / m
        ak[k + i], bk[k + i] = (1.0 - w) * a0 + w * a1, (1.0 - w) * b0 + w * b1
    return ak, bk


# table -> (nlev, ak/bk or None for hybrid_coefficients(nlev))
TABLES = {"L%d" % n: (n, None) for n in (12, 31, 60, 91, 137, 160, 161)}
TABLES["L137thick"] = (137, "thick")
TABLES["L137wide"] = (137, "wide")
_BUILDERS = {"thick": thick_layer_table, "wide": wide_layer_table}

# (table, p_ref): plan of the default flavour (tma, fast, lst, np, tmem_cols, l137) and of the generic one
# (fast, lst, np).  ps_bound 110000 Pa.
PLANS = {
    ("L12", 30000): ((1, 0, 6, 6, 32, 0), (0, 7, 5)),
    ("L31", 30000): ((1, 0, 17, 14, 32, 0), (0, 18, 13)),
    ("L60", 30000): ((1, 1, 36, 24, 64, 0), (1, 36, 24)),         # largest s 0.0537: the series at its edge
    ("L60", 10000): ((1, 0, 28, 32, 64, 0), (0, 29, 31)),
    ("L91", 10000): ((1, 0, 45, 46, 128, 0), (0, 45, 46)),
    ("L160", 10000): ((1, 1, 78, 82, 256, 0), (1, 79, 81)),
    ("L160", 100): ((1, 0, 20, 140, 512, 0), (0, 21, 139)),
    ("L137", 30000): ((1, 1, 81, 56, 128, 1), (1, 82, 55)),
    ("L137thick", 30000): ((1, 0, 81, 56, 128, 1), (0, 82, 55)),
    ("L137wide", 30000): ((1, 0, 81, 56, 128, 1), (0, 82, 55)),
    ("L161", 30000): ((0, 1, 96, 65, 0, 0), (1, 96, 65)),           # nlev > kTmaMaxLev: cp.async
}


def _plan(tma, fast, lst, np_, tmem_cols, l137):
    return dict(tma=tma, fast=fast, lst=lst, np=np_, tmem_cols=tmem_cols, l137=l137)


def _generic_plan(fast, lst, np_):
    return _plan(0, fast, lst, np_, 0, 0)


def table(name):
    nlev, kind = TABLES[name]
    return _BUILDERS[kind]() if kind else S.hybrid_coefficients(nlev)


def make_case(name, ny=NY, nx=NX, seed=SEED, device="cpu"):
    """make_case of cases.py on the European grid, with the level table `name`."""
    nlev, kind = TABLES[name]
    lat, lon = np.linspace(30.0, 80.0, ny), np.linspace(-20.0, 50.0, nx)
    era = S.make_era5(ny, nx, seed, device=device, nlev=nlev, lat=lat, lon=lon)
    if kind:
        ak, bk = _BUILDERS[kind]()
        era.update(ak=ak, bk=bk, akm=0.5 * (ak[1:] + ak[:-1]), bkm=0.5 * (bk[1:] + bk[:-1]))
    return era, S.make_deltas(era, seed, device=device)


@contextmanager
def _settings(**kw):
    from pgw4era5_b200 import settings
    old = {k: getattr(settings, k) for k in kw}
    for k, v in kw.items():
        setattr(settings, k, v)
    try:
        yield
    finally:
        for k, v in old.items():
            setattr(settings, k, v)


def _engine(era, deltas, streamed=False):
    from pgw4era5_b200.deltastream import StreamedDeltaSet
    from pgw4era5_b200.engine import DeltaSet, PGWEngine
    ds = StreamedDeltaSet(deltas, slots=2) if streamed else DeltaSet(deltas, device="cuda")
    return PGWEngine(era["ak"], era["bk"], ds, soil1=era["soil1"])


def _dev(era):
    return {k: (v.cuda() if isinstance(v, torch.Tensor) else v) for k, v in era.items()}


def _run(eng, era, p_ref=30000, k_spec=None, **kw):
    """One submit: (result, plan of the column kernel it launched)."""
    from pgw4era5_b200 import _native as N
    with _settings(p_ref_inp=p_ref, **kw):
        p = eng.submit(_dev(era), ERA_DATE, ignore_top_pressure_error=True, k_spec=k_spec)
        plan = N.plan_info(p.args)
        res = p.result()
    return res, plan


def _check_margin(ref, thresh=THRESH):
    """The iteration count is no coin flip: every E_k is further than 1e-3 thresh from the threshold."""
    E = np.asarray(ref["phi_max_errors"])
    assert np.min(np.abs(E - thresh)) > 1e-3 * thresh, E


def _check_oracle(res, ref):
    assert res["n_iter"] == ref["n_iter"], (res["phi_max_errors"], ref["phi_max_errors"])
    np.testing.assert_allclose(res["phi_max_errors"], ref["phi_max_errors"], rtol=0, atol=1e-3)
    errs = compare(res, ref)
    for name, e in errs.items():
        assert e <= TOL[name], (name, e, errs)


ULP_PS = 2.0 ** -7           # float32 spacing of ps between 65536 and 131072 Pa


def _check_flavours_agree(res_t, res_g, plan_g):
    """The bounds of test_timestep_gpu.test_tma_and_generic_flavours_agree, for two runs that took the same
    speculation path (the rewrite of PS and QV for N < k_spec rounds differently from an exact hit), with two
    differences that other level tables bring out:

    - PS: the flavours' geopotentials differ by at most 5e-6 m2/s2 (the TMA flavour's polynomial in dps), which moves
      the ps update by adj_factor * ps / (Rd * T) * 5e-6 ~ 7e-6 Pa, far below one float32 ulp of ps (2^-7 Pa).  A
      column's float32 ps can then differ only where that value sits within 7e-6 Pa of a rounding boundary, by one
      ulp; QV follows with |dq| <= q * dps / ps (p = akm + ps * bkm, so dp / p <= dps / ps).
    - QV at the levels the cp.async flavour sweeps unpaired -- the last parked level when np is odd, level 0 when the
      levels above the stash are odd in number: there it evaluates the saturation vapour pressure in its general
      form, while the TMA flavour, which pairs every level, takes the all-ice form of a cold warp (one reciprocal of
      a two-term instead of a four-term product).  A few float32 ulps of e, amplified where RELHUM_era + dhur nearly
      cancels (RELHUM is 1 % at the model top of these cases): up to 4e-5 relative, 2.4e-8 kg/kg on the B200.  At
      these levels the two flavours are held to the north_star tolerance, 1e-7, which each meets against the oracle.
    """
    assert res_t["n_iter"] == res_g["n_iter"]
    for name in ("T", "U", "V", "T_SKIN", "T_SO", "FR_SEA_ICE"):
        assert torch.equal(res_t[name].view(torch.int32), res_g[name].view(torch.int32)), name
    dps = (res_t["PS"] - res_g["PS"]).abs().double()
    assert float(dps.max()) <= ULP_PS
    unpaired = ([plan_g["lst"]] if plan_g["np"] % 2 else []) + ([0] if plan_g["lst"] % 2 else [])
    dq = (res_t["QV"] - res_g["QV"]).abs().double()[0]
    bound = 1e-9 + res_g["QV"].double()[0] * (dps / res_g["PS"].double())
    paired = torch.ones(dq.shape[0], dtype=torch.bool, device=dq.device)
    paired[unpaired] = False
    assert bool((dq[paired] <= bound[paired]).all()), float((dq[paired] - bound[paired]).max())
    if unpaired:
        assert float(dq[unpaired].max()) <= TOL["QV"], unpaired
    np.testing.assert_allclose(res_t["phi_max_errors"], res_g["phi_max_errors"], rtol=0, atol=5e-6)


def _assert_bitwise(got, want, names=FIELDS):
    assert got["n_iter"] == want["n_iter"] and got["phi_max_errors"] == want["phi_max_errors"]
    for name in names:
        g, w = got[name].cpu().reshape(-1), want[name].cpu().reshape(-1)
        assert torch.equal(g.isnan(), w.isnan()) and torch.equal(g.nan_to_num(), w.nan_to_num()), name


# ---------------------------------------------------------------------------------------------------------------
# level tables x p_ref, TMA and generic flavours
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,p_ref", list(PLANS))
def test_level_table_flavours_match_oracle(name, p_ref, monkeypatch):
    era, deltas = make_case(name)
    ref = run_oracle(era, deltas, p_ref_inp=p_ref)
    _check_margin(ref)
    eng = _engine(era, deltas)
    want_t, want_g = PLANS[(name, p_ref)]
    monkeypatch.delenv("PGW_COLUMN_PATH", raising=False)
    res_t, plan_t = _run(eng, era, p_ref, k_spec=ref["n_iter"])
    assert plan_t == _plan(*want_t)
    monkeypatch.setenv("PGW_COLUMN_PATH", "generic")
    res_g, plan_g = _run(eng, era, p_ref, k_spec=ref["n_iter"])
    assert plan_g == _generic_plan(*want_g)
    _check_oracle(res_t, ref)
    _check_oracle(res_g, ref)
    _check_flavours_agree(res_t, res_g, plan_g)
    assert eng.stats["reruns"] == 0


# ---------------------------------------------------------------------------------------------------------------
# the other cp.async instances: per-column p_ref, re-interpolation, reference dtypes
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,fast", [("L31", 0), ("L137", 1)])
def test_local_p_ref_instances_match_oracle(name, fast):
    """p_ref_inp = None: the stash reaches p_floor (300 hPa), so the plan is that of the table at 30000 Pa."""
    era, deltas = make_case(name)
    ref = run_oracle(era, deltas, p_ref_inp=None)
    _check_margin(ref)
    res, plan = _run(_engine(era, deltas), era, p_ref=None)
    assert plan == _generic_plan(fast, *PLANS[(name, 30000)][1][1:])
    _check_oracle(res, ref)
    np.testing.assert_array_equal(res["p_ref"].cpu().numpy().reshape(-1), np.asarray(ref["p_ref"]).reshape(-1))


@pytest.mark.parametrize("name,fast", [("L31", 0), ("L137", 1)])
def test_reinterp_instances_match_oracle_and_staged_path(name, fast):
    """i_reinterp = 1 at the bounds of test_reinterp_gpu.py.  k_spec 8 > N: finalize replays the column kernel for
    iteration N (the RI replay)."""
    era, deltas = make_case(name)
    ref = run_oracle(era, deltas, i_reinterp=1)
    _check_margin(ref)
    eng = _engine(era, deltas)
    res, plan = _run(eng, era, i_reinterp=1, k_spec=8)
    assert plan == _generic_plan(fast, *PLANS[(name, 30000)][1][1:])
    assert res["n_iter"] < 8 and eng.stats["rewrites"] == 1
    _check_oracle(res, ref)
    with _settings(i_reinterp=1, p_ref_inp=30000):
        st = _engine(era, deltas).apply(_dev(era), ERA_DATE, ignore_top_pressure_error=True)
    assert res["n_iter"] == st["n_iter"]
    for f in FIELDS:
        g, r = res[f].double().cpu().numpy(), st[f].double().cpu().numpy()
        assert np.array_equal(np.isnan(g), np.isnan(r)), f
        d = float(np.nanmax(np.abs(g - r)))
        assert d <= TOL[f], (f, d)


def test_reference_dtypes_instance_on_a_coarse_table():
    """i_reference_dtypes = 1 on L31 against oracle(emulate_file_dtypes=True), at the bounds of
    test_ref_dtypes_gpu.py (the instance has no FAST form)."""
    from test_ref_dtypes_gpu import ULP_PHI, ULP_PS, _ps_stats
    era, deltas = make_case("L31")
    ref = run_oracle(era, deltas, emulate_file_dtypes=True)
    E = np.asarray(ref["phi_max_errors"])
    assert np.min(np.abs(E - THRESH)) > 1.5 * ULP_PHI, E
    res, plan = _run(_engine(era, deltas), era, i_reference_dtypes=1)
    assert plan == _generic_plan(0, *PLANS[("L31", 30000)][1][1:])
    assert res["n_iter"] == ref["n_iter"], (res["phi_max_errors"], E)
    np.testing.assert_allclose(res["phi_max_errors"], E, rtol=0, atol=1.01 * ULP_PHI)
    st = _ps_stats(res, ref["PS"])
    assert st["max"] <= 4 * ULP_PS + 1e-9, st
    assert st["within_tol"] >= 0.995, st
    assert st["exact"] >= 0.97, st
    errs = compare(res, ref)
    for f in ("T", "U", "V", "T_SKIN", "T_SO", "FR_SEA_ICE"):
        assert errs[f] <= TOL[f], (f, errs)


# ---------------------------------------------------------------------------------------------------------------
# the 512-column tensor-memory stash
# ---------------------------------------------------------------------------------------------------------------
def test_512_column_stash_on_two_waves(monkeypatch):
    """L160 at p_ref = 1 hPa: 140 parked levels, 512 TMEM columns and 227 KB of shared memory, one CTA per SM.  96 x 400
    columns are 300 CTAs, more than two waves on 148 SMs.  The whole grid against the generic flavour and against
    the oracle (about 10 s of CPU)."""
    era, deltas = make_case("L160", 96, 400, device="cuda")
    ref = run_oracle(S.to_numpy(era), S.to_numpy(deltas), p_ref_inp=100)
    _check_margin(ref)
    eng = _engine(era, deltas)
    monkeypatch.delenv("PGW_COLUMN_PATH", raising=False)
    res_t, plan_t = _run(eng, era, 100, k_spec=ref["n_iter"])
    assert plan_t == _plan(*PLANS[("L160", 100)][0])
    monkeypatch.setenv("PGW_COLUMN_PATH", "generic")
    res_g, plan_g = _run(eng, era, 100, k_spec=ref["n_iter"])
    assert plan_g == _generic_plan(*PLANS[("L160", 100)][1])
    _check_flavours_agree(res_t, res_g, plan_g)
    _check_oracle(res_t, ref)


def test_two_tensor_memory_plans_on_two_streams():
    """A 512-column plan (L160, 1 hPa) and a 128-column plan (L137, 300 hPa) submitted on two streams at once.  The
    shared memory of each CTA is padded to its share of the SM's tensor memory, so CTAs of the two kernels that
    share an SM never wait in tcgen05.alloc; each result is bit for bit that of the engine running alone."""
    era_a, deltas_a = make_case("L160", 96, 400, device="cuda")
    era_b, deltas_b = make_case("L137", 96, 400, seed=3, device="cuda")
    eng_a, eng_b = _engine(era_a, deltas_a), _engine(era_b, deltas_b)
    alone_a, plan_a = _run(eng_a, era_a, 100, k_spec=8)
    alone_b, plan_b = _run(eng_b, era_b, 30000, k_spec=8)
    assert plan_a["tmem_cols"] == 512 and plan_b["tmem_cols"] == 128 and plan_b["l137"] == 1
    alone_a = {k: (v.clone() if isinstance(v, torch.Tensor) else v) for k, v in alone_a.items()}
    alone_b = {k: (v.clone() if isinstance(v, torch.Tensor) else v) for k, v in alone_b.items()}
    dev_a, dev_b = _dev(era_a), _dev(era_b)
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    torch.cuda.synchronize()
    with torch.cuda.stream(s1), _settings(p_ref_inp=100):
        pa = eng_a.submit(dev_a, ERA_DATE, ignore_top_pressure_error=True, k_spec=8)
    with torch.cuda.stream(s2), _settings(p_ref_inp=30000):
        pb = eng_b.submit(dev_b, ERA_DATE, ignore_top_pressure_error=True, k_spec=8)
    ra, rb = pa.result(), pb.result()
    torch.cuda.synchronize()
    assert eng_a.stats["reruns"] == 0 and eng_b.stats["reruns"] == 0
    _assert_bitwise(ra, alone_a)
    _assert_bitwise(rb, alone_b)


# ---------------------------------------------------------------------------------------------------------------
# ascending delta axes (plev_descending = 0)
# ---------------------------------------------------------------------------------------------------------------
def _reversed(deltas, names):
    out = dict(deltas)
    for n in names:
        d = deltas[n]
        out[n] = dict(d, plev=np.ascontiguousarray(np.asarray(d["plev"])[::-1]), data=d["data"].flip(1).contiguous())
    return out


PATHS = {
    "tma": (dict(), 1),
    "generic": (dict(), 0),
    "local": (dict(p_ref=None), 0),
    "reinterp": (dict(i_reinterp=1), 0),
    "streamed": (dict(), 1),
}


@pytest.mark.parametrize("name", ["L137", "L31"])
@pytest.mark.parametrize("path", list(PATHS))
def test_ascending_delta_axes_equal_descending(path, name, monkeypatch):
    """ta, hur, ua, va with plev ascending (zg kept descending): the kernels walk the same nodes in the same order,
    so every output is bit for bit that of the descending file.  The reference raises on such a file
    (functions.py:383-384 flips the axis unconditionally), so the descending file is the reference here."""
    era, deltas = make_case(name)
    asc = _reversed(deltas, ("ta", "hur", "ua", "va"))
    kw, tma = PATHS[path]
    if path == "generic":
        monkeypatch.setenv("PGW_COLUMN_PATH", "generic")
    else:
        monkeypatch.delenv("PGW_COLUMN_PATH", raising=False)
    got = {}
    for tag, d in (("desc", deltas), ("asc", asc)):
        eng = _engine(era, d, streamed=(path == "streamed"))
        assert bool(eng.deltas.plev_descending) == (tag == "desc")
        got[tag], plan = _run(eng, era, **kw)
        assert plan["tma"] == tma
    names = FIELDS + (("p_ref",) if path == "local" else ())
    _assert_bitwise(got["asc"], got["desc"], names)


def test_ascending_zg_with_scalar_p_ref():
    """zg alone reversed: the engine takes the p_ref level by value, like the reference's .sel(plev=p_ref); bit for bit
    the descending result, and the oracle (which handles zg in either order) agrees."""
    era, deltas = make_case("L137")
    asc = _reversed(deltas, ("zg",))
    ref = run_oracle(era, asc)
    _check_margin(ref)
    want, _ = _run(_engine(era, deltas), era)
    got, plan = _run(_engine(era, asc), era)
    assert plan["tma"] == 1
    _assert_bitwise(got, want)
    _check_oracle(got, ref)

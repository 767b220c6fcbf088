"""p_ref_inp = None (step_03_apply_to_era.py:219-251) in the fused column kernel: PGWEngine.submit with the
reference pressure picked per column and iteration among zg's levels, against the fp64 oracle, the executed
reference and the staged path."""
import ctypes as C
from contextlib import contextmanager

import numpy as np
import pytest
import torch

from cases import ERA_DATE, TOL, compare, make_case, run_oracle

pytestmark = pytest.mark.gpu


@contextmanager
def _settings(**kw):
    from pgw4era5_b200 import settings
    kw.setdefault("p_ref_inp", None)
    old = {k: getattr(settings, k) for k in kw}
    for k, v in kw.items():
        setattr(settings, k, v)
    try:
        yield
    finally:
        for k, v in old.items():
            setattr(settings, k, v)


def _engine(era, deltas, **kw):
    from pgw4era5_b200.engine import DeltaSet, PGWEngine
    return PGWEngine(era["ak"], era["bk"], DeltaSet(deltas, device="cuda"), soil1=era["soil1"], **kw)


def _dev(era):
    return {k: (v.cuda() if isinstance(v, torch.Tensor) else v) for k, v in era.items()}


def _submit(eng, era, when=ERA_DATE, **kw):
    with _settings():
        return eng.submit(_dev(era), when, ignore_top_pressure_error=True, **kw).result()


def _p_ref(res):
    return res["p_ref"].detach().cpu().numpy().reshape(-1)


def _check_oracle(res, ref):
    assert res["n_iter"] == ref["n_iter"], (res["phi_max_errors"], ref["phi_max_errors"])
    np.testing.assert_allclose(res["phi_max_errors"], ref["phi_max_errors"], rtol=0, atol=1e-3)
    errs = compare(res, ref)
    for name, e in errs.items():
        assert e <= TOL[name], (name, e, errs)
    assert res["p_ref"].dtype == torch.float64
    np.testing.assert_array_equal(_p_ref(res), np.asarray(ref["p_ref"]).reshape(-1))


def _first_choice(ps, plev):
    """p_ref of the first iteration, from 0.95 PS alone (determine_p_ref with ps_pgw == PS)."""
    pe = 0.95 * np.asarray(ps, dtype=np.float64).reshape(-1)
    out = np.full(pe.shape, np.nan)
    for i, x in enumerate(pe):
        for p in plev:
            if x > p:
                out[i] = p
                break
    return out


def _moving_case(ny=24, nx=40, seed=1, ncols=7, dzg=-30.0):
    """0.95 PS sits 20 Pa above the 850 hPa level in `ncols` columns and at least 1000 Pa above the next
    lower zg level everywhere else; a uniformly negative zg delta drives dps to about -300 Pa, so p_ref moves
    from 850 to 700 hPa in exactly those columns."""
    era, deltas = make_case(ny, nx, seed)
    plev = np.asarray(deltas["zg"]["plev"], dtype=np.float64)
    ps = era["PS"].to(torch.float64).reshape(-1).clone()
    pe = 0.95 * ps.numpy()
    for i, x in enumerate(pe):
        gap = x - plev[plev < x].max()
        if gap < 1000.0:
            ps[i] += (1000.0 - gap) / 0.95 + 10.0
    cols = np.linspace(0, ny * nx - 1, ncols).astype(int)
    ps[cols] = (85000.0 + 20.0) / 0.95
    era["PS"] = ps.to(torch.float32).reshape(era["PS"].shape)
    deltas["zg"] = dict(deltas["zg"], data=deltas["zg"]["data"] + dzg)
    return era, deltas, cols


@pytest.mark.parametrize("ny,nx,seed", [(24, 40, 1), (33, 129, 2), (7, 31, 3)])
def test_submit_matches_oracle(ny, nx, seed):
    from pgw4era5_b200 import _native as N
    era, deltas = make_case(ny, nx, seed)
    ref = run_oracle(era, deltas, p_ref_inp=None)
    eng = _engine(era, deltas)
    with _settings():
        p = eng.submit(_dev(era), ERA_DATE, ignore_top_pressure_error=True)
        res = p.result()
    _check_oracle(res, ref)
    assert eng.stats["reruns"] == 0
    # the per-column p_ref runs in the cp.async flavour on every grid, TMA-eligible ones (ncol % 4 == 0) included
    assert N.lib.pgw_timestep_uses_tma(C.byref(p.args)) == 0
    if (ny * nx) % 4 == 0:
        q = eng.submit(_dev(era), ERA_DATE, ignore_top_pressure_error=True)
        assert N.lib.pgw_timestep_uses_tma(C.byref(q.args)) == 1
        assert "p_ref" not in q.result()


def test_submit_matches_oracle_european_domain():
    """BASELINE configs[0]: 201x281 European subdomain, 137 levels, plev19."""
    era, deltas = make_case(201, 281, 1)
    ref = run_oracle(era, deltas, p_ref_inp=None)
    _check_oracle(_submit(_engine(era, deltas), era), ref)


def test_submit_matches_executed_reference():
    """The golden case the reference itself ran with p_ref_inp = None, with the tolerances of the staged path."""
    from test_timestep_gpu import _golden_case, _vs_reference
    G, era, deltas, when = _golden_case()
    res = _submit(_engine(era, deltas), era, when=when)
    assert res["n_iter"] == int(G["pgw_pref_none64_n_iter"])
    np.testing.assert_allclose(res["phi_max_errors"], G["pgw_pref_none64_errs"], rtol=0, atol=1e-3)
    tol = dict(TOL)
    tol.pop("delta_ps")
    _vs_reference(G, "pref_none64", res, tol)


def test_submit_matches_staged_path():
    era, deltas = make_case(24, 40, 1)
    res = _submit(_engine(era, deltas), era)
    with _settings():
        st = _engine(era, deltas).apply(_dev(era), ERA_DATE, ignore_top_pressure_error=True)
    assert res["n_iter"] == st["n_iter"]
    np.testing.assert_array_equal(_p_ref(res), _p_ref(st))
    for name in ("PS", "delta_ps", "T", "QV", "U", "V", "T_SKIN", "T_SO", "FR_SEA_ICE"):
        g, r = res[name].double().cpu().numpy(), st[name].double().cpu().numpy()
        assert np.array_equal(np.isnan(g), np.isnan(r)), name          # sea ice is NaN over land
        d = float(np.nanmax(np.abs(g - r)))
        assert d <= TOL[name], (name, d)


def test_p_ref_moves_during_the_iteration():
    era, deltas, cols = _moving_case()
    ref = run_oracle(era, deltas, p_ref_inp=None)
    first = _first_choice(era["PS"].numpy(), np.asarray(deltas["zg"]["plev"]))
    final = np.asarray(ref["p_ref"]).reshape(-1)
    moved = np.nonzero(final != first)[0]
    np.testing.assert_array_equal(moved, cols)
    assert np.all(first[cols] == 85000.0) and np.all(final[cols] == 70000.0)
    res = _submit(_engine(era, deltas), era)
    _check_oracle(res, ref)


@pytest.mark.parametrize("k_spec", [3, 5, 9, 19])
def test_speculation_paths_agree(k_spec):
    """rerun (k_spec too small), exact hit and rewrite (k_spec too large): p_ref is that of iteration N."""
    era, deltas, _ = _moving_case()
    ref = run_oracle(era, deltas, p_ref_inp=None)
    eng = _engine(era, deltas)
    res = _submit(eng, era, k_spec=k_spec)
    _check_oracle(res, ref)
    if k_spec < ref["n_iter"]:
        assert eng.stats["reruns"] == 1
    if k_spec > ref["n_iter"]:
        assert eng.stats["rewrites"] == 1


def test_no_reference_level_raises():
    """zg truncated to 1000-850 hPa: a column with 0.95 PS below 850 hPa has no candidate level."""
    from pgw4era5_b200.staged import MSG_NO_PREF
    era, deltas = make_case(24, 40, 1)
    zg = deltas["zg"]
    deltas["zg"] = dict(zg, plev=np.asarray(zg["plev"])[:3], data=zg["data"][:, :3].contiguous())
    ps = era["PS"].clone()
    ps.view(-1)[17] = 80000.0
    era["PS"] = ps
    with pytest.raises(ValueError) as e:
        _submit(_engine(era, deltas), era)
    assert str(e.value) == MSG_NO_PREF
    with _settings(), pytest.raises(ValueError) as e2:
        _engine(era, deltas).apply(_dev(era), ERA_DATE, ignore_top_pressure_error=True)
    assert str(e2.value) == MSG_NO_PREF


def test_stash_floor_rerun():
    """A stash sized for p_ref >= 900 hPa: columns that pick 850 hPa or higher make the engine lower the floor
    and rerun; the result still matches the oracle."""
    era, deltas = make_case(24, 40, 1)
    ref = run_oracle(era, deltas, p_ref_inp=None)
    assert np.nanmin(ref["p_ref"]) < 90000.0
    eng = _engine(era, deltas, p_floor=90000.0)
    res = _submit(eng, era)
    assert eng.stats["reruns"] >= 1
    assert eng.p_floor <= np.nanmin(ref["p_ref"])
    _check_oracle(res, ref)


def test_host_pipeline_matches_submit():
    from pgw4era5_b200.hostpipe import HostPipeline
    era, deltas, _ = _moving_case(33, 129, 2)
    res = _submit(_engine(era, deltas), era)
    eng = _engine(era, deltas)
    pipe = HostPipeline(eng, 33, 129, nslots=2)
    hin, hout = pipe.pin_inputs(era), pipe.alloc_host_outputs()
    with _settings():
        assert pipe.run(hin, ERA_DATE, hout, ignore_top_pressure_error=True) is None
        got = [r for r in pipe.drain() if r is not None]
    assert len(got) == 1 and got[0]["n_iter"] == res["n_iter"]
    for name in ("PS", "delta_ps", "T", "QV", "U", "V", "T_SKIN", "T_SO", "FR_SEA_ICE"):
        np.testing.assert_array_equal(got[0][name].reshape(-1).numpy(), res[name].cpu().reshape(-1).numpy(),
                                      err_msg=name)          # NaN (sea ice over land) equals NaN


def test_submit_still_refuses_what_it_does_not_cover():
    era, deltas = make_case(7, 31, 3)
    eng = _engine(era, deltas)
    for kw in (dict(i_reinterp=1), dict(i_reference_dtypes=1)):
        with _settings(**kw), pytest.raises(ValueError, match="staged path"):
            eng.submit(_dev(era), ERA_DATE, ignore_top_pressure_error=True)

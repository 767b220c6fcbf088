"""i_reinterp = 1 (step_03_apply_to_era.py:155-173, :202-216, :330-343) in the fused column kernel: PGWEngine.submit
re-interpolates the ERA state onto every iteration's pressures, against the fp64 oracle, the executed reference
and the staged path."""
import ctypes as C
from contextlib import contextmanager

import numpy as np
import pytest
import torch

from cases import ERA_DATE, TOL, compare, make_case, run_oracle

pytestmark = pytest.mark.gpu

FIELDS = ("PS", "delta_ps", "T", "QV", "U", "V", "T_SKIN", "T_SO", "FR_SEA_ICE")


@contextmanager
def _settings(**kw):
    from pgw4era5_b200 import settings
    kw.setdefault("i_reinterp", 1)
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


def _submit(eng, era, when=ERA_DATE, settings=None, **kw):
    with _settings(**(settings or {})):
        return eng.submit(_dev(era), when, ignore_top_pressure_error=True, **kw).result()


def _check_oracle(res, ref):
    assert res["n_iter"] == ref["n_iter"], (res["phi_max_errors"], ref["phi_max_errors"])
    np.testing.assert_allclose(res["phi_max_errors"], ref["phi_max_errors"], rtol=0, atol=1e-3)
    errs = compare(res, ref)
    for name, e in errs.items():
        assert e <= TOL[name], (name, e, errs)


def _assert_bitwise(got, want, names=FIELDS):
    for name in names:
        g, w = got[name].cpu().reshape(-1), want[name].cpu().reshape(-1)
        assert torch.equal(g.isnan(), w.isnan()) and torch.equal(g.nan_to_num(), w.nan_to_num()), name


def _mid(era):
    ak, bk = np.asarray(era["ak"], dtype=np.float64), np.asarray(era["bk"], dtype=np.float64)
    return 0.5 * np.diff(ak) + ak[:-1], 0.5 * np.diff(bk) + bk[:-1]


def _levels_crossed(era, ref):
    """Per column: how many ERA levels the lowest level's final target lies above its own ERA level
    (negative: below the lowest ERA level, i.e. constant extrapolation)."""
    akm, bkm = _mid(era)
    PS = era["PS"].double().numpy().reshape(-1)
    ps = np.asarray(ref["ps_traj"][-1], dtype=np.float64).reshape(-1)
    pe = akm[None, :] + PS[:, None] * bkm[None, :]
    pt = akm[-1] + ps * bkm[-1]
    return (pe > pt[:, None]).sum(axis=1) - 1, ps - PS


def _shifted_zg(dzg, ny=24, nx=40, seed=1):
    era, deltas = make_case(ny, nx, seed)
    deltas["zg"] = dict(deltas["zg"], data=deltas["zg"]["data"] + dzg)
    return era, deltas


@pytest.mark.parametrize("ny,nx,seed", [(24, 40, 1), (33, 129, 2), (7, 31, 3)])
def test_submit_matches_oracle(ny, nx, seed):
    from pgw4era5_b200 import _native as N
    era, deltas = make_case(ny, nx, seed)
    ref = run_oracle(era, deltas, i_reinterp=1)
    eng = _engine(era, deltas)
    with _settings():
        p = eng.submit(_dev(era), ERA_DATE, ignore_top_pressure_error=True)
        res = p.result()
    _check_oracle(res, ref)
    assert eng.stats["reruns"] == 0
    # the re-interpolation runs in the cp.async flavour on every grid, TMA-eligible ones (ncol % 4 == 0) included
    assert p.args.flags & N.FLAG_REINTERP
    assert N.lib.pgw_timestep_uses_tma(C.byref(p.args)) == 0
    if (ny * nx) % 4 == 0:
        with _settings(i_reinterp=0):
            q = eng.submit(_dev(era), ERA_DATE, ignore_top_pressure_error=True)
            assert N.lib.pgw_timestep_uses_tma(C.byref(q.args)) == 1
            q.result()


def test_submit_matches_oracle_european_domain():
    """BASELINE configs[0]: 201x281 European subdomain, 137 levels, plev19."""
    era, deltas = make_case(201, 281, 1)
    ref = run_oracle(era, deltas, i_reinterp=1)
    _check_oracle(_submit(_engine(era, deltas), era), ref)


def test_submit_matches_executed_reference():
    """The golden case the reference itself ran with i_reinterp = 1, with the tolerances of the staged path."""
    from test_timestep_gpu import _golden_case, _vs_reference
    G, era, deltas, when = _golden_case()
    res = _submit(_engine(era, deltas), era, when=when)
    assert res["n_iter"] == int(G["pgw_reinterp64_n_iter"])
    np.testing.assert_allclose(res["phi_max_errors"], G["pgw_reinterp64_errs"], rtol=0, atol=1e-3)
    tol = dict(TOL)
    tol.pop("delta_ps")
    _vs_reference(G, "reinterp64", res, tol)


def test_submit_matches_staged_path():
    era, deltas = make_case(24, 40, 1)
    res = _submit(_engine(era, deltas), era)
    with _settings():
        st = _engine(era, deltas).apply(_dev(era), ERA_DATE, ignore_top_pressure_error=True)
    assert res["n_iter"] == st["n_iter"]
    for name in FIELDS:
        g, r = res[name].double().cpu().numpy(), st[name].double().cpu().numpy()
        assert np.array_equal(np.isnan(g), np.isnan(r)), name          # sea ice is NaN over land
        d = float(np.nanmax(np.abs(g - r)))
        assert d <= TOL[name], (name, d)


def test_invariants_against_i_reinterp_0(monkeypatch):
    """Iteration 1 has pa_pgw == pa_era (every target an exact hit): the same first error bit for bit.  Levels with
    bkm == 0 keep their pressure in every iteration: T, U and V there equal the i_reinterp = 0 result bit for bit."""
    monkeypatch.setenv("PGW_COLUMN_PATH", "generic")
    era, deltas = make_case(33, 129, 2)
    eng = _engine(era, deltas)
    r1 = _submit(eng, era)
    r0 = _submit(eng, era, settings=dict(i_reinterp=0))
    assert r1["phi_max_errors"][0] == r0["phi_max_errors"][0]
    assert r1["n_iter"] > 1 and r1["phi_max_errors"][1] != r0["phi_max_errors"][1]
    _, bkm = _mid(era)
    flat = np.nonzero(bkm == 0.0)[0]
    assert len(flat) > 0
    for name in ("T", "U", "V"):
        g, w = r1[name][0, flat].cpu(), r0[name][0, flat].cpu()
        assert torch.equal(g, w), name
    deep = np.nonzero(bkm > 0.5)[0]
    assert not torch.equal(r1["T"][0, deep].cpu(), r0["T"][0, deep].cpu())


def test_targets_move_across_two_era_levels():
    """A strongly negative zg delta lowers ps by ~500-1100 Pa: the lowest level's targets move across 2 or more
    ERA levels, and the top parked level brackets with the level above the stash."""
    era, deltas = _shifted_zg(-80.0)
    ref = run_oracle(era, deltas, i_reinterp=1, n_iter_fixed=4)
    crossed, dps = _levels_crossed(era, ref)
    assert np.all(dps < 0.0) and np.count_nonzero(crossed >= 2) > 100
    ref = run_oracle(era, deltas, i_reinterp=1)
    _check_oracle(_submit(_engine(era, deltas), era), ref)


def test_targets_below_the_lowest_era_level():
    """A positive zg delta raises ps: the lowest targets lie below ERA level L-1 (constant extrapolation)."""
    era, deltas = _shifted_zg(30.0)
    ref = run_oracle(era, deltas, i_reinterp=1, n_iter_fixed=4)
    crossed, dps = _levels_crossed(era, ref)
    assert np.all(dps > 0.0) and np.all(crossed == -1)
    ref = run_oracle(era, deltas, i_reinterp=1)
    _check_oracle(_submit(_engine(era, deltas), era), ref)


def test_tight_stash_reads_above_it():
    """ps_bound just above the largest PS: the stash ends at the layer that contains p_ref, and with dps < 0 the
    sweeps bracket its top level with the ERA level above the stash (read from global memory)."""
    era, deltas = _shifted_zg(-80.0)
    ps_max = float(era["PS"].max())
    ak, bk = np.asarray(era["ak"], dtype=np.float64), np.asarray(era["bk"], dtype=np.float64)
    h = int(np.argmax(ak + (ps_max + 1.0) * bk >= 30000.0))
    lst = h - 1                                                        # stash_top of pgw_timestep.cu
    akm, bkm = _mid(era)
    ref = run_oracle(era, deltas, i_reinterp=1)
    PS = era["PS"].double().numpy().reshape(-1)
    ps = np.asarray(ref["PS"], dtype=np.float64).reshape(-1)
    assert bkm[lst] > 0.0 and np.all(akm[lst] + ps * bkm[lst] < akm[lst] + PS * bkm[lst])
    eng = _engine(era, deltas, ps_bound=ps_max + 1.0)
    _check_oracle(_submit(eng, era), ref)
    assert eng.stats["reruns"] == 0


@pytest.mark.parametrize("k_spec", [3, 5, 9, 19])
def test_speculation_paths_agree(k_spec):
    """With a threshold of 0.01 m2/s2, N = 5: k_spec 3 reruns (with 19), 5 hits, 9 and 19 replay the column
    kernel for N.  All four give the same outputs bit for bit."""
    era, deltas = make_case(24, 40, 1)
    ref = run_oracle(era, deltas, i_reinterp=1, thresh_phi_ref_max_error=0.01)
    assert ref["n_iter"] == 5
    s = dict(thresh_phi_ref_max_error=0.01)
    base = _submit(_engine(era, deltas), era, settings=s, k_spec=5)
    _check_oracle(base, ref)
    eng = _engine(era, deltas)
    res = _submit(eng, era, settings=s, k_spec=k_spec)
    _check_oracle(res, ref)
    _assert_bitwise(res, base)
    assert res["phi_max_errors"] == base["phi_max_errors"]
    assert eng.stats["reruns"] == (1 if k_spec < 5 else 0)
    assert eng.stats["rewrites"] == (0 if k_spec == 5 else 1)           # a rerun speculates max_n_iter - 1


def test_ps_bound_rerun():
    """ps_bound below the smallest PS: every column leaves the stash in iteration 1; the engine widens the bound
    and reruns."""
    era, deltas = make_case(24, 40, 1)
    ref = run_oracle(era, deltas, i_reinterp=1)
    eng = _engine(era, deltas, ps_bound=float(era["PS"].min()) - 100.0)
    _check_oracle(_submit(eng, era), ref)
    assert eng.stats["reruns"] >= 1


def test_p_ref_below_the_surface_raises():
    from pgw4era5_b200.engine import MSG_PREF
    era, deltas = make_case(24, 40, 1)
    ps = era["PS"].clone()
    ps.view(-1)[17] = 95000.0
    era["PS"] = ps
    with pytest.raises(ValueError) as e:
        _submit(_engine(era, deltas), era, settings=dict(p_ref_inp=100000))
    assert str(e.value) == MSG_PREF


def test_did_not_converge_raises():
    """max_n_iter = 3 allows 2 iterations; this case needs 4."""
    era, deltas = make_case(24, 40, 1)
    with pytest.raises(ValueError, match="did not converge"):
        _submit(_engine(era, deltas), era, settings=dict(max_n_iter=3))


def test_host_pipeline_matches_submit():
    from pgw4era5_b200.hostpipe import HostPipeline
    era, deltas = _shifted_zg(-80.0, 33, 129, 2)
    res = _submit(_engine(era, deltas), era)
    eng = _engine(era, deltas)
    pipe = HostPipeline(eng, 33, 129, nslots=2)
    hin, hout = pipe.pin_inputs(era), pipe.alloc_host_outputs()
    with _settings():
        assert pipe.run(hin, ERA_DATE, hout, ignore_top_pressure_error=True) is None
        got = [r for r in pipe.drain() if r is not None]
    assert len(got) == 1 and got[0]["n_iter"] == res["n_iter"]
    for name in FIELDS:
        np.testing.assert_array_equal(got[0][name].reshape(-1).numpy(), res[name].cpu().reshape(-1).numpy(),
                                      err_msg=name)          # NaN (sea ice over land) equals NaN


def test_submit_refuses_reinterp_with_reference_dtypes():
    era, deltas = make_case(7, 31, 3)
    eng = _engine(era, deltas)
    for kw in (dict(i_reference_dtypes=1), dict(p_ref_inp=None)):
        with _settings(**kw), pytest.raises(ValueError, match="staged path"):
            eng.submit(_dev(era), ERA_DATE, ignore_top_pressure_error=True)

"""Host logic of p_ref_inp = None in PGWEngine._complete on hand-made status blocks (no GPU needed):
PGW_ERR_NO_PREF raises the reference's message, PGW_ERR_PREF_FLOOR lowers the stash floor and reruns, and
either is ignored when it first fired in an iteration the reference never ran."""
import contextlib
import types

import numpy as np
import pytest


def _run(monkeypatch, err, first_k, n_iter, p_floor=30000.0):
    from pgw4era5_b200 import _native as N
    from pgw4era5_b200 import engine as E
    from pgw4era5_b200 import settings
    monkeypatch.setattr(settings, "i_debug", 0)
    monkeypatch.setattr(E.torch.cuda, "stream", lambda s: contextlib.nullcontext())
    st = N.TimestepStatus()
    st.err = err
    for i, k in enumerate(first_k):
        st.first_k[i] = k
    st.result.n_iter, st.result.converged, st.result.rewritten = n_iter, 1, 0
    st.stats[0], st.stats[1] = 500.0, 100.0
    eng = object.__new__(E.PGWEngine)
    eng.deltas = types.SimpleNamespace(plev=np.array([100000.0, 100.0]))
    eng.stats = dict(timesteps=0, rewrites=0, reruns=0, launches=0)
    eng._n_hist, eng.k_pred, eng.ps_bound, eng.p_floor = [], 8, 110000.0, p_floor
    eng._zg_tables = (np.array([100000.0, 92500.0, 85000.0, 50000.0, 30000.0, 20000.0, 10000.0]), None)
    reruns = []
    eng.submit = lambda *a, **k: reruns.append(eng.p_floor) or types.SimpleNamespace(result=lambda: "rerun")
    p = types.SimpleNamespace(snapshot=lambda: st, out={}, ctx=dict(
        ignore_top=True, k_spec=8, k_max=19, file_name="f", stream=None, era=None, when=None, slot=0,
        direct=False, local_pref=True))
    return E.PGWEngine._complete(eng, p), eng, reruns


def test_no_pref_raises_unless_only_in_speculative_iterations(monkeypatch):
    from pgw4era5_b200 import _native as N
    from pgw4era5_b200.staged import MSG_NO_PREF
    big = N.INT32_MAX
    with pytest.raises(ValueError) as e:
        _run(monkeypatch, N.ERR_NO_PREF, (big, big, 2, big), 6)
    assert str(e.value) == MSG_NO_PREF
    res, _, reruns = _run(monkeypatch, N.ERR_NO_PREF, (big, big, 6, big), 6)
    assert res["n_iter"] == 6 and not reruns


def test_stash_floor_is_lowered_one_zg_level_and_rerun(monkeypatch):
    from pgw4era5_b200 import _native as N
    big = N.INT32_MAX
    res, eng, reruns = _run(monkeypatch, N.ERR_PREF_FLOOR, (big, big, big, 1), 6)
    assert res == "rerun" and reruns == [20000.0] and eng.stats["reruns"] == 1
    res, _, reruns = _run(monkeypatch, N.ERR_PREF_FLOOR, (big, big, big, 7), 6)
    assert res["n_iter"] == 6 and not reruns
    # NO_PREF that follows a column leaving the stash is a consequence of it: rerun, do not raise
    res, _, reruns = _run(monkeypatch, N.ERR_PREF_FLOOR | N.ERR_NO_PREF, (big, big, 3, 2), 6)
    assert res == "rerun"
    res, eng, reruns = _run(monkeypatch, N.ERR_PS_BOUND | N.ERR_NO_PREF, (big, 1, 4, big), 6)
    assert res == "rerun" and eng.ps_bound == 110000.0 * 1.25 and eng.p_floor == 30000.0

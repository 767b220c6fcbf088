"""Host side of the column-kernel plan (no GPU needed): pgw_timestep_plan_info on the level tables of
test_level_tables_gpu.py.  The cp.async flavour (PGW_COLUMN_PATH=generic) needs no driver, so its stash (lst, np)
and the FAST choice -- the ln series for every layer with s = (pb-pt)/(pb+pt) < 0.055 at ps in {p_ref, ps_bound} --
are checked here against a restatement of the rule in numpy."""
import ctypes as C

import numpy as np
import pytest

from test_level_tables_gpu import PLANS, TABLES, table

PS_BOUND = 110000.0


def _args(ak, bk, p_ref, flags=0, p_floor=30000.0, zg_plev=None):
    """pgw_timestep_args with the level table (ak, bk) and dummy device pointers (nothing is launched)."""
    from pgw4era5_b200 import _native as N
    keep = [np.ascontiguousarray(ak, dtype=np.float64), np.ascontiguousarray(bk, dtype=np.float64)]
    keep += [0.5 * (keep[0][1:] + keep[0][:-1]), 0.5 * (keep[1][1:] + keep[1][:-1])]
    dummy = 4096                                   # 16-byte aligned, never dereferenced by the plan
    a = N.TimestepArgs()
    a.ncol, a.nlev, a.nplev, a.nsoil, a.k_spec = 384, len(ak) - 1, 19, 0, 8
    for name, t in N.TimestepArgs._fields_:
        if t is N.c_fp:
            setattr(a, name, dummy)
        elif t is N.TSlab:
            setattr(a, name, N.TSlab(dummy, dummy, 1.0, 0.0))
    a.ak_host, a.bk_host, a.akm_host, a.bkm_host = (x.ctypes.data for x in keep)
    a.T_SO = a.T_SO_out = a.first_k = a.poly_fallback = 0
    a.p_ref, a.ps_bound, a.flags, a.p_floor = float(p_ref), PS_BOUND, flags, p_floor
    if zg_plev is not None:
        keep.append(np.ascontiguousarray(zg_plev, dtype=np.float64))
        a.zg_plev_host, a.nzg = keep[-1].ctypes.data, len(zg_plev)
    return a, keep


def _numpy_plan(ak, bk, p_stash):
    """stash_top and the FAST rule of pgw_timestep.cu, for the cp.async flavour."""
    nlev = len(ak) - 1
    h = np.nonzero(ak + PS_BOUND * bk >= p_stash)[0]
    lst = min(max((h[0] if len(h) else nlev) - 1, 0), nlev - 1)
    s = []
    for ps in (p_stash, PS_BOUND):
        p = ak + ps * bk
        s.append((p[lst + 1:] - p[lst:-1]) / (p[lst + 1:] + p[lst:-1]))
    fast = int(all(p[lst] > 0.0 for p in (ak + p_stash * bk, ak + PS_BOUND * bk)) and np.max(s) < 0.055)
    return dict(tma=0, fast=fast, lst=lst, np=nlev - lst, tmem_cols=0, l137=0)


@pytest.mark.parametrize("name,p_ref", list(PLANS))
def test_cp_async_plan_of_level_tables(name, p_ref, monkeypatch):
    from pgw4era5_b200 import _native as N
    monkeypatch.setenv("PGW_COLUMN_PATH", "generic")
    ak, bk = table(name)
    a, _keep = _args(ak, bk, p_ref)
    got = N.plan_info(a)
    fast, lst, np_ = PLANS[(name, p_ref)][1]
    assert got == dict(tma=0, fast=fast, lst=lst, np=np_, tmem_cols=0, l137=0)
    assert got == _numpy_plan(ak, bk, p_ref)
    assert N.lib.pgw_timestep_uses_tma(C.byref(a)) == 0


def test_flags_choose_their_instances(monkeypatch):
    """The per-column p_ref sizes the stash for p_floor; the reference-dtype instance has no FAST form; the
    thick layer of L137thick makes every flag take the exact-log instance."""
    from pgw4era5_b200 import _native as N
    from pgw4era5_b200.synthetic import PLEV19
    monkeypatch.setenv("PGW_COLUMN_PATH", "generic")
    for name, fast in (("L137", 1), ("L137thick", 0), ("L31", 0)):
        ak, bk = table(name)
        want = dict(tma=0, fast=fast, lst=PLANS[(name, 30000)][1][1], np=PLANS[(name, 30000)][1][2], tmem_cols=0,
                    l137=0)
        a, _k1 = _args(ak, bk, 85000.0, flags=N.FLAG_LOCAL_PREF, p_floor=30000.0, zg_plev=PLEV19)
        assert N.plan_info(a) == want, name
        a, _k2 = _args(ak, bk, 30000.0, flags=N.FLAG_REINTERP)
        assert N.plan_info(a) == want, name
        a, _k3 = _args(ak, bk, 30000.0, flags=N.FLAG_REF_DTYPES)
        assert N.plan_info(a) == dict(want, fast=0), name


def test_plan_info_rejects_invalid_args():
    from pgw4era5_b200 import _native as N
    ak, bk = table("L31")
    a, _keep = _args(ak, bk, 30000.0)
    a.nlev = 1
    info = (C.c_int * 6)()
    assert N.lib.pgw_timestep_plan_info(C.byref(a), C.byref(info)) == N.PGW_E_INVALID
    with pytest.raises(N.NativeError):
        N.plan_info(a)

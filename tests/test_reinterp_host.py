"""Host side of i_reinterp = 1 in the fused pass (no GPU needed): the library rejects PGW_FLAG_REINTERP together
with PGW_FLAG_LOCAL_PREF or PGW_FLAG_REF_DTYPES and never plans the TMA flavour for it, and PGWEngine.submit
routes the setting to the fused kernel or refuses the combinations that run through the staged path only."""
import ctypes as C
import types
from datetime import datetime

import numpy as np
import pytest
import torch

NY, NX, L, K = 8, 16, 137, 19


def _fake_engine():
    """A PGWEngine on CPU tensors: enough for _fill_args, which only takes addresses (nothing is launched)."""
    from pgw4era5_b200 import _native as N
    from pgw4era5_b200 import synthetic as S
    from pgw4era5_b200.engine import PGWEngine
    era = S.make_era5(NY, NX, 1)
    plev = np.asarray(S.PLEV19, dtype=np.float64)
    slab = N.TSlab(4096, 4096, 1.0, 0.0)
    eng = object.__new__(PGWEngine)
    eng.deltas = types.SimpleNamespace(
        ncol=NY * NX, shape2d=(NY, NX), vars={"zg": dict(plev=plev)}, plev=plev, plev_descending=int(plev[0] > plev[-1]),
        plev_dev=torch.as_tensor(plev), ts_clim=torch.zeros(NY * NX), slab4=lambda when: slab,
        slab=lambda name, when, level=None: slab)
    eng.device = torch.device("cpu")
    ak, bk = np.asarray(era["ak"], dtype=np.float64), np.asarray(era["bk"], dtype=np.float64)
    eng.ak, eng.bk = ak, bk
    eng.akm, eng.bkm = 0.5 * np.diff(ak) + ak[:-1], 0.5 * np.diff(bk) + bk[:-1]
    eng.ak_d, eng.bk_d, eng.akm_d, eng.bkm_d = (torch.as_tensor(x) for x in (eng.ak, eng.bk, eng.akm, eng.bkm))
    eng.nlev, eng.soil_decay, eng.ps_bound, eng.p_floor = L, np.exp(-np.asarray(era["soil1"]) / 2.8), 110000.0, 30000.0
    eng.k_pred, eng._zg_tables, eng._zg_level, eng._ws = 8, None, {}, {}
    status = N.TimestepStatus()
    eng._workspace = lambda ncol, max_iter, slot=0: dict(
        traj=torch.zeros(max_iter, ncol), status=torch.zeros(C.sizeof(status), dtype=torch.uint8), inflight=None)
    eng.alloc_outputs = lambda ny, nx, nsoil: {n: torch.zeros(s) for n, s in (
        ("PS", (1, ny, nx)), ("T_SKIN", (1, ny, nx)), ("FR_SEA_ICE", (1, ny, nx)), ("T_SO", (1, nsoil, ny, nx)),
        ("T", (1, L, ny, nx)), ("QV", (1, L, ny, nx)), ("U", (1, L, ny, nx)), ("V", (1, L, ny, nx)),
        ("delta_ps", (1, ny, nx)))}
    return eng, {k: v for k, v in era.items() if isinstance(v, torch.Tensor)}


def _args(monkeypatch, **kw):
    from pgw4era5_b200 import settings
    monkeypatch.setattr(settings, "i_reinterp", 0)
    for k, v in kw.items():
        monkeypatch.setattr(settings, k, v)
    eng, era = _fake_engine()
    return eng._fill_args(era, datetime(2006, 8, 2, 6))[0], eng


def test_reinterp_flag_is_set_and_plans_the_cp_async_flavour(monkeypatch):
    from pgw4era5_b200 import _native as N
    monkeypatch.setenv("PGW_COLUMN_PATH", "generic")
    a0, _ = _args(monkeypatch)
    a1, _ = _args(monkeypatch, i_reinterp=1)
    assert not a0.flags & N.FLAG_REINTERP and a1.flags == N.FLAG_REINTERP
    # the stash holds (T, RELHUM) of the ERA state in place of (T_pgw, e_pgw): the same bytes
    smem = N.lib.pgw_timestep_smem_bytes(C.byref(a1))
    assert smem > 0 and smem == N.lib.pgw_timestep_smem_bytes(C.byref(a0))
    monkeypatch.delenv("PGW_COLUMN_PATH")
    assert N.lib.pgw_timestep_uses_tma(C.byref(a1)) == 0


def test_library_rejects_reinterp_with_local_pref_or_reference_dtypes(monkeypatch):
    from pgw4era5_b200 import _native as N
    a, _ = _args(monkeypatch, p_ref_inp=None)                 # fills the PGW_FLAG_LOCAL_PREF arguments
    assert N.lib.pgw_timestep_smem_bytes(C.byref(a)) > 0
    for extra in (N.FLAG_LOCAL_PREF, N.FLAG_REF_DTYPES):
        b = N.TimestepArgs.from_buffer_copy(a)
        b.flags = N.FLAG_REINTERP | extra
        assert N.lib.pgw_timestep_smem_bytes(C.byref(b)) == N.PGW_E_INVALID
        assert N.lib.pgw_timestep_uses_tma(C.byref(b)) == N.PGW_E_INVALID
        assert N.lib.pgw_timestep(C.byref(b), None) == N.PGW_E_INVALID


@pytest.mark.parametrize("kw", [dict(p_ref_inp=None), dict(i_reference_dtypes=1)])
def test_submit_refuses_combinations(monkeypatch, kw):
    from pgw4era5_b200 import settings
    from pgw4era5_b200.engine import PGWEngine
    monkeypatch.setattr(settings, "i_reinterp", 1)
    for k, v in kw.items():
        monkeypatch.setattr(settings, k, v)
    eng = object.__new__(PGWEngine)
    eng._fill_args = lambda *a, **k: pytest.fail("reached the fused pass")
    with pytest.raises(ValueError, match="staged path"):
        eng.submit({}, datetime(2006, 8, 2, 6))


def test_submit_routes_reinterp_to_the_fused_pass(monkeypatch):
    from pgw4era5_b200 import settings
    from pgw4era5_b200.engine import PGWEngine
    monkeypatch.setattr(settings, "i_reinterp", 1)

    class Routed(Exception):
        pass

    def fill(*a, **k):
        raise Routed()

    eng = object.__new__(PGWEngine)
    eng._fill_args = fill
    with pytest.raises(Routed):
        eng.submit({}, datetime(2006, 8, 2, 6))

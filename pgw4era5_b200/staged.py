"""
The staged per-timestep path: the loop of the reference's ``pgw_for_era5``
(step_03_apply_to_era.py:60-343) run stage by stage on float64 device arrays, every stage a
CUDA operator of libpgw_b200 (the drop-ins of ``functions.py`` plus the small kernels of
csrc/pgw_staged.cu).  It covers the settings the fused column kernel does not:

* ``i_reinterp = 1`` (settings.py:150): the ERA state and the deltas are re-interpolated onto the
  updated model levels in every iteration (:202-216) and ua/va at the end (:330-343);
* ``p_ref_inp = None``: the reference pressure is picked per column and iteration among the zg
  pressure levels (:219-251, determine_p_ref functions.py:583-598).

It mirrors the reference statement by statement (float64 after promotion, one field-wide
max|error| per iteration) and is not a performance path: ~30 kernel launches and a host
synchronisation per iteration.
"""
import ctypes as C

import numpy as np
import torch

from . import _native as N
from . import functions as F
from . import settings
from .constants import CON_G

MSG_NO_PREF = ('No reference pressure level above the required local minimum pressure level could not '
               'be found everywhere. This is likely the case because your geopotential data set does '
               'not reach up high enough (e.g. only to 500 hPa instead of e.g. 300 hPa?)')


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _axpy(x, y, alpha=1.0):
    out = torch.empty_like(x)
    N.check(N.lib.pgw_axpy_f64(_p(x), _p(y), float(alpha), _p(out), x.numel(), _stream()), "pgw_axpy_f64")
    return out


def _hybrid(ps, a, b, ny, nx):
    """a[l] + ps * b[l]  ->  [1, len(a), ny, nx]"""
    out = torch.empty((1, a.numel(), ny, nx), device=ps.device, dtype=torch.float64)
    N.check(N.lib.pgw_hybrid_pressure_f64(_p(ps), _p(a), _p(b), _p(out), a.numel(), ny * nx, _stream()),
            "pgw_hybrid_pressure_f64")
    return out


def _blend(ds, name, when, level=None):
    """load_delta's two-point time interpolation (functions.py:288-292) of one resident delta:
    float64 arithmetic, float32 storage (pgw_time_interp_f32), returned as float64."""
    b = ds.bracket(name, when)
    lo, hi = ds.stamp(name, b.ind_before), ds.stamp(name, b.ind_after)
    if level is not None:
        lo, hi = lo[level], hi[level]
    lo, hi = lo.contiguous(), hi.contiguous()
    out = torch.empty_like(lo)
    N.check(N.lib.pgw_time_interp_f32(_p(lo), _p(hi), b.x_hi, b.x_new, _p(out), lo.numel(), _stream()),
            "pgw_time_interp_f32")
    return out.to(torch.float64)


def apply_staged(eng, era, era_step_dt, out=None, ignore_top_pressure_error=False, file_name="<memory>"):
    """One ERA5 timestep through the staged path.  Same inputs and outputs as ``PGWEngine.apply``;
    with ``p_ref_inp = None`` the result also carries ``p_ref`` [1, ny, nx]."""
    try:
        return _apply_staged(eng, era, era_step_dt, out, ignore_top_pressure_error, file_name)
    finally:                                         # a streamed delta set keeps the stamps read here until then
        eng.deltas.hold(torch.cuda.current_stream())


def _apply_staged(eng, era, era_step_dt, out, ignore_top_pressure_error, file_name):
    ds = eng.deltas
    a, f, out, ws, _, _ = eng._fill_args(era, era_step_dt, out, k_spec=1)
    ny, nx = f["PS"].shape[-2:]
    ncol, L = ny * nx, eng.nlev
    dev = eng.device
    f64 = lambda t: t.to(torch.float64)

    # ---- sea ice, skin and soil (:103-146)
    N.check(N.lib.pgw_surface_update(C.byref(a), _stream()), "pgw_surface_update")

    # ---- pressures and RELHUM of the ERA state (:64-94)
    PS = f64(f["PS"]).reshape(ncol)
    FIS = f64(f["FIS"]).reshape(1, ny, nx)
    T, QV, U, V = (f64(f[k]).reshape(1, L, ny, nx) for k in ("T", "QV", "U", "V"))
    pa_hl_era = _hybrid(PS, eng.ak_d, eng.bk_d, ny, nx)
    pa_era = _hybrid(PS, eng.akm_d, eng.bkm_d, ny, nx)
    vars_era = {"ta": T, "hur": F.specific_to_relative_humidity(QV, pa_era, T), "ua": U, "va": V}

    # ---- deltas at the ERA5 time (load_delta, functions.py:195-303)
    K = len(ds.plev)
    d3 = {v: _blend(ds, v, era_step_dt).reshape(1, K, ny, nx) for v in ("ta", "hur", "ua", "va")}
    sfc = {"ta": _blend(ds, "tas", era_step_dt), "hur": _blend(ds, "hurs", era_step_dt)}
    ps_hist = _blend(ds, "ps_hist", era_step_dt)

    def delta_on(var, target_P):                     # load_delta_interp, functions.py:306-340
        if var in ("ta", "hur"):
            return F.vert_interp_delta(d3[var], target_P, sfc[var].reshape(1, ny, nx), ps_hist.reshape(1, ny, nx),
                                       ignore_top_pressure_error, plev=ds.plev)
        return F.vert_interp_delta(d3[var], target_P, None, None, ignore_top_pressure_error, plev=ds.plev)

    vars_pgw = {}
    if not settings.i_reinterp:                      # :155-173
        for var in ("ta", "hur", "ua", "va"):
            vars_pgw[var] = _axpy(vars_era[var], delta_on(var, pa_era))

    # ---- iterative surface-pressure adjustment (:182-319)
    zg = ds.vars["zg"]
    plev_zg = np.asarray(zg["plev"], dtype=np.float64)
    if settings.p_ref_inp is None:
        opts_d = torch.as_tensor(plev_zg, device=dev)
        dzg_all = _blend(ds, "zg", era_step_dt).reshape(len(plev_zg), ncol)
        zeros = torch.zeros(ncol, device=dev, dtype=torch.float64)
        p_min_era = _axpy(zeros, PS, 0.95)           # pa_hl_era at the surface half level * 0.95
    else:
        sel = np.nonzero(plev_zg == float(settings.p_ref_inp))[0]      # .sel(plev=p_ref), :294
        if len(sel) != 1:
            raise KeyError(float(settings.p_ref_inp))
        dzg_ref = _blend(ds, "zg", era_step_dt, level=int(sel[0])).reshape(ncol)
        zeros = torch.zeros(ncol, device=dev, dtype=torch.float64)
        dphi_clim = _axpy(zeros, dzg_ref, CON_G)
    delta_ps = torch.zeros(ncol, device=dev, dtype=torch.float64)
    adj_ps = torch.zeros(ncol, device=dev, dtype=torch.float64)
    maxerr = torch.zeros(1, device=dev, dtype=torch.float64)
    err_word = torch.zeros(1, device=dev, dtype=torch.int32)
    p_ref = p_ref_last = None
    errs = []
    it = 1
    thresh = float(settings.thresh_phi_ref_max_error)
    phi_ref_max_error = np.inf
    while phi_ref_max_error > thresh:
        delta_ps = _axpy(delta_ps, adj_ps)
        ps_pgw = _axpy(PS, delta_ps)
        pa_pgw = _hybrid(ps_pgw, eng.akm_d, eng.bkm_d, ny, nx)
        pa_hl_pgw = _hybrid(ps_pgw, eng.ak_d, eng.bk_d, ny, nx)
        if settings.i_reinterp:                      # :202-216
            for var in ("ta", "hur"):
                v_era = F.interp_logp_4d(vars_era[var], pa_era, pa_pgw, extrapolate='constant')
                vars_pgw[var] = _axpy(v_era, delta_on(var, pa_pgw))
        if settings.p_ref_inp is None:               # :219-251
            p_min_pgw = _axpy(zeros, ps_pgw, 0.95)
            p_ref = torch.empty(ncol, device=dev, dtype=torch.float64)
            N.check(N.lib.pgw_determine_p_ref_f64(_p(p_min_era), _p(p_min_pgw), _p(opts_d), len(plev_zg),
                                                  _p(p_ref_last), _p(p_ref), ncol, _p(err_word), _stream()),
                    "pgw_determine_p_ref_f64")
            if int(err_word.item()) & N.ERR_NO_PREF:
                raise ValueError(MSG_NO_PREF)
            p_ref_last = p_ref
            p_ref_arg = p_ref.reshape(1, ny, nx)
            sel_field = torch.empty(ncol, device=dev, dtype=torch.float64)
            N.check(N.lib.pgw_select_plev_f64(_p(dzg_all), _p(opts_d), len(plev_zg), _p(p_ref), _p(sel_field),
                                              ncol, _stream()), "pgw_select_plev_f64")
            dphi_clim = _axpy(zeros, sel_field, CON_G)
        else:
            p_ref_arg = float(settings.p_ref_inp)
        hus = F.relative_to_specific_humidity(vars_pgw["hur"], pa_pgw, vars_pgw["ta"])          # :262-266
        phi_pgw = F.integ_geopot(pa_hl_pgw, FIS, vars_pgw["ta"], hus, None, p_ref_arg)           # :269-276
        # the float32 T and QV of the file are handed over as they are: Rd * Tv in float32, like numpy (:144)
        phi_era = F.integ_geopot(pa_hl_era, FIS, f["T"].reshape(1, L, ny, nx), f["QV"].reshape(1, L, ny, nx),
                                 None, p_ref_arg)                                                 # :280-287
        ta_low = vars_pgw["ta"][0, L - 1].reshape(ncol).contiguous()
        maxerr.zero_()
        N.check(N.lib.pgw_ps_adjust_f64(_p(phi_pgw), _p(phi_era), _p(dphi_clim), _p(ps_pgw), _p(ta_low),
                                        float(settings.adj_factor), _p(adj_ps), _p(maxerr), ncol, _stream()),
                "pgw_ps_adjust_f64")
        phi_ref_max_error = float(maxerr.item())
        errs.append(phi_ref_max_error)
        if settings.i_debug >= 2:
            print('### iteration {:03d}, phi max error: {}'.format(it, phi_ref_max_error))
        it += 1
        if it > settings.max_n_iter:                 # :315-319
            from .engine import MSG_NOCONV
            raise ValueError(MSG_NOCONV.format(file_name))

    if settings.i_reinterp:                          # :330-343
        for var in ("ua", "va"):
            v_era = F.interp_logp_4d(vars_era[var], pa_era, pa_pgw, extrapolate='constant')
            vars_pgw[var] = _axpy(v_era, delta_on(var, pa_pgw))

    # ---- results, float32 like the ERA5 file (:360-364)
    out["PS"].copy_(ps_pgw.reshape(out["PS"].shape))
    out["delta_ps"].copy_(delta_ps.reshape(out["delta_ps"].shape))
    for name, key in (("T", "ta"), ("U", "ua"), ("V", "va")):
        out[name].copy_(vars_pgw[key].reshape(out[name].shape))
    out["QV"].copy_(hus.reshape(out["QV"].shape))
    eng.stats["timesteps"] += 1
    res = dict(out)
    res["n_iter"] = it - 1
    res["phi_max_errors"] = errs
    if p_ref is not None:
        res["p_ref"] = p_ref.reshape(1, ny, nx)
    return res

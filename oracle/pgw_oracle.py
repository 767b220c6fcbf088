"""
TEST INFRASTRUCTURE ONLY -- CPU oracle for the PGW4ERA5 per-timestep path.

This module is a float64 numpy restatement of the reference algorithm.  It is
the *checker* for the CUDA path: only ``tests/``, ``__graft_entry__.smoke()``
and the ``cpu_baseline`` / ``--impl reference`` legs of ``bench.py`` may import
it.  Nothing under ``pgw4era5_b200/`` imports it; the product path fails loudly
when the CUDA library is missing.

Pinning status (see DESIGN.md section 5).  The reference has no tests and ships no data, and it
needs xarray, which the build container lacks; the oracle is pinned by EXECUTING the reference in
the build container and committing what it returns:
  * ``oracle/make_golden.py`` -> tests/golden/reference_functions.npz: the numpy/numba functions of
    /root/reference/functions.py imported unmodified (xarray/pyvista/pyproj stubbed): interp_extrap_1d,
    interp_1d_for_timelatlon, replace_delta_sfc, determine_p_ref, integrate_tos,
    harmonic_ac_analysis, the humidity helpers, dt64_to_dt.  Bit-exact (tests/test_oracle_golden.py).
  * ``oracle/make_golden_glue.py`` -> tests/golden/reference_glue.npz: the xarray-bound functions
    (integ_geopot, load_delta, load_delta_interp, vert_interp_delta, interp_logp_4d, regrid_lat_lon,
    filter_data, the alpha-blended saturation pressure) and the WHOLE of step_03's pgw_for_era5
    (six settings), run unmodified over ``oracle/xrlite.py``, a restatement of the xarray semantics
    they use.  tests/test_oracle_glue_golden.py: identical iteration counts and per-iteration max
    errors, PS to 2e-10 Pa, functions to float64 round-off.
  * scipy's interp1d (the arithmetic behind xarray ``.interp``): tests/test_oracle_properties.py.
  * PARITY UNPINNED for xarray itself only: xrlite restates its documented behaviour.
Each function cites the file:line it restates.

All arrays are numpy, C-order, dims ``(time, level, lat, lon)``.
"""
import math
import ctypes
import os
from datetime import datetime, timezone

import numpy as np

# constants.py:3-7
CON_RD = 287.05
CON_G = 9.80665
CON_MW_MD = 0.622


# ---------------------------------------------------------------------------
# optional compiled column loops (oracle/oracle_kernels.c), same algorithm as
# the reference's two numba functions; built by oracle/build.py
# ---------------------------------------------------------------------------
_HERE = os.path.dirname(os.path.abspath(__file__))
_CLIB = None


def _clib():
    global _CLIB
    if _CLIB is None:
        path = os.path.join(_HERE, "_build", "liboracle_kernels.so")
        if not os.path.exists(path):
            from . import build as _b  # type: ignore
            _b.build()
        lib = ctypes.CDLL(path)
        dp = ctypes.POINTER(ctypes.c_double)
        lib.oracle_interp_1d_for_timelatlon.argtypes = [
            dp, dp, dp, dp, ctypes.c_long, ctypes.c_long, ctypes.c_long,
            ctypes.c_long, ctypes.c_long, ctypes.c_int]
        lib.oracle_interp_1d_for_timelatlon.restype = ctypes.c_int
        lib.oracle_replace_delta_sfc.argtypes = [
            dp, dp, dp, dp, dp, dp, ctypes.c_long, ctypes.c_long]
        lib.oracle_replace_delta_sfc.restype = ctypes.c_int
        _CLIB = lib
    return _CLIB


def _dptr(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_double))


# ---------------------------------------------------------------------------
# humidity (functions.py:58-125)
# ---------------------------------------------------------------------------
def specific_humidity_to_vapor_pressure(hus, pa):
    """functions.py:58-64"""
    return hus * pa / (CON_MW_MD + 0.378 * hus)


def vapor_pressure_to_specific_humidity(vapp, pa):
    """functions.py:66-72"""
    return CON_MW_MD * vapp / (pa - (1 - CON_MW_MD) * vapp)


def saturation_vapor_pressure_water_or_ice(pa, ta, water=True):
    """functions.py:74-89 (IFS 7.93)"""
    T0 = 273.16
    if water:
        a1, a3, a4 = 611.21, 17.502, 32.19
    else:
        a1, a3, a4 = 611.21, 22.587, -0.7
    return a1 * np.exp(a3 * (ta - T0) / (ta - a4))


def saturation_vapor_pressure_water_and_ice(pa, ta):
    """functions.py:91-105 (IFS 7.92): alpha blend of water and ice."""
    T0 = 273.16
    Ti = 250.16
    ta = np.asarray(ta)                  # the dtype of ta is kept, as in the reference
    if ta.dtype.kind != "f":
        ta = ta.astype(np.float64)
    alpha = np.full_like(ta, np.nan)
    alpha = np.where(ta >= T0, 1, alpha)
    alpha = np.where(ta <= Ti, 0, alpha)
    with np.errstate(invalid="ignore"):
        alpha = np.where((ta < T0) & (ta > Ti),
                         np.power((ta - Ti) / (T0 - Ti), 2.), alpha)
    return (alpha * saturation_vapor_pressure_water_or_ice(pa, ta, True) +
            (1 - alpha) * saturation_vapor_pressure_water_or_ice(pa, ta, False))


def specific_to_relative_humidity(hus, pa, ta):
    """functions.py:107-116"""
    return (specific_humidity_to_vapor_pressure(hus, pa) /
            saturation_vapor_pressure_water_and_ice(pa, ta)) * 100


def relative_to_specific_humidity(hur, pa, ta):
    """functions.py:118-125 (no clipping of hur)"""
    vapp = hur / 100 * saturation_vapor_pressure_water_and_ice(pa, ta)
    return vapor_pressure_to_specific_humidity(vapp, pa)


# ---------------------------------------------------------------------------
# geopotential (functions.py:128-189)
# ---------------------------------------------------------------------------
def integ_geopot(pa_hl, zgs, ta, hus, p_ref, phi_dtype=np.float64):
    """
    functions.py:128-189.  pa_hl [nt,L+1,ny,nx], zgs [nt,ny,nx], ta/hus
    [nt,L,ny,nx], p_ref scalar or [nt,ny,nx].  Half-level labels are assumed
    1..L+1 and full-level labels 1..L (so ``level = hl_ref_star - 1`` is the
    layer just above the selected half level, functions.py:176).

    dtypes as in the reference, where they follow from numpy's promotion rules: ``ta``/``hus`` are
    NOT promoted -- with the float32 fields of an ERA5 file, ``tav`` (:144) and ``CON_RD * tav``
    (:151, :177) are float32 products, with the float64 PGW state they are float64.  ``phi_dtype``
    is the dtype the half-level geopotential is stored in (:141 copies the dtype of FIS: float32
    for a real ERA5 file; float64, the default here, when FIS is stored as double).
    Pinned by tests/test_oracle_glue_golden.py against the reference executed over oracle/xrlite.py.
    """
    pa_hl = np.asarray(pa_hl, dtype=np.float64)
    ta = np.asarray(ta)
    hus = np.asarray(hus)
    zgs = np.asarray(zgs)
    pa_hl = np.where(pa_hl > 0, pa_hl, 0.0001)              # :135
    lnp = np.log(pa_hl)
    dlnpa = lnp[:, 1:] - lnp[:, :-1]                         # :136-138
    tav = ta * (1 + 0.61 * hus)                              # :144
    nl = ta.shape[1]
    phi_hl = np.empty(pa_hl.shape, dtype=phi_dtype)
    phi_hl[:, nl] = zgs                                      # :141
    for l in range(nl - 1, -1, -1):                          # :147-152
        phi_hl[:, l] = phi_hl[:, l + 1] + (CON_RD * tav[:, l] * dlnpa[:, l])
    p_ref_b = np.asarray(p_ref, dtype=np.float64)
    if p_ref_b.ndim == 3:
        p_ref_b = p_ref_b[:, None]
    p_diff = pa_hl - p_ref_b                                 # :160-161
    with np.errstate(invalid="ignore"):
        p_diff = np.where(p_diff >= 0, p_diff, np.nan)
    if np.any(np.all(np.isnan(p_diff), axis=1)):             # :162-165
        raise ValueError("p_ref locally lies below the surface. Please set a "
                         "lower reference pressue (p_ref_inp) in settings.py")
    ind = np.nanargmin(p_diff, axis=1)                       # [nt,ny,nx]
    idx = ind[:, None]
    p_ref_star = np.take_along_axis(pa_hl, idx, axis=1)[:, 0]
    phi_ref_star = np.take_along_axis(phi_hl, idx, axis=1)[:, 0]
    if np.any(ind < 1):
        raise KeyError("reference half level has no full level above it")
    tav_star = np.take_along_axis(tav, idx - 1, axis=1)[:, 0]
    p_ref_s = np.asarray(p_ref, dtype=np.float64)
    phi_ref = (phi_ref_star - (CON_RD * tav_star) *
               (np.log(p_ref_s) - np.log(p_ref_star)))       # :174-179
    return phi_ref


# ---------------------------------------------------------------------------
# time handling of climate deltas (functions.py:39-51, 195-303)
# ---------------------------------------------------------------------------
def dt64_to_dt(dt64):
    """functions.py:39-51 (seconds since epoch -> naive UTC datetime)."""
    timestamp = ((np.datetime64(dt64, "ns") - np.datetime64("1970-01-01T00:00:00"))
                 / np.timedelta64(1, "s"))
    return datetime.fromtimestamp(float(timestamp), tz=timezone.utc).replace(tzinfo=None)


def delta_time_bracket(times, target_date_time):
    """
    Calendar logic of load_delta, functions.py:223-292, without the file I/O.

    times: datetime64 stamps of the delta file (12 monthly or 365/366 daily).
    Returns (keep, ind_before, ind_after, x_hi, x_new) where ``keep`` indexes
    the stamps left after dropping 29 Feb, ind_* index into the kept stamps,
    and the two floats are the nanosecond abscissae xarray hands to scipy
    (offset = the 'before' stamp).  ind_before == ind_after means exact hit.
    """
    times = np.asarray(times).astype("datetime64[ns]")
    keep = []
    leap = None
    for i, t in enumerate(times):                            # :224-230
        dt = dt64_to_dt(t)
        if dt.month == 2 and dt.day == 29:
            leap = i
    keep = [i for i in range(len(times)) if i != leap]
    stamps = []
    for i in keep:                                           # :235-238
        stamps.append(np.datetime64(
            dt64_to_dt(times[i]).replace(year=target_date_time.year), "ns"))
    stamps = np.array(stamps, dtype="datetime64[ns]")
    tgt = np.datetime64(target_date_time, "ns")
    is_before = stamps <= tgt                                # :242-258
    if np.sum(is_before) > 0:
        ind_before = int(np.argwhere(is_before)[-1].squeeze())
        t_before = stamps[ind_before]
    else:
        ind_before = -1
        t_before = np.datetime64(dt64_to_dt(stamps[-1]).replace(
            year=target_date_time.year - 1), "ns")
    is_after = stamps >= tgt                                 # :262-278
    if np.sum(is_after) > 0:
        ind_after = int(np.argwhere(is_after)[0].squeeze())
        t_after = stamps[ind_after]
    else:
        ind_after = 0
        t_after = np.datetime64(dt64_to_dt(stamps[0]).replace(
            year=target_date_time.year + 1), "ns")
    # xarray _floatize_x: offset = min stamp, float64 nanoseconds
    x_hi = float((t_after - t_before) / np.timedelta64(1, "ns"))
    x_new = float((tgt - t_before) / np.timedelta64(1, "ns"))
    return keep, ind_before, ind_after, x_hi, x_new


def interp1d_linear_2pt(y_lo, y_hi, x_hi, x_new):
    """scipy interp1d._call_linear (scipy 1.9.3) with x = [0, x_hi]."""
    slope = (y_hi - y_lo) / (x_hi - 0.0)
    return slope * (x_new - 0.0) + y_lo


def load_delta(delta, target_date_time=None):
    """
    functions.py:195-303 on an in-memory delta {'time': datetime64[nt],
    'data': [nt,(K),ny,nx], 'plev': [K] or None}.  Returns the time-interpolated
    field with a leading time axis of length 1 ([1,(K),ny,nx], float64), or the
    full series (29 Feb dropped) if target_date_time is None.
    """
    data = np.asarray(delta["data"], dtype=np.float64)
    keep, ib, ia, x_hi, x_new = delta_time_bracket(
        delta["time"], target_date_time if target_date_time is not None
        else dt64_to_dt(np.asarray(delta["time"]).astype("datetime64[ns]")[0]))
    data = data[keep]
    if target_date_time is None:                             # :300-301
        return data
    if ib == ia:                                             # :282-283
        return data[ib][None]
    return interp1d_linear_2pt(data[ib], data[ia], x_hi, x_new)[None]


# ---------------------------------------------------------------------------
# vertical interpolation (functions.py:343-580)
# ---------------------------------------------------------------------------
_MODES = {"off": 0, "linear": 1, "constant": 2, "nan": 3}


def interp_extrap_1d(src_x, src_y, targ_x, extrapolate):
    """functions.py:511-580, pure-Python restatement (small cases only)."""
    n = len(src_x)
    targ_y = np.zeros(len(targ_x))
    for ti in range(len(targ_x)):
        i1 = i2 = -1
        require_extrap = False
        for si in range(n):
            if si == 0 and src_x[si] > targ_x[ti]:           # :530-538
                if extrapolate == "linear":
                    i1, i2 = si, si + 1
                elif extrapolate == "constant":
                    i1, i2 = si, si
                require_extrap = True
                break
            elif src_x[si] == targ_x[ti]:                    # :540-543
                i1 = i2 = si
                break
            elif src_x[si] > targ_x[ti]:                     # :545-548
                i1, i2 = si - 1, si
                break
        if i1 == -1:                                         # :554-561
            if extrapolate == "linear":
                i1, i2 = n - 2, n - 1
            elif extrapolate == "constant":
                i1 = i2 = n - 1
            require_extrap = True
        if require_extrap and extrapolate == "off":          # :564-566
            raise ValueError("Extrapolation deactivated but data out of bounds.")
        if require_extrap and extrapolate == "nan":          # :569-570
            targ_y[ti] = np.nan
        elif i1 == i2:
            targ_y[ti] = src_y[i1]
        else:
            targ_y[ti] = (src_y[i1] + (targ_x[ti] - src_x[i1]) *
                          (src_y[i2] - src_y[i1]) / (src_x[i2] - src_x[i1]))
    return targ_y


def interp_1d_for_timelatlon(orig_array, src_p, targ_p, interp_array,
                             ntime, nlat, nlon, extrapolate):
    """functions.py:479-508 via the compiled C restatement (same loops)."""
    lib = _clib()
    for a in (orig_array, src_p, targ_p, interp_array):
        assert a.dtype == np.float64 and a.flags.c_contiguous
    rc = lib.oracle_interp_1d_for_timelatlon(
        _dptr(orig_array), _dptr(src_p), _dptr(targ_p), _dptr(interp_array),
        ntime, src_p.shape[1], targ_p.shape[1], nlat, nlon, _MODES[extrapolate])
    if rc == 1:
        raise ValueError("Source pressure values must be ascending!")
    if rc == 2:
        raise ValueError("Target pressure values must be ascending!")
    if rc == 3:
        raise ValueError("Extrapolation deactivated but data out of bounds.")


def interp_logp_4d(var, source_P, targ_P, extrapolate="off"):
    """functions.py:434-477"""
    if extrapolate not in _MODES:
        raise ValueError('Invalid input value for "extrapolate"')
    var = np.ascontiguousarray(var, dtype=np.float64)
    source_P = np.ascontiguousarray(source_P, dtype=np.float64)
    targ_P = np.ascontiguousarray(targ_P, dtype=np.float64)
    if var.shape[0] != source_P.shape[0] or var.shape[0] != targ_P.shape[0]:
        raise ValueError("Time dimension of input files is inconsistent!")
    if var.shape[2] != source_P.shape[2] or var.shape[2] != targ_P.shape[2]:
        raise ValueError("Lat dimension of input files is inconsistent!")
    if var.shape[3] != source_P.shape[3] or var.shape[3] != targ_P.shape[3]:
        raise ValueError("Lon dimension of input files is inconsistent!")
    tmp = np.zeros_like(targ_P)
    with np.errstate(divide="ignore"):
        interp_1d_for_timelatlon(var, np.log(source_P), np.log(targ_P), tmp,
                                 targ_P.shape[0], targ_P.shape[2],
                                 targ_P.shape[3], extrapolate)
    return tmp


def replace_delta_sfc(source_P, ps_hist, delta, delta_sfc):
    """functions.py:343-366 for ONE column (1-D source_P ascending)."""
    out_source_P = source_P.copy()
    out_delta = delta.copy()
    if ps_hist > np.max(source_P):
        sfc_ind = len(source_P) - 1
        out_source_P[sfc_ind] = ps_hist
        out_delta[sfc_ind] = delta_sfc
    elif ps_hist < np.min(source_P):
        raise ValueError()
    else:
        sfc_ind = np.max(np.argwhere(ps_hist > source_P))
        out_delta[sfc_ind:] = delta_sfc
        out_source_P[sfc_ind] = ps_hist
    return out_source_P, out_delta


def replace_delta_sfc_4d(source_P, ps_hist, delta, delta_sfc):
    """apply_ufunc(vectorize=True) of replace_delta_sfc, functions.py:396-404."""
    lib = _clib()
    source_P = np.ascontiguousarray(source_P, dtype=np.float64)
    delta = np.ascontiguousarray(delta, dtype=np.float64)
    ps_hist = np.ascontiguousarray(np.broadcast_to(ps_hist, delta[:, 0].shape), dtype=np.float64)
    delta_sfc = np.ascontiguousarray(np.broadcast_to(delta_sfc, delta[:, 0].shape), dtype=np.float64)
    out_P = np.empty_like(source_P)
    out_d = np.empty_like(delta)
    nt, K, ny, nx = delta.shape
    rc = lib.oracle_replace_delta_sfc(_dptr(source_P), _dptr(ps_hist), _dptr(delta),
                                      _dptr(delta_sfc), _dptr(out_P), _dptr(out_d),
                                      K, nt * ny * nx) if nt == 1 else None
    if rc is None:
        for t in range(nt):
            p1, d1 = replace_delta_sfc_4d(source_P[t:t + 1], ps_hist[t:t + 1],
                                          delta[t:t + 1], delta_sfc[t:t + 1])
            out_P[t], out_d[t] = p1[0], d1[0]
        return out_P, out_d
    if rc != 0:
        raise ValueError()
    return out_P, out_d


def vert_interp_delta(delta, plev, target_P, delta_sfc=None, ps_hist=None,
                      ignore_top_pressure_error=False):
    """
    functions.py:369-431.  delta [1,K,ny,nx] on pressure levels ``plev`` in file
    order; target_P [1,L,ny,nx]; delta_sfc/ps_hist [1,ny,nx] or None.
    """
    delta = np.asarray(delta, dtype=np.float64)[:, ::-1]     # :383-384
    plev_r = np.asarray(plev, dtype=np.float64)[::-1]
    source_P = np.broadcast_to(plev_r[None, :, None, None], delta.shape).copy()  # :387-391
    if delta_sfc is not None:                                # :395-404
        source_P, delta = replace_delta_sfc_4d(source_P, ps_hist, delta, delta_sfc)
    if np.min(target_P) < np.min(source_P):                  # :417-425
        if not ignore_top_pressure_error:
            raise ValueError("ERA5 top pressure is lower than climate delta top pressure.")
    return interp_logp_4d(delta, source_P, target_P, extrapolate="constant")  # :429


def determine_p_ref(p_min_era, p_min_pgw, p_ref_opts, p_ref_last=None):
    """functions.py:583-598"""
    for p in p_ref_opts:
        if (p_min_era > p) & (p_min_pgw > p):
            if p_ref_last is None:
                return p
            return min(p, p_ref_last)
    return None


def integrate_tos(tos_field, ts_field, land_frac, ice_frac):
    """functions.py:1145-1186"""
    dims = tos_field.shape
    ice = np.asarray(ice_frac, dtype=np.float64).reshape(-1)
    tos = np.asarray(tos_field, dtype=np.float64).reshape(-1)
    ts = np.asarray(ts_field, dtype=np.float64).reshape(-1)
    land = np.asarray(land_frac, dtype=np.float64).reshape(-1)
    mask = ~np.isnan(ice) & ~np.isnan(tos)
    out = ts.copy()
    ts_frac = np.clip(ice[mask] + land[mask], 0, 1)
    out[mask] = ts_frac * ts[mask] + (1 - ts_frac) * tos[mask]
    return out.reshape(dims)


# ---------------------------------------------------------------------------
# step_02: smoothing and regridding (functions.py:606-898)
# ---------------------------------------------------------------------------
def harmonic_ac_analysis(ts):
    """functions.py:678-740: mean + first three annual harmonics."""
    ts = np.asarray(ts, dtype=np.float64)
    if np.any(np.isnan(ts)):
        return np.full_like(ts, np.nan)
    mean = ts.mean()
    lt = len(ts)
    P = lt
    hcts = np.zeros((4, lt))
    timevector = np.arange(1, lt + 1, 1)
    q = math.floor(P / 2.)
    for i in range(1, 4):
        if i < q:
            bracket = 2. * math.pi * i / P * timevector
            a = 2. / lt * (ts.dot(np.cos(bracket)))
            b = 2. / lt * (ts.dot(np.sin(bracket)))
            hcts[i - 1, :] = a * np.cos(bracket) + b * np.sin(bracket)
        else:
            raise SystemExit("reconstruction grade larger than len/2")
    return sum(hcts[0:3, :]) + mean


def filter_data(diff):
    """functions.py:639-667 on an array [nt,(K),ny,nx]; vectorised over grid points
    (dot products via einsum keep the reference's summation per series only up to
    float64 rounding, documented tolerance 1e-12 relative)."""
    diff = np.asarray(diff, dtype=np.float64)
    nt = diff.shape[0]
    flat = diff.reshape(nt, -1)
    out = np.empty_like(flat)
    for j in range(flat.shape[1]):
        out[:, j] = harmonic_ac_analysis(flat[:, j])
    return out.reshape(diff.shape)


def filter_data_fast(diff):
    """Same maths as filter_data but whole-array (used for larger checks)."""
    diff = np.asarray(diff, dtype=np.float64)
    nt = diff.shape[0]
    flat = diff.reshape(nt, -1)
    tv = np.arange(1, nt + 1, 1)
    out = np.tile(flat.mean(axis=0), (nt, 1))
    for i in range(1, 4):
        br = 2. * math.pi * i / nt * tv
        c, s = np.cos(br), np.sin(br)
        a = 2. / nt * (c @ flat)
        b = 2. / nt * (s @ flat)
        out += np.outer(c, a) + np.outer(s, b)
    bad = np.any(np.isnan(flat), axis=0)
    out[:, bad] = np.nan
    return out.reshape(diff.shape)


def _interp1d_axis(x, y, x_new, axis):
    """scipy interp1d(kind='linear', bounds_error=False, fill_value=nan)
    (scipy 1.9.3 interpolate/_interpolate.py:_call_linear) along ``axis``."""
    x = np.asarray(x, dtype=np.float64)
    x_new = np.asarray(x_new, dtype=np.float64)
    y = np.moveaxis(np.asarray(y, dtype=np.float64), axis, 0)
    idx = np.searchsorted(x, x_new)
    idx = idx.clip(1, len(x) - 1).astype(int)
    lo = idx - 1
    hi = idx
    x_lo, x_hi = x[lo], x[hi]
    y_lo, y_hi = y[lo], y[hi]
    shp = (-1,) + (1,) * (y.ndim - 1)
    slope = (y_hi - y_lo) / (x_hi - x_lo).reshape(shp)
    y_new = slope * (x_new - x_lo).reshape(shp) + y_lo
    oob = (x_new < x[0]) | (x_new > x[-1])
    y_new[oob] = np.nan
    return np.moveaxis(y_new, 0, axis)


def _nanmean_lastaxis(x):
    """xarray's DataArray.mean(dim=...) on float data (skipna): the mean of the valid points, NaN if none."""
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", RuntimeWarning)       # "Mean of empty slice" for an all-NaN row
        return np.nanmean(x, axis=-1, keepdims=True)


def regrid_lat_lon(data, lat_gcm, lon_gcm, targ_lat, targ_lon):
    """
    functions.py:748-898 (xarray-only branch).  data [..., nlat_gcm, nlon_gcm]
    -> [..., len(targ_lat), len(targ_lon)], float64.
    """
    data = np.asarray(data, dtype=np.float64)
    lat = np.asarray(lat_gcm, dtype=np.float64).copy()
    lon = np.asarray(lon_gcm, dtype=np.float64).copy()
    targ_lat = np.asarray(targ_lat, dtype=np.float64)
    targ_lon = np.asarray(targ_lon, dtype=np.float64)
    dlon_gcm = np.median(np.diff(lon))                       # :778-789
    dlat_gcm = np.median(np.diff(lat))
    periodic_lon = (dlon_gcm + np.max(lon) - np.min(lon)) >= 359.9
    if lat[0] > lat[-1]:                                     # :822-829
        lat = lat[::-1]
        data = data[..., ::-1, :]
    # the pole rows are xarray means over lon, which skip NaN (all-NaN row -> NaN)
    if np.max(targ_lat) + dlat_gcm > 89.9:                   # :833-837
        north = np.broadcast_to(_nanmean_lastaxis(data[..., -1:, :]), data[..., -1:, :].shape)
        data = np.concatenate([data, north], axis=-2)
        lat = np.concatenate([lat, [90.0]])
    if np.min(targ_lat) - dlat_gcm < -89.9:                  # :838-842
        south = np.broadcast_to(_nanmean_lastaxis(data[..., :1, :]), data[..., :1, :].shape)
        data = np.concatenate([south, data], axis=-2)
        lat = np.concatenate([[-90.0], lat])
    if (np.max(targ_lat) > np.max(lat)) or (np.min(targ_lat) < np.min(lat)):  # :845-856
        raise ValueError("ERA5 dataset extends further North or South than GCM dataset!")
    data = _interp1d_axis(lat, data, targ_lat, axis=data.ndim - 2)   # :859
    if periodic_lon:                                         # :866-874
        if np.max(targ_lon) > np.max(lon):
            data = np.concatenate([data, data], axis=-1)
            lon = np.concatenate([lon, lon + 360])
        if np.min(targ_lon) < np.min(lon):
            # lon_below is the *current* dataset (incl. a +360 copy) shifted by -360
            data = np.concatenate([data, data], axis=-1)
            lon = np.concatenate([lon - 360, lon])
    if (np.max(targ_lon) > np.max(lon)) or (np.min(targ_lon) < np.min(lon)):  # :877-888
        raise ValueError("ERA5 dataset extends further East or West than GCM dataset!")
    return _interp1d_axis(lon, data, targ_lon, axis=data.ndim - 1)   # :892


# ---------------------------------------------------------------------------
# NaN-ignoring Gaussian-kernel regridding of tos / siconc (functions.py:900-1060)
#
# PARITY UNPINNED: the arithmetic lives in two third-party packages that are neither vendored in
# /root/reference nor installed here -- pyproj 3.4.0 (``Geod(ellps="WGS84").inv``, PROJ's geodesic.c
# after Karney 2013) and pyvista 0.37.0 / vtk 9.2.2 (``PolyData.interpolate`` = vtkPointInterpolator
# with a vtkGaussianKernel on a radius footprint, null-points strategy NULL_VALUE).  Their published
# algorithms are restated: geodesic distances from the exact integrals of Karney (2013), eqs 7-8,
# evaluated by Gauss-Legendre quadrature (the three distances the reference asks for are a meridian
# arc, a geodesic between two points of EQUAL latitude and the distance to the point 180 degrees
# away, which runs over the pole); the kernel as in vtkGaussianKernel::ComputeWeights:
# w_i = exp(-(sharpness/radius)^2 d_i^2) over the points with d_i <= radius, normalised; an exact hit
# (d^2 < 256 eps) takes that point's value; no point in the radius -> null value.
# ---------------------------------------------------------------------------
WGS84_A = 6378137.0
WGS84_F = 1.0 / 298.257223563
_GLX, _GLW = np.polynomial.legendre.leggauss(32)


def _quad(f, lo, hi):
    """Gauss-Legendre integral of f over [lo, hi] (arrays broadcast against the node axis)."""
    lo, hi = np.asarray(lo, dtype=np.float64), np.asarray(hi, dtype=np.float64)
    mid, half = 0.5 * (hi + lo), 0.5 * (hi - lo)
    return half * np.sum(_GLW * f(mid[..., None] + half[..., None] * _GLX), axis=-1)


def wgs84_meridian_arc(lat_deg):
    """Distance along the meridian from the equator to |lat| [m]: Karney (2013) eq. 7 with alpha0 = 0
    (sigma = reduced latitude, k = e'), i.e. what ``geod.inv(lon, 0, lon, lat)`` returns."""
    f = WGS84_F
    b = WGS84_A * (1 - f)
    ep2 = f * (2 - f) / (1 - f) ** 2
    beta = np.arctan((1 - f) * np.tan(np.radians(np.abs(np.asarray(lat_deg, dtype=np.float64)))))
    return b * _quad(lambda s: np.sqrt(1 + ep2 * np.sin(s) ** 2), np.zeros_like(beta), beta)


def wgs84_same_lat_distance(lat_deg, dlon_deg):
    """Geodesic distance [m] between (lat, 0) and (lat, dlon), 0 <= dlon <= 180, i.e. what
    ``geod.inv(0, lat, lon, lat)`` returns.  By symmetry the vertex of the geodesic lies half way;
    the azimuth alpha0 at the equator crossing is found by bisection on the longitude integral
    (Karney 2013, eq. 8), the distance follows from eq. 7."""
    f = WGS84_F
    b = WGS84_A * (1 - f)
    ep2 = f * (2 - f) / (1 - f) ** 2
    lat = np.abs(np.asarray(lat_deg, dtype=np.float64))
    lat, dlon = np.broadcast_arrays(lat, np.abs(np.asarray(dlon_deg, dtype=np.float64)))
    beta = np.arctan((1 - f) * np.tan(np.radians(lat)))
    half = 0.5 * np.radians(dlon)
    sb = np.sin(beta)

    def half_dlon_and_dist(a0):
        ca, sa = np.cos(a0), np.sin(a0)
        k2 = ep2 * ca * ca
        sig1 = np.arcsin(np.clip(sb / ca, -1.0, 1.0))
        omega1 = np.arctan2(sa * np.sin(sig1), np.cos(sig1))
        J = _quad(lambda s: (2 - f) / (1 + (1 - f) * np.sqrt(1 + k2[..., None] * np.sin(s) ** 2)),
                  sig1, np.full_like(sig1, 0.5 * np.pi))
        I1 = _quad(lambda s: np.sqrt(1 + k2[..., None] * np.sin(s) ** 2), sig1, np.full_like(sig1, 0.5 * np.pi))
        return (0.5 * np.pi - omega1) - f * sa * J, 2.0 * b * I1

    lo = np.zeros_like(beta)
    hi = 0.5 * np.pi - beta                      # the point itself is the vertex: dlon = 0
    for _ in range(100):
        mid = 0.5 * (lo + hi)
        h, _ = half_dlon_and_dist(mid)
        big = h > half                           # half-longitude decreases with alpha0
        lo = np.where(big, mid, lo)
        hi = np.where(big, hi, mid)
    _, dist = half_dlon_and_dist(0.5 * (lo + hi))
    # on the equator the geodesic stays on the equator up to dlon = (1 - f) 180 degrees
    equatorial = (beta == 0) & (half <= (1 - f) * 0.5 * np.pi)
    dist = np.where(equatorial, WGS84_A * 2.0 * half, dist)
    return np.where(dlon == 0, 0.0, dist)


def wgs84_half_turn_distance(lat_deg):
    """``geod.inv(0, lat, 180, lat)``: the geodesic to the point 180 degrees away runs over the pole."""
    return 2.0 * (wgs84_meridian_arc(90.0) - wgs84_meridian_arc(lat_deg))


def lonlat_to_meter(lon_deg, lat_deg):
    """functions.py:958-973 / :1011-1022: (lat, lon) in degrees -> signed 'meter' coordinates."""
    lon = np.asarray(lon_deg, dtype=np.float64)
    lat = np.asarray(lat_deg, dtype=np.float64)
    lat_m = wgs84_meridian_arc(lat) * np.sign(lat)
    lon_m = wgs84_same_lat_distance(lat, lon) * np.sign(lon)
    return lat_m, lon_m


def gaussian_kernel_interp(src_xy, src_val, dst_xy, radius, sharpness, null_value=np.nan, chunk=2048):
    """vtkPointInterpolator + vtkGaussianKernel (radius footprint, NULL_VALUE strategy), see above."""
    src_xy, dst_xy = np.asarray(src_xy, dtype=np.float64), np.asarray(dst_xy, dtype=np.float64)
    src_val = np.asarray(src_val, dtype=np.float64)
    f2 = (sharpness / radius) ** 2
    out = np.full(len(dst_xy), null_value, dtype=np.float64)
    eps = np.finfo(np.float64).eps * 256.0
    for i0 in range(0, len(dst_xy), chunk):
        d = dst_xy[i0:i0 + chunk]
        d2 = (d[:, None, 0] - src_xy[None, :, 0]) ** 2 + (d[:, None, 1] - src_xy[None, :, 1]) ** 2
        inside = d2 <= radius * radius
        w = np.where(inside, np.exp(-f2 * d2), 0.0)
        sw = w.sum(axis=1)
        val = (w * src_val[None, :]).sum(axis=1)
        res = np.where(sw > 0, val / np.where(sw > 0, sw, 1.0), null_value)
        hit = inside & (d2 < eps)
        anyhit = hit.any(axis=1)
        res[anyhit] = src_val[hit.argmax(axis=1)[anyhit]]
        res[~inside.any(axis=1)] = null_value
        out[i0:i0 + chunk] = res
    return out


def nan_ignoring_interp(land_fr, era5_lat, era5_lon, delta, gcm_lat2d, gcm_lon2d, kernel_radius, sharpness):
    """functions.py:900-1060 for one 2-D field ``delta`` on a curvilinear grid (2-D lat/lon arrays).
    Returns [len(era5_lat), len(era5_lon)] float64."""
    gcm_lat_raw = np.asarray(gcm_lat2d, dtype=np.float64).reshape(-1).copy()
    gcm_lon_raw = np.asarray(gcm_lon2d, dtype=np.float64).reshape(-1).copy()
    gcm_val_raw = np.asarray(delta, dtype=np.float64).reshape(-1)
    gcm_lon_raw[gcm_lon_raw > 180] -= 360                    # :946-948
    ok = ~np.isnan(gcm_val_raw)                              # :951-954
    gcm_val, gcm_lon, gcm_lat = gcm_val_raw[ok], gcm_lon_raw[ok], gcm_lat_raw[ok]
    lat_m, lon_m = lonlat_to_meter(gcm_lon, gcm_lat)         # :958-973
    off = wgs84_half_turn_distance(gcm_lat)
    n = len(gcm_val)
    val_bd = np.tile(gcm_val, 3)                             # :978-988
    lat_bd = np.tile(lat_m, 3)
    lon_bd = np.tile(lon_m, 3)
    lon_bd[:n] -= off * 2
    lon_bd[2 * n:] += off * 2
    era5_lat = np.asarray(era5_lat, dtype=np.float64)
    era5_lon = np.asarray(era5_lon, dtype=np.float64).copy()
    era5_lon[era5_lon > 180] -= 360                          # :1006-1008
    lat_f = np.repeat(era5_lat, len(era5_lon))               # :1011-1012
    lon_f = np.tile(era5_lon, len(era5_lat))
    e_lat_m, e_lon_m = lonlat_to_meter(lon_f, lat_f)
    res = gaussian_kernel_interp(np.stack([lat_bd, lon_bd], axis=1), val_bd,
                                 np.stack([e_lat_m, e_lon_m], axis=1), kernel_radius, sharpness)
    res[np.asarray(land_fr, dtype=np.float64).reshape(-1) > 0.7] = np.nan      # :1031, :1055
    return res.reshape(len(era5_lat), len(era5_lon))


# ---------------------------------------------------------------------------
# the per-timestep routine (step_03_apply_to_era.py:44-381)
# ---------------------------------------------------------------------------
def pgw_for_era5(era, deltas, era_step_dt, *, p_ref_inp=30000, adj_factor=0.95,
                 thresh_phi_ref_max_error=0.15, max_n_iter=20,
                 ignore_top_pressure_error=False, n_iter_fixed=None, i_reinterp=0,
                 emulate_file_dtypes=False):
    """
    step_03_apply_to_era.py:44-381.  ``i_reinterp`` (settings.py:150) re-interpolates the ERA
    state and the deltas onto the updated model levels every iteration (:202-216, :330-343);
    ``p_ref_inp=None`` picks the reference pressure per column and iteration from the zg
    pressure levels (:219-251, determine_p_ref).

    era:    dict of float arrays: ak,bk [L+1]; optionally akm,bkm [L];
            PS [1,ny,nx]; FIS [1,ny,nx]; T,QV,U,V [1,L,ny,nx]; FR_LAND,
            FR_SEA_ICE, T_SKIN [1,ny,nx]; T_SO [1,S,ny,nx]; soil1 [S].
    deltas: dict var -> {'time','data','plev'} for ta,hur,ua,va,zg (3-D),
            tas,hurs,ts,tos,siconc (2-D) and 'ps_hist' (HIST ps, 2-D).
    Returns dict with PS,T,QV,U,V,T_SKIN,T_SO,FR_SEA_ICE (float64), 'n_iter',
    'phi_max_errors' (one per iteration) and 'deltas' (interpolate_full taps).

    dtypes.  The reference never casts: what it computes in follows from the dtypes of the ERA5 file
    through numpy's promotion rules (found by executing it over oracle/xrlite.py, see
    oracle/make_golden_glue.py).  Always reproduced here: the virtual temperature of the ERA state is a
    product of the float32 T and QV (functions.py:144), the PGW state is float64.  Reproduced with
    ``emulate_file_dtypes=True``, for PS/FIS/T/QV passed in as float32 like in a real ERA5 file:
    ``delta_ps`` and hence ``ps_pgw`` are float32 (xarray's in-place ``+=`` keeps the dtype of
    zeros_like(PS), :186-195), the half-level geopotential is stored as float32 (functions.py:141)
    and RELHUM of the ERA state is evaluated in float32 (:91-94).  These add rounding noise of
    ~2e-2 m2/s2 to the geopotential error and ~3e-2 Pa to ps_pgw; a threshold below ~1e-2 m2/s2 can
    then not be met.  The default (False) models PS and FIS stored as double and RELHUM in float64.

    n_iter_fixed (test hook, not in the reference): run exactly that many iterations
    regardless of the threshold and also return 'ps_traj' (ps after each iteration's
    update); used to check the latitude-band scheme in which the stopping rule is
    evaluated on the MAX over all bands.
    """
    f64 = lambda a: np.asarray(a, dtype=np.float64)
    asis = (lambda a: np.asarray(a)) if emulate_file_dtypes else f64
    ak, bk = f64(era["ak"]), f64(era["bk"])
    PS = asis(era["PS"])
    FIS = asis(era["FIS"])
    T, QV = np.asarray(era["T"]), np.asarray(era["QV"])      # dtype of the file (see above)
    U, V = f64(era["U"]), f64(era["V"])
    lev = lambda c: c[None, :, None, None]
    pa_hl_era = lev(ak) + PS[:, None] * lev(bk)              # :64-66
    if "akm" in era:                                         # :68-85
        akm, bkm = f64(era["akm"]), f64(era["bkm"])
    else:
        akm = 0.5 * np.diff(ak) + ak[:-1]
        bkm = 0.5 * np.diff(bk) + bk[:-1]
    pa_era = lev(akm) + PS[:, None] * lev(bkm)               # :87-88
    with np.errstate(all="ignore"):
        RELHUM = specific_to_relative_humidity(asis(QV), pa_era, asis(T))    # :91-94

    # ---- surface and soil (:103-146); ERA5 fields are float32 in the file and
    # updated in place there; the oracle keeps float64.
    sic = f64(era["FR_SEA_ICE"]) + load_delta(deltas["siconc"], era_step_dt) / 100
    sic = np.clip(sic, 0, 1)
    delta_ts = load_delta(deltas["ts"], era_step_dt)
    delta_tos = load_delta(deltas["tos"], era_step_dt)
    delta_ts_combined = integrate_tos(delta_tos, delta_ts,
                                      f64(era["FR_LAND"])[0], sic[0])
    T_SKIN = f64(era["T_SKIN"]) + delta_ts_combined
    delta_st_clim = load_delta(deltas["ts"], None).mean(axis=0)       # :134-136
    soil1 = f64(era["soil1"])
    delta_soilt = (delta_st_clim[None, None] + np.exp(-soil1 / 2.8)[None, :, None, None] *
                   (delta_ts_combined[:, None] - delta_st_clim[None, None]))  # :139-143
    T_SO = f64(era["T_SO"]) + delta_soilt

    # ---- 3-D deltas on ERA model levels (:158-173)
    out_deltas = {"ts": delta_ts_combined, "st": delta_soilt}
    vars_era = {"ta": T, "hur": RELHUM, "ua": U, "va": V}
    vars_pgw = {}
    def delta_on(var, target_P):                              # load_delta_interp, functions.py:306-340
        d = load_delta(deltas[var], era_step_dt)
        if var in ("ta", "hur"):                             # functions.py:325-332
            d_sfc = load_delta(deltas[var + "s"], era_step_dt)
            ps_hist = load_delta(deltas["ps_hist"], era_step_dt)
        else:
            d_sfc = ps_hist = None
        return vert_interp_delta(d, deltas[var]["plev"], target_P, d_sfc, ps_hist,
                                 ignore_top_pressure_error)

    if not i_reinterp:                                       # :155-173
        for var in ["ta", "hur", "ua", "va"]:
            dv = delta_on(var, pa_era)
            out_deltas[var] = dv
            vars_pgw[var] = vars_era[var] + dv

    # ---- iterative surface-pressure adjustment (:182-319)
    delta_ps = np.zeros_like(PS)                             # dtype of PS (:186)
    adj_ps = np.zeros_like(PS)
    phi_ref_max_error = np.inf
    errs = []
    it = 1
    plev_zg = f64(deltas["zg"]["plev"])
    p_ref_field = None
    ps_traj, hus_traj = [], []
    while (phi_ref_max_error > thresh_phi_ref_max_error if n_iter_fixed is None
           else it <= n_iter_fixed):
        delta_ps = (delta_ps + adj_ps).astype(delta_ps.dtype)   # in place in the reference (:194)
        ps_pgw = PS + delta_ps
        pa_pgw = lev(akm) + ps_pgw[:, None] * lev(bkm)
        pa_hl_pgw = lev(ak) + ps_pgw[:, None] * lev(bk)
        if i_reinterp:                                       # :202-216
            for var in ["ta", "hur"]:
                v_era = interp_logp_4d(vars_era[var], pa_era, pa_pgw, extrapolate="constant")
                out_deltas[var] = delta_on(var, pa_pgw)
                vars_pgw[var] = v_era + out_deltas[var]
        if p_ref_inp is None:                                # :219-251
            p_min_era = pa_hl_era[:, -1] * 0.95
            p_min_pgw = pa_hl_pgw[:, -1] * 0.95
            p_new = np.full(PS.shape, np.nan)
            for idx in np.ndindex(PS.shape):
                r = determine_p_ref(p_min_era[idx], p_min_pgw[idx], plev_zg,
                                    None if p_ref_field is None else p_ref_field[idx])
                p_new[idx] = np.nan if r is None else r
            p_ref_field = p_new
            if np.any(np.isnan(p_ref_field)):
                raise ValueError("No reference pressure level above the required local minimum "
                                 "pressure level could not be found everywhere.")
            p_ref = p_ref_field
        else:
            p_ref = p_ref_inp
        vars_pgw["hus"] = relative_to_specific_humidity(
            vars_pgw["hur"], pa_pgw, vars_pgw["ta"])
        phi_ref_pgw = integ_geopot(pa_hl_pgw, FIS, vars_pgw["ta"],
                                   vars_pgw["hus"], p_ref, FIS.dtype)
        phi_ref_era = integ_geopot(pa_hl_era, FIS, T, QV, p_ref, FIS.dtype)
        delta_phi_ref = phi_ref_pgw - phi_ref_era
        dzg = load_delta(deltas["zg"], era_step_dt) * CON_G  # :292-295
        if p_ref_inp is None:                                # .sel(plev=p_ref), pointwise
            lev_idx = np.argmax(plev_zg[None, :, None, None] == p_ref[:, None], axis=1)
            climate_delta_phi_ref = np.take_along_axis(dzg, lev_idx[:, None], axis=1)[:, 0]
        else:
            sel = np.nonzero(plev_zg == p_ref)[0]
            if len(sel) != 1:
                raise KeyError("p_ref not found among zg pressure levels")
            climate_delta_phi_ref = dzg[:, sel[0]]
        phi_ref_error = delta_phi_ref - climate_delta_phi_ref
        adj_ps = - adj_factor * ps_pgw / (CON_RD * vars_pgw["ta"][:, -1]) * phi_ref_error
        with np.errstate(invalid="ignore"):
            phi_ref_max_error = (np.nanmax(np.abs(phi_ref_error))
                                 if not np.all(np.isnan(phi_ref_error)) else np.nan)
        errs.append(float(phi_ref_max_error))
        if n_iter_fixed is not None:
            ps_traj.append(ps_pgw.copy())
            hus_traj.append(vars_pgw["hus"].copy())
        it += 1
        if n_iter_fixed is None and it > max_n_iter:
            raise ValueError("ERROR! Pressure adjustment did not converge")
    out_deltas["ps"] = ps_pgw - PS
    if i_reinterp:                                           # :330-343
        for var in ["ua", "va"]:
            v_era = interp_logp_4d(vars_era[var], pa_era, pa_pgw, extrapolate="constant")
            out_deltas[var] = delta_on(var, pa_pgw)
            vars_pgw[var] = v_era + out_deltas[var]
    return dict(PS=ps_pgw, T=vars_pgw["ta"], QV=vars_pgw["hus"], U=vars_pgw["ua"],
                V=vars_pgw["va"], T_SKIN=T_SKIN, T_SO=T_SO, FR_SEA_ICE=sic,
                n_iter=it - 1, phi_max_errors=errs, deltas=out_deltas,
                RELHUM_era=RELHUM, ps_traj=ps_traj, hus_traj=hus_traj,
                p_ref=p_ref if p_ref_inp is None else None)

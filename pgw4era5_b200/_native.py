"""
ctypes binding of libpgw_b200.so (include/pgw_b200.h).

There is no CPU fallback: if the shared library is missing or cannot be loaded
the import of this module raises, and every operator in this package with it.
``python -m pgw4era5_b200.build`` (or ``__graft_entry__.build()``) compiles it
with nvcc for sm_100a.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# PGW_B200_LIB selects another build of the same library (kernel A/B runs)
LIB_PATH = os.environ.get("PGW_B200_LIB") or os.path.join(_HERE, "libpgw_b200.so")

PGW_MAX_SOIL = 16
PGW_MAX_ITER = 64

PGW_OK, PGW_E_INVALID, PGW_E_LAUNCH, PGW_E_SMEM = 0, -1, -2, -3

ERR_SRC_NOT_ASCENDING = 1 << 0
ERR_TARG_NOT_ASCENDING = 1 << 1
ERR_EXTRAP_OFF = 1 << 2
ERR_PS_HIST_RANGE = 1 << 4
ERR_PREF_BELOW_SFC = 1 << 5
ERR_NO_PREF = 1 << 6
ERR_PS_BOUND = 1 << 7
ERR_BAND_TIMEOUT = 1 << 8
ERR_PREF_FLOOR = 1 << 9
BAND_SLOT = 64 + 2 + 32 + 4 + 4
BAND_PARITIES = 8
FLAG_DIRECT = 1
FLAG_REF_DTYPES = 2
FLAG_LOCAL_PREF = 4
FLAG_REINTERP = 8
RUN_NO_FINALIZE = 1
BAND_WORDS = 64 + 2 + 32 + 4
INT32_MAX = 2 ** 31 - 1
REGRID_PACK_MAX_NX_S = 1536     # PGW_REGRID_PACK_MAX_NX_S: wider GCM grids need the scratch of pgw_regrid_pack_d4_f32

EXTRAP_MODES = {"off": 0, "linear": 1, "constant": 2, "nan": 3}

c_fp = C.c_void_p   # device pointers travel as plain addresses


class TSlab(C.Structure):
    _fields_ = [("lo", c_fp), ("hi", c_fp), ("x_hi", C.c_double), ("x_new", C.c_double)]


class TimestepArgs(C.Structure):
    _fields_ = (
        [("ncol", C.c_longlong), ("nlev", C.c_int), ("nplev", C.c_int), ("nsoil", C.c_int),
         ("plev_descending", C.c_int), ("flags", C.c_int), ("reserved0", C.c_int)]
        + [(n, c_fp) for n in ("ak", "bk", "akm", "bkm", "plev", "ak_host", "bk_host", "akm_host", "bkm_host")]
        + [(n, c_fp) for n in ("PS", "FIS", "FR_LAND", "FR_SEA_ICE", "T_SKIN", "T_SO", "T", "QV", "U", "V")]
        + [(n, TSlab) for n in ("d4", "tas", "hurs", "ps_hist", "ts", "tos", "siconc", "zg_ref")]
        + [("ts_clim", c_fp), ("soil_decay", C.c_double * PGW_MAX_SOIL),
           ("p_ref", C.c_double), ("adj_factor", C.c_double),
           ("thresh_phi_ref_max_error", C.c_double), ("k_spec", C.c_int), ("ps_bound", C.c_double)]
        + [(n, c_fp) for n in ("PS_out", "T_SKIN_out", "FR_SEA_ICE_out", "T_SO_out", "T_out", "QV_out",
                               "U_out", "V_out", "dps_out", "dps_traj", "maxerr", "stats", "err", "first_k", "poly_fallback")]
        + [("zg", TSlab), ("zg_plev", c_fp), ("zg_plev_host", c_fp), ("nzg", C.c_int), ("reserved1", C.c_int),
           ("p_floor", C.c_double), ("pref_traj", c_fp), ("p_ref_out", c_fp)]
    )


class TimestepResult(C.Structure):
    _fields_ = [("n_iter", C.c_int), ("converged", C.c_int), ("rewritten", C.c_int), ("reserved", C.c_int)]


class TimestepStatus(C.Structure):
    """pgw_timestep_status: the device block the kernels report into and its pinned host copy."""
    _fields_ = [("maxerr", C.c_uint64 * PGW_MAX_ITER), ("result", TimestepResult), ("stats", C.c_float * 2),
                ("err", C.c_uint32), ("first_k", C.c_int32 * 4), ("poly_fallback", C.c_uint32)]


ABI_VERSION = 10        # PGW_B200_ABI_VERSION of include/pgw_b200.h


class NativeError(RuntimeError):
    pass


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "libpgw_b200.so not found at %s: build it with `python -m pgw4era5_b200.build` "
            "(nvcc, sm_100a).  This package has no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    ll, i, d, vp = C.c_longlong, C.c_int, C.c_double, C.c_void_p
    sig = {
        "pgw_version": (C.c_char_p, []),
        "pgw_abi_version": (i, []),
        "pgw_last_error": (C.c_char_p, []),
        "pgw_sizeof_timestep_args": (ll, []),
        "pgw_interp_logp_f64": (i, [vp, vp, vp, vp, i, i, i, ll, i, i, i, vp, vp]),
        "pgw_interp_logp_f32": (i, [vp, vp, vp, vp, i, i, i, ll, i, i, i, vp, vp]),
        "pgw_specific_to_relative_humidity_f32": (i, [vp, vp, vp, vp, ll, vp]),
        "pgw_relative_to_specific_humidity_f32": (i, [vp, vp, vp, vp, ll, vp]),
        "pgw_specific_to_relative_humidity_f64": (i, [vp, vp, vp, vp, ll, vp]),
        "pgw_relative_to_specific_humidity_f64": (i, [vp, vp, vp, vp, ll, vp]),
        "pgw_humidity_op_f32": (i, [i, vp, vp, vp, ll, vp]),
        "pgw_humidity_op_f64": (i, [i, vp, vp, vp, ll, vp]),
        "pgw_replace_delta_sfc_f32": (i, [vp, vp, vp, vp, vp, vp, i, ll, i, vp, vp]),
        "pgw_replace_delta_sfc_f64": (i, [vp, vp, vp, vp, vp, vp, i, ll, i, vp, vp]),
        "pgw_integ_geopot_f32": (i, [vp, vp, vp, vp, vp, d, vp, i, ll, vp, vp]),
        "pgw_integ_geopot_f64": (i, [vp, vp, vp, vp, vp, d, vp, i, ll, vp, vp]),
        "pgw_integ_geopot_f64_f32": (i, [vp, vp, vp, vp, vp, d, vp, i, ll, vp, vp]),
        "pgw_integrate_tos_f32": (i, [vp, vp, vp, vp, vp, ll, vp]),
        "pgw_integrate_tos_f64": (i, [vp, vp, vp, vp, vp, ll, vp]),
        "pgw_time_interp_f32": (i, [vp, vp, d, d, vp, ll, vp]),
        "pgw_byteswap32": (i, [vp, ll, vp]),
        "pgw_pack_d4_f32": (i, [vp, vp, vp, vp, vp, ll, i, vp]),
        "pgw_geod_to_meter_f64": (i, [vp, vp, vp, vp, vp, ll, vp]),
        "pgw_gauss_interp_f64": (i, [vp, vp, vp, ll, i, vp, vp, vp, vp, ll, d, d, vp]),
        "pgw_time_mean_f32": (i, [vp, i, vp, ll, vp]),
        "pgw_timestep_smem_bytes": (ll, [C.POINTER(TimestepArgs)]),
        "pgw_timestep_uses_tma": (i, [C.POINTER(TimestepArgs)]),
        "pgw_timestep_plan_info": (i, [C.POINTER(TimestepArgs), C.POINTER(C.c_int * 6)]),
        "pgw_column_tma_layout": (i, [i, i, i, C.POINTER(C.c_int), C.POINTER(C.c_longlong)]),
        "pgw_timestep": (i, [C.POINTER(TimestepArgs), vp]),
        "pgw_timestep_finalize": (i, [C.POINTER(TimestepArgs), vp, vp]),
        "pgw_sizeof_timestep_status": (ll, []),
        "pgw_timestep_run": (i, [C.POINTER(TimestepArgs), vp, vp, i, vp]),
        "pgw_timestep_finish": (i, [C.POINTER(TimestepArgs), vp, vp, vp]),
        "pgw_band_pack": (i, [vp, vp, vp]),
        "pgw_band_unpack": (i, [vp, vp, vp]),
        "pgw_band_exchange": (i, [vp, vp, i, i, C.c_ulonglong, d, vp]),
        "pgw_zonal_mean_f32": (i, [vp, vp, ll, i, i, vp]),
        "pgw_regrid_bilinear_f32": (i, [vp, vp, vp, ll, i, i, i, i, vp, vp, vp, vp, vp, vp, vp]),
        "pgw_regrid_bilinear_band_f32": (i, [vp, vp, vp, ll, i, i, i, i, i, i, vp, vp, vp, vp, vp, vp, vp]),
        "pgw_regrid_pack_d4_f32": (i, [vp, vp, vp, i, i, i, i, i, i, i, vp, vp, vp, vp, vp, vp, vp, vp]),
        "pgw_smooth_harmonic_f32": (i, [vp, vp, i, ll, vp]),
        "pgw_surface_update": (i, [C.POINTER(TimestepArgs), vp]),
        "pgw_hybrid_pressure_f64": (i, [vp, vp, vp, vp, i, ll, vp]),
        "pgw_axpy_f64": (i, [vp, vp, d, vp, ll, vp]),
        "pgw_determine_p_ref_f64": (i, [vp, vp, vp, i, vp, vp, ll, vp, vp]),
        "pgw_select_plev_f64": (i, [vp, vp, i, vp, vp, ll, vp]),
        "pgw_ps_adjust_f64": (i, [vp, vp, vp, vp, vp, d, vp, vp, ll, vp]),
    }
    for name, (res, args) in sig.items():
        try:
            fn = getattr(lib, name)
        except AttributeError:
            raise ImportError("%s does not export %s: stale build, run `python -m pgw4era5_b200.build`"
                              % (LIB_PATH, name))
        fn.restype, fn.argtypes = res, args
    if lib.pgw_abi_version() != ABI_VERSION:
        raise ImportError("libpgw_b200.so has ABI %d, this package expects %d (include/pgw_b200.h): rebuild"
                          % (lib.pgw_abi_version(), ABI_VERSION))
    if lib.pgw_sizeof_timestep_args() != C.sizeof(TimestepArgs):
        raise ImportError("pgw_timestep_args layout mismatch: C %d vs ctypes %d"
                          % (lib.pgw_sizeof_timestep_args(), C.sizeof(TimestepArgs)))
    if lib.pgw_sizeof_timestep_status() != C.sizeof(TimestepStatus):
        raise ImportError("pgw_timestep_status layout mismatch: C %d vs ctypes %d"
                          % (lib.pgw_sizeof_timestep_status(), C.sizeof(TimestepStatus)))
    return lib, sorted(sig)


lib, EXPORTED = _load()


def check(rc, what):
    """Raise for a negative host-side return code."""
    if rc == PGW_OK:
        return
    msg = lib.pgw_last_error().decode() if rc in (PGW_E_LAUNCH, PGW_E_SMEM) else ""
    name = {PGW_E_INVALID: "invalid argument", PGW_E_LAUNCH: "CUDA error", PGW_E_SMEM:
            "shared memory"}.get(rc, "error %d" % rc)
    raise NativeError("%s: %s %s" % (what, name, msg))


PLAN_KEYS = ("tma", "fast", "lst", "np", "tmem_cols", "l137")


def plan_info(args):
    """The column-kernel plan pgw_timestep() launches for ``args`` (pgw_timestep_plan_info), as a dict."""
    info = (C.c_int * 6)()
    check(lib.pgw_timestep_plan_info(C.byref(args), C.byref(info)), "pgw_timestep_plan_info")
    return dict(zip(PLAN_KEYS, info))

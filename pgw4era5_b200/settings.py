"""
Namelist of the PGW-for-ERA5 path.  Same names, meaning and default values as
the reference's ``settings.py:15-150`` so that a user's edited copy can be used
unchanged (``PGW_SETTINGS=/path/to/settings.py`` replaces this module's values
at import time, see ``_load_user_settings``).

Unlike the reference, the five surface-pressure-adjustment knobs are read at
*call* time by the engine and handed to the CUDA kernels as arguments, so
changing them needs no rebuild (SURVEY.md section 5, "Config").
"""
import os as _os
import runpy as _runpy

# verbosity of progress messages, 0..2
i_debug = 2

# file-name templates of the GCM inputs ({} = CMOR variable name)
file_name_bases = {
    'SCEN-HIST': '{}_delta.nc',
    'HIST': '{}_historical.nc',
}

# file-name template of the ERA5 files that are read and written
era5_file_name_base = 'cas{:%Y%m%d%H}0000.nc'

# dimension names: ERA5 files
TIME_ERA = 'time'
LON_ERA = 'lon'
LAT_ERA = 'lat'
LEV_ERA = 'level'
HLEV_ERA = 'level1'
SOIL_HLEV_ERA = 'soil1'

# dimension names: GCM atmosphere files
TIME_GCM = 'time'
LON_GCM = 'lon'
LAT_GCM = 'lat'
PLEV_GCM = 'plev'
LEV_GCM = 'lev'

# dimension names: GCM ocean files (tos)
TIME_GCM_OCEAN = 'time'
LON_GCM_OCEAN = 'longitude'
LAT_GCM_OCEAN = 'latitude'

# CMOR name -> variable name inside the ERA5 files (None: auxiliary delta only)
var_name_map = {
    'ta': 'T', 'ua': 'U', 'va': 'V', 'hur': 'RELHUM',
    'zg': 'PHI',
    'tas': None, 'hurs': None, 'tos': None,
    'ps': 'PS',
    'hus': 'QV', 'zgs': 'FIS', 'ts': 'T_SKIN', 'st': 'T_SO',
    'sftlf': 'FR_LAND', 'sic': 'FR_SEA_ICE',
}

# step_02 regridding
i_use_xesmf_regridding = 0
nan_interp_kernel_radius = 1000000  # m
nan_interp_sharpness = 4

# surface-pressure adjustment
p_ref_inp = 30000  # Pa; None = choose locally (PGWEngine.submit: fused kernel; apply: staged path)
adj_factor = 0.95
thresh_phi_ref_max_error = 0.15
max_n_iter = 20
i_reinterp = 0     # 1: re-interpolate the ERA state every iteration (PGWEngine.submit: fused kernel; apply: staged path)

# Not in the reference's settings.py.  The reference never casts, so what it computes in follows from the
# dtypes of the ERA5 file: with float32 PS and FIS (every real file) delta_ps / ps_pgw are float32 and the
# half-level geopotential is a float32 running sum (step_03_apply_to_era.py:186-195, functions.py:141),
# which adds ~1e-2 m2/s2 of rounding noise to the geopotential error and ~3e-2 Pa to ps_pgw.
#   0 (default): float64 accumulation = the reference on a file that stores PS and FIS as double;
#                thresholds below ~1e-2 m2/s2 converge (the reference's float32 path cannot reach them).
#   1: reproduce the float32 rounding steps of the reference exactly where it applies them.
i_reference_dtypes = 0

# Not in the reference's settings.py.  The reference replaces PS, T, QV, U, V by its float64 PGW state and
# to_netcdf writes them as float64 (step_03_apply_to_era.py:367-381) although the ERA5 file holds float32.
#   0 (default): written in the dtype of the input file (half the bytes; files stay NetCDF-3 raw-pipeline capable)
#   1: float64 like the reference, for users who diff outputs against a reference run
i_reference_output_dtypes = 0


def _load_user_settings():
    path = _os.environ.get('PGW_SETTINGS')
    if path:
        user = _runpy.run_path(path)
        globals().update({k: v for k, v in user.items() if not k.startswith('_')})


_load_user_settings()

"""
TEST INFRASTRUCTURE ONLY -- generates tests/golden/reference_functions.npz by
running the UNMODIFIED reference functions from the functions.py of a PGW4ERA5
checkout (its directory in $PGW4ERA5_REFERENCE).

The reference cannot be imported as-is in the build container (xarray, pyvista,
pyproj are absent), so empty stand-in modules are inserted into ``sys.modules``
for those three names only; every function exercised below is pure
numpy/numba and never touches them.  The reference is not part of this
repository, hence the outputs are committed as a small fixture.

    PGW4ERA5_REFERENCE=/path/to/PGW4ERA5 python oracle/make_golden.py
"""
import os
import sys
import types

import numpy as np

REF = os.environ.get("PGW4ERA5_REFERENCE", "")
OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tests", "golden",
                   "reference_functions.npz")


def import_reference_functions():
    for name, attrs in (("xarray", ()), ("pyvista", ("PolyData",)), ("pyproj", ("Geod",))):
        if name not in sys.modules:
            mod = types.ModuleType(name)
            for a in attrs:
                setattr(mod, a, object)
            sys.modules[name] = mod
    if not os.path.isfile(os.path.join(REF, "functions.py")):
        raise SystemExit("set PGW4ERA5_REFERENCE to the directory of a PGW4ERA5 checkout")
    sys.path.insert(0, REF)
    import functions  # noqa: the reference's functions.py
    return functions


def main(out_path=OUT):
    F = import_reference_functions()
    rng = np.random.default_rng(20240611)
    g = {}

    # --- interp_extrap_1d, all four modes (functions.py:511-580)
    src_x = np.log(np.array([1000., 5000., 1e4, 5e4, 1e5]))
    src_y = np.arange(1., 6.)
    targ_x = np.log(np.array([500., 1000., 3000., 7e4, 101000.]))
    g["ie1_src_x"], g["ie1_src_y"], g["ie1_targ_x"] = src_x, src_y, targ_x
    for mode in ("linear", "constant", "nan"):
        g["ie1_out_" + mode] = F.interp_extrap_1d(src_x, src_y, targ_x, mode)
    inner = np.log(np.array([1000., 2500., 5e4, 1e5]))
    g["ie1_targ_inner"] = inner
    g["ie1_out_off_inner"] = F.interp_extrap_1d(src_x, src_y, inner, "off")

    # --- interp_1d_for_timelatlon on random columns (functions.py:479-508)
    nt, ks, kt, ny, nx = 2, 7, 23, 5, 6
    sp = np.sort(rng.uniform(np.log(100.), np.log(1e5), (nt, ks, ny, nx)), axis=1)
    tp = np.sort(rng.uniform(np.log(1.), np.log(1.1e5), (nt, kt, ny, nx)), axis=1)
    tp[0, 3, 2, 2] = sp[0, 2, 2, 2]          # an exact node hit
    tp = np.sort(tp, axis=1)
    val = rng.normal(size=(nt, ks, ny, nx))
    val[1, 4, 1, 1] = np.nan                  # NaNs propagate through a bracket
    g["i4_src_p"], g["i4_targ_p"], g["i4_val"] = sp, tp, val
    for mode in ("linear", "constant", "nan"):
        out = np.zeros((nt, kt, ny, nx))
        F.interp_1d_for_timelatlon(val, sp, tp, out, nt, ny, nx, mode)
        g["i4_out_" + mode] = out

    # --- replace_delta_sfc (functions.py:343-366), the three branches
    plev = np.array([100., 500., 1000., 2000., 3000., 5000., 7000., 10000., 15000.,
                     20000., 25000., 30000., 40000., 50000., 60000., 70000., 85000.,
                     92500., 100000.])
    g["rds_plev"] = plev
    delta = np.arange(19.)
    cases = np.array([96000., 101500., 100000., 92500., 150., 50000.0001])
    g["rds_ps_hist"] = cases
    for i, ph in enumerate(cases):
        P, D = F.replace_delta_sfc(plev, ph, delta, 99.0)
        g["rds_P_%d" % i], g["rds_D_%d" % i] = P, D

    # --- determine_p_ref (functions.py:583-598)
    opts = plev[::-1].copy()
    g["dpr_opts"] = opts
    g["dpr_a"] = np.array(F.determine_p_ref(95000., 96000., opts, None))
    g["dpr_b"] = np.array(F.determine_p_ref(95000., 96000., opts, 85000.))
    g["dpr_c"] = np.array(F.determine_p_ref(60000., 71000., opts, None))

    # --- integrate_tos (functions.py:1145-1186)
    tos = rng.normal(size=(6, 7)); tos[rng.uniform(size=tos.shape) < 0.3] = np.nan
    ts = rng.normal(size=(6, 7))
    land = rng.uniform(size=(6, 7))
    ice = rng.uniform(size=(6, 7)); ice[rng.uniform(size=ice.shape) < 0.3] = np.nan
    g["it_tos"], g["it_ts"], g["it_land"], g["it_ice"] = tos, ts, land, ice
    g["it_out"] = F.integrate_tos(tos.copy(), ts.copy(), land.copy(), ice.copy())
    g["it_out_small"] = F.integrate_tos(np.array([[1., np.nan]]), np.array([[2., 3.]]),
                                        np.array([[.2, .5]]), np.array([[.1, 0.]]))

    # --- harmonic_ac_analysis (functions.py:678-740)
    t = np.arange(1, 366)
    series = (2.0 + 1.5 * np.cos(2 * np.pi * t / 365) - 0.7 * np.sin(2 * np.pi * 2 * t / 365)
              + 0.4 * np.cos(2 * np.pi * 3 * t / 365) + 0.9 * np.cos(2 * np.pi * 5 * t / 365)
              + 0.1 * rng.normal(size=365))
    g["hac_in"] = series
    g["hac_out"] = F.harmonic_ac_analysis(series.copy())
    s12 = rng.normal(size=12)
    g["hac_in12"], g["hac_out12"] = s12, F.harmonic_ac_analysis(s12.copy())
    snan = series.copy(); snan[17] = np.nan
    g["hac_out_nan"] = F.harmonic_ac_analysis(snan)

    # --- humidity helpers that need no xarray (functions.py:58-89)
    hus = rng.uniform(1e-6, 0.02, 50)
    pa = rng.uniform(100., 1.05e5, 50)
    ta = rng.uniform(190., 315., 50)
    g["hum_hus"], g["hum_pa"], g["hum_ta"] = hus, pa, ta
    g["hum_e"] = F.specific_humidity_to_vapor_pressure(hus, pa)
    g["hum_q"] = F.vapor_pressure_to_specific_humidity(g["hum_e"], pa)
    g["hum_esw"] = F.saturation_vapor_pressure_water_or_ice(pa, ta, water=True)
    g["hum_esi"] = F.saturation_vapor_pressure_water_or_ice(pa, ta, water=False)

    np.savez_compressed(out_path, **g)
    print("wrote", os.path.abspath(out_path), len(g), "arrays")


if __name__ == "__main__":
    main()

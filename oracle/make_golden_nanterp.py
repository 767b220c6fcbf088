#!/usr/bin/env python
"""
Golden vectors for the ocean-variable regridding (nan_ignoring_interp, functions.py:900-1060) from the REAL
third-party arithmetic: pyproj's ``Geod(ellps="WGS84").inv`` and pyvista/VTK's ``PolyData.interpolate``.

Neither package exists in the build container or on the GPU box (no network), so
oracle/pgw_oracle.py::nan_ignoring_interp restates their published algorithms and says "parity unpinned".
Run this script on any machine that has numpy, pyproj and pyvista (xarray is NOT needed: the reference function
only touches ``.coords[...] .values`` of its two arguments, which the tiny stand-in below provides) with the
reference checkout next to it:

    python oracle/make_golden_nanterp.py /path/to/PGW4ERA5  ->  tests/golden/reference_nanterp.npz

and commit the file.  tests/test_nanterp.py::test_oracle_matches_pyproj_vtk_fixture and the GPU twin then pin the
oracle and the CUDA operator (pgw_geod_to_meter_f64 / pgw_gauss_interp_f64) to it; until then they are skipped.
The fixture also stores the raw geodesic distances, so the coordinate mapping is pinned separately from the kernel.
"""
import os
import sys
import types

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = os.path.join(ROOT, "tests", "golden", "reference_nanterp.npz")


class _Coord:
    def __init__(self, values):
        self.values = np.asarray(values, dtype=np.float64)
        self.shape = self.values.shape


class _DA:
    """What nan_ignoring_interp uses of an xarray.DataArray: ``.values`` and ``.coords[name].values/.shape``."""

    def __init__(self, values, coords):
        self.values = np.asarray(values, dtype=np.float64)
        self.coords = {k: _Coord(v) for k, v in coords.items()}


def case(seed=12, nj=34, ni=72, ny=37, nx=72):
    rng = np.random.default_rng(seed)
    glat, glon = np.meshgrid(np.linspace(-78.0, 89.5, nj), 2.5 + 5.0 * np.arange(ni), indexing="ij")
    glat = glat + 0.4 * np.sin(np.radians(glon) * 2)             # curvilinear: 2-D latitudes
    tos = 2.0 + np.cos(np.radians(glat)) + 0.2 * rng.normal(size=(nj, ni))
    tos[rng.uniform(size=(nj, ni)) < 0.3] = np.nan               # land
    lat_t, lon_t = np.linspace(-90.0, 90.0, ny), 5.0 * np.arange(nx)
    land_fr = (rng.uniform(size=(ny, nx)) < 0.3).astype(np.float64)
    return dict(gcm_lat2d=glat, gcm_lon2d=glon, tos=tos, era5_lat=lat_t, era5_lon=lon_t, land_fr=land_fr,
                kernel_radius=np.float64(1000000.0), sharpness=np.float64(4.0))


def main(ref_dir):
    try:
        import pyproj
        import pyvista
    except ImportError as e:
        raise SystemExit("this script needs the packages the reference uses for this path (pyproj, pyvista/vtk): %s" % e)
    if "xarray" not in sys.modules:
        try:
            import xarray  # noqa: F401
        except ImportError:
            sys.modules["xarray"] = types.ModuleType("xarray")   # only imported at the top of functions.py
    sys.path.insert(0, ref_dir)
    import functions as RF                                        # the UNMODIFIED reference
    from settings import LAT_ERA, LAT_GCM_OCEAN, LON_ERA, LON_GCM_OCEAN
    c = case()
    delta = _DA(c["tos"], {LAT_GCM_OCEAN: c["gcm_lat2d"].copy(), LON_GCM_OCEAN: c["gcm_lon2d"].copy()})
    land = _DA(c["land_fr"], {LAT_ERA: c["era5_lat"].copy(), LON_ERA: c["era5_lon"].copy()})
    out = RF.nan_ignoring_interp(land, delta, float(c["kernel_radius"]), float(c["sharpness"]))
    # the three geodesic distances of every source point, straight from pyproj (functions.py:964-969)
    geod = pyproj.Geod(ellps="WGS84")
    lon = c["gcm_lon2d"].reshape(-1).copy()
    lon[lon > 180] -= 360
    lat = c["gcm_lat2d"].reshape(-1)
    z = np.zeros(len(lat))
    _, _, lat_m = geod.inv(lon, z, lon, lat)
    _, _, lon_m = geod.inv(z, lat, lon, lat)
    _, _, half = geod.inv(z, lat, np.ones(len(lat)) * 180, lat)
    np.savez_compressed(OUT, result=np.asarray(out, dtype=np.float64), geod_lat_m=lat_m, geod_lon_m=lon_m,
                        geod_half_turn=half, pyproj_version=pyproj.__version__, pyvista_version=pyvista.__version__,
                        **c)
    print("wrote", OUT)


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else os.environ.get("PGW4ERA5_REFERENCE", "."))

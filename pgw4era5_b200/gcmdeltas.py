"""
Climate deltas still on the GCM grid: what ``step_02_preproc_deltas regridding`` reads rather than what it writes.
On the global 0.25 degree ERA5 grid the regridded daily plev19 climatology takes 153 GB, more than HBM; on a
192 x 384 GCM grid the same deltas take about 2 GB per variable and stay resident.  ``GcmGridDeltaSet`` keeps them
so and produces each ERA5-grid stamp on the device when a timestep first needs it, in the rings of
``deltastream`` (eviction and ``hold`` unchanged): a load is one regrid launch on the set's copy stream,

- ta, hur, ua, va: ``pgw_regrid_pack_d4_f32`` regrids the four variables of the stamp and packs them into the
  column kernel's node layout in one pass;
- zg: ``pgw_regrid_bilinear_band_f32`` straight into its slot.

The 2-D deltas are regridded once at construction: tas, hurs, ts and ps_hist bilinearly (``regrid_arrays``), tos
and siconc from the curvilinear ocean grid with the NaN-ignoring Gaussian kernel (``nan_ignoring_interp_arrays``).
Every value is bit-identical to step_02 regridding followed by a resident ``DeltaSet`` of its files.
"""
import ctypes as C

import numpy as np
import torch

from . import _native as N
from . import functions as F
from . import ncio, settings
from .deltastream import StreamedDeltaSet, _Ring, delta_file
from .engine import VARS_2D, VARS_3D, VARS_PACKED, read_axes

OCEAN_VARS = ("tos", "siconc")


class _Grid:
    """A GCM source grid regridded to the ERA5 grid: the tables of ``regrid_tables`` on the device."""

    def __init__(self, lat, lon, era_lat, era_lon, device):
        tb = F.regrid_tables(lat, lon, era_lat, era_lon)
        ti = lambda a: torch.as_tensor(np.ascontiguousarray(a), device=device, dtype=torch.int32)
        tf = lambda a: torch.as_tensor(np.ascontiguousarray(a), device=device, dtype=torch.float64)
        self.j0, self.j1, self.wy = ti(tb["j0"]), ti(tb["j1"]), tf(tb["wy"])
        self.i0, self.i1, self.wx = ti(tb["i0"]), ti(tb["i1"]), tf(tb["wx"])
        self.ny_s, self.nx_s = len(lat), len(lon)
        self.ny_t, self.nx_t = len(era_lat), len(era_lon)

    def tensors(self):
        return [self.j0, self.j1, self.wy, self.i0, self.i1, self.wx]

    def args(self):
        """ny_t, nx_t, jt_begin, jt_end and the six tables, as the regrid entries take them (every target row)."""
        p = [C.c_void_p(t.data_ptr()) for t in self.tensors()]
        return [self.ny_t, self.nx_t, 0, self.ny_t] + p


class _RegridRing(_Ring):
    """A ring whose stamps are regridded on the device from ``src`` ([nt, nvar, K, ny_s, nx_s], kept stamps only)
    with the pole means ``pm`` ([nt, nvar * K, 2])."""

    def __init__(self, owner, name, src, pm, grid, slots):
        nt, nvar, K = src.shape[:3]
        super().__init__(owner, name, np.arange(nt), K * owner.ncol, nvar, slots)
        self.src, self.pm, self.grid, self.K = src, pm, grid, K
        self.scratch = None
        if nvar == 4 and grid.nx_s > N.REGRID_PACK_MAX_NX_S:
            self.scratch = torch.empty(4 * ((self.n + 3) // 4 * 4), device=owner.device, dtype=torch.float32)

    def device_tensors(self):
        return self.bufs + ([self.scratch] if self.scratch is not None else [])

    def _fill(self, s, rec, cs, ev):
        self._wait_uses(s, cs)
        if ev:
            ev[1].record(cs)
        g, st = self.grid, C.c_void_p(cs.cuda_stream)
        src, dst, pm = (C.c_void_p(t.data_ptr()) for t in (self.src[rec], self.bufs[s], self.pm[rec]))
        if self.src.shape[1] == 4:
            scratch = C.c_void_p(self.scratch.data_ptr() if self.scratch is not None else 0)
            N.check(N.lib.pgw_regrid_pack_d4_f32(src, dst, pm, self.K, g.ny_s, g.nx_s, *g.args(), scratch, st),
                    "pgw_regrid_pack_d4_f32")
        else:
            N.check(N.lib.pgw_regrid_bilinear_band_f32(src, dst, pm, self.K, g.ny_s, g.nx_s, *g.args(), st),
                    "pgw_regrid_bilinear_band_f32")


class GcmGridDeltaSet(StreamedDeltaSet):
    """
    The interface of ``engine.DeltaSet`` for deltas on the GCM grid, regridded to the ERA5 grid on the device.

    ``deltas``: the dict form ``DeltaSet`` takes, on the GCM grid, with the source grid of each variable as
    ``lat`` and ``lon``: 1-D axes for ta, hur, ua, va, zg, tas, hurs, ts and ps_hist (ta, hur, ua, va on one grid),
    the 2-D coordinates of the curvilinear ocean grid for tos and siconc.  ``era_lat``, ``era_lon``: the ERA5 grid;
    ``land_fr`` [ny, nx]: its land fraction, which masks tos and siconc (step_02 takes it from its ``-e`` file).
    ``slots``: stamps per ring.  A grid that does not cover the ERA5 domain raises step_02's ValueError here.
    Like ``StreamedDeltaSet`` it cannot be broadcast to other ranks nor serve an engine in latitude-band mode.
    """

    def __init__(self, deltas, era_lat, era_lon, land_fr, device="cuda", slots=4,
                 kernel_radius=None, sharpness=None):
        if slots < 2:
            raise ValueError("a streamed delta set needs at least 2 slots per ring")
        kernel_radius = settings.nan_interp_kernel_radius if kernel_radius is None else kernel_radius
        sharpness = settings.nan_interp_sharpness if sharpness is None else sharpness
        self.device = torch.device(device)
        era_lat = np.asarray(era_lat, dtype=np.float64)
        era_lon = np.asarray(era_lon, dtype=np.float64)
        self.shape2d = (len(era_lat), len(era_lon))
        self.ncol = self.shape2d[0] * self.shape2d[1]
        self.vars, keeps = {}, {}
        for name in VARS_3D + VARS_2D:
            if name not in deltas:
                raise KeyError("climate delta %r missing" % name)
            stamps, keeps[name], plev = read_axes(name, deltas[name])
            self.vars[name] = dict(time=stamps, plev=plev, data=None)
            if np.shape(deltas[name]["data"])[0] != len(deltas[name]["time"]):
                raise ValueError("%s delta: data of shape %s for %d time stamps" % (
                    name, np.shape(deltas[name]["data"]), len(deltas[name]["time"])))
        ta = deltas["ta"]
        for name in VARS_PACKED:
            if len(np.shape(deltas[name]["data"])) != 4:
                raise ValueError("%s delta must be [time, plev, lat, lon]" % name)
            if not (np.array_equal(np.asarray(deltas[name]["lat"]), np.asarray(ta["lat"])) and
                    np.array_equal(np.asarray(deltas[name]["lon"]), np.asarray(ta["lon"]))):
                raise ValueError("ta, hur, ua, va deltas must share their grid")
        self._check_axes({name: np.shape(deltas[name]["data"]) for name in VARS_PACKED})
        grid4 = _Grid(ta["lat"], ta["lon"], era_lat, era_lon, self.device)
        zg = deltas["zg"]
        gridz = grid4 if (np.array_equal(np.asarray(zg["lat"]), np.asarray(ta["lat"])) and
                          np.array_equal(np.asarray(zg["lon"]), np.asarray(ta["lon"]))) else \
            _Grid(zg["lat"], zg["lon"], era_lat, era_lon, self.device)
        self.grids = [grid4] if gridz is grid4 else [grid4, gridz]
        # the GCM-grid stamps as float32 (the conversion regrid_arrays applies), 29 February dropped
        K = np.shape(ta["data"])[1]
        self.src4 = torch.empty((len(keeps["ta"]), 4, K, grid4.ny_s, grid4.nx_s), device=self.device,
                                dtype=torch.float32)
        for v, name in enumerate(VARS_PACKED):
            self.src4[:, v].copy_(self._kept(deltas[name]["data"], keeps[name]))
        self.srcz = self._kept(deltas["zg"]["data"], keeps["zg"])[:, None]
        self.pm4 = self._pole_means(self.src4)
        self.pmz = self._pole_means(self.srcz)
        # 2-D deltas: regridded as step_02 writes them (every stamp), then what DeltaSet does with those files
        land_fr = np.asarray(land_fr)
        flat = {}
        for name in VARS_2D:
            d = deltas[name]
            if name in OCEAN_VARS:
                out = F.nan_ignoring_interp_arrays(land_fr, era_lat, era_lon, np.asarray(d["data"]), d["lat"],
                                                   d["lon"], kernel_radius, sharpness)
            else:
                out = F.regrid_arrays(np.asarray(d["data"]), d["lat"], d["lon"], era_lat, era_lon)
            data = torch.as_tensor(np.asarray(out))
            if len(keeps[name]) != len(d["time"]):
                data = data[torch.as_tensor(keeps[name])]
            flat[name] = data
        self._upload_2d(flat)
        self.copy_stream = torch.cuda.Stream(device=self.device)
        # set to [] to collect every load: the host fill time (none here) and three CUDA events on the copy stream
        # (start; the slot's users done; slot filled)
        self.load_events = None
        self.rings = dict(d4=_RegridRing(self, "d4", self.src4, self.pm4, grid4, slots),
                          zg=_RegridRing(self, "zg", self.srcz, self.pmz, gridz, slots))
        self.ts_clim = None
        self.refresh_derived()          # also: the copy stream's loads find the sources and pole means complete

    def _kept(self, data, keep):
        t = F._dev(data, torch.float32)
        if len(keep) != t.shape[0]:
            t = t[torch.as_tensor(keep, device=t.device)]
        return t.contiguous()

    def _pole_means(self, src):
        """Zonal means of the first and last source row of every field of ``src`` [nt, nvar, K, ny_s, nx_s]:
        [nt, nvar * K, 2]."""
        nt, nvar, K, ny_s, nx_s = src.shape
        pm = torch.empty((nt, nvar * K, 2), device=self.device, dtype=torch.float32)
        N.check(N.lib.pgw_zonal_mean_f32(C.c_void_p(src.data_ptr()), C.c_void_p(pm.data_ptr()), nt * nvar * K, ny_s,
                                         nx_s, C.c_void_p(torch.cuda.current_stream().cuda_stream)),
                "pgw_zonal_mean_f32")
        return pm

    def device_bytes(self):
        """Device memory of the set: the GCM-grid sources and their pole means, the regrid tables, the 2-D arena
        and the ring slots (and the scratch of a source grid wider than the fused kernel takes)."""
        ts = [self.src4, self.srcz, self.pm4, self.pmz, self.arena] + \
            [t for g in self.grids for t in g.tensors()] + [t for r in self.rings.values() for t in r.device_tensors()]
        return sum(t.numel() * t.element_size() for t in ts)


def read_gcm_deltas(delta_input_dir):
    """The delta files of ``delta_input_dir`` on the GCM grid (the names step_03 reads, as step_02 smoothing writes
    them) in the dict form of ``GcmGridDeltaSet``."""
    deltas = {}
    for name in VARS_3D + VARS_2D:
        path, var_name = delta_file(delta_input_dir, name)
        ds = ncio.open_dataset(path)
        var = ds[var_name]
        lat, lon = (settings.LAT_GCM_OCEAN, settings.LON_GCM_OCEAN) if name in OCEAN_VARS else \
            (settings.LAT_GCM, settings.LON_GCM)
        plev = np.asarray(ds[settings.PLEV_GCM].data, dtype=np.float64) if settings.PLEV_GCM in var.dims else None
        deltas[name] = dict(time=ncio.decode_time(ds[settings.TIME_GCM]), plev=plev, data=var.data,
                            lat=np.asarray(ds[lat].data), lon=np.asarray(ds[lon].data))
    return deltas

#!/usr/bin/python
# -*- coding: utf-8 -*-
"""
PGW for ERA5, main routine: drop-in for the reference's ``step_03_apply_to_era.py``.

Same command line (``-i -o -f -l -H -d -p -t -D``), same ``settings.py`` names, same file
naming; the per-file work (step_03_apply_to_era.py:44-381 of the reference) runs as one fused
CUDA pass per ERA5 file on a B200 through ``PGWEngine``.  ``-p N`` starts N worker processes,
worker i bound to GPU i % device_count (the reference's pool of CPU workers, parallel.py).
``--latitude_bands`` (under torchrun, not in the reference) splits every file into latitude bands instead, one
rank per GPU, each rank reading, computing and writing its own rows (``pgw_for_era5_files(band=...)``):

    torchrun --standalone --nproc-per-node 8 -m pgw4era5_b200.step_03_apply_to_era \\
           -i era_in -o era_out -d deltas -f 2006080200 -l 2006080200 -H 3 -t --latitude_bands

    python -m pgw4era5_b200.step_03_apply_to_era -i era_in -o era_out -d deltas \\
           -f 2006080200 -l 2006080300 -H 3 -t
"""
import argparse
import os
from argparse import RawDescriptionHelpFormatter
from collections import namedtuple
from datetime import datetime, timedelta
from pathlib import Path

import numpy as np

from . import ncio, settings
from .parallel import IterMP

_ENGINES = {}


def load_delta_set(delta_input_dir, device="cuda", max_resident_bytes=None, rows=None):
    """Read every delta file the path needs (ta, hur, ua, va, zg, tas, hurs, ts, tos, siconc as
    SCEN-HIST, ps as HIST; step_03_apply_to_era.py:533-539) into one device-resident DeltaSet, or, when
    that set and the staging copy of one variable would take more than ``max_resident_bytes`` (default:
    half of the device's free memory), into a ``StreamedDeltaSet`` that reads the 3-D deltas of NetCDF-3
    files stamp by stamp.  Only the headers and coordinates of the 3-D files are read to decide.

    ``rows = (r0, r1)``: a resident DeltaSet of those latitude rows only (latitude-band mode); the 3-D deltas of
    NetCDF-3 files are read band by band with ``RawNC3.read_rows``, other files are decoded and sliced.  A band
    set is never streamed: one that exceeds the limit raises ValueError before anything is uploaded."""
    from . import deltastream
    from .engine import DeltaSet, VARS_2D, VARS_3D
    headers = deltastream.read_3d_headers(delta_input_dir)
    if rows is not None and headers is not None:
        ta = headers["ta"][0].vars[headers["ta"][1]]
        _check_band_fits(deltastream.resident_bytes(headers), ta.shape[-2], device, max_resident_bytes, rows)
    elif rows is None and deltastream.should_stream(headers, device, max_resident_bytes):
        return deltastream.open_streamed(delta_input_dir, headers, device=device)
    deltas, decoded_bytes = {}, []
    for name in VARS_3D + VARS_2D:
        if rows is not None and headers is not None and name in VARS_3D:
            raw, var_name, axes = headers[name]
            deltas[name] = dict(axes, data=_read_band(raw, var_name, rows))
            continue
        path, var_name = deltastream.delta_file(delta_input_dir, name)
        ds = ncio.open_dataset(path)
        var = ds[var_name]
        plev = None
        if settings.PLEV_GCM in var.dims:
            plev = np.asarray(ds[settings.PLEV_GCM].data, dtype=np.float64)
        decoded_bytes.append(4 * int(var.data.size))
        ny = var.data.shape[-2]
        data = var.data if rows is None else np.ascontiguousarray(var.data[..., rows[0]:rows[1], :])
        deltas[name] = dict(time=ncio.decode_time(ds[settings.TIME_GCM]), plev=plev, data=data)
    if rows is not None and headers is None:
        # decoded 3-D deltas: the whole set as DeltaSet would hold it (its arena, plus the staging copy of the
        # largest variable), sized from the decoded arrays; 29 February counted, so an upper bound
        _check_band_fits(sum(decoded_bytes) + max(decoded_bytes), ny, device, max_resident_bytes, rows)
    return DeltaSet(deltas, device=device)


def _read_band(raw, name, rows):
    """Rows [r0, r1) of a 4-D float32 variable of a NetCDF-3 file as a native-endian array, entry by entry of its
    first axis (record by record for a record variable)."""
    v = raw.vars[name]
    r0, r1 = rows
    out = np.empty(v.shape[:-2] + (r1 - r0, v.shape[-1]), dtype=v.dtype)
    with open(raw.path, "rb", buffering=0) as f:
        if v.is_record:
            for rec in range(raw.numrecs):
                raw.read_rows(f, name, out[rec], r0, r1, record=rec)
        else:
            raw.read_rows(f, name, out, r0, r1)
    return out.byteswap(inplace=True).view(v.dtype.newbyteorder("="))


def _check_band_fits(whole, ny, device, max_resident_bytes, rows):
    """ValueError when the band of a delta set that needs ``whole`` bytes of device memory for all ``ny`` rows
    (linear in the number of rows) needs more than ``max_resident_bytes`` (default: half of the device's free
    memory), naming the number of ranks whose bands would fit."""
    import torch
    from .parallel import split_rows
    if max_resident_bytes is None:
        max_resident_bytes = torch.cuda.mem_get_info(torch.device(device))[0] // 2
    need = whole * (rows[1] - rows[0]) // ny
    if need <= max_resident_bytes:
        return
    fit = next((w for w in range(1, ny + 1) if whole * max(b - a for a, b in split_rows(ny, w)) // ny
                <= max_resident_bytes), None)
    raise ValueError("the delta band of rows %d..%d needs %.2f GB on the device, more than the %.2f GB allowed; "
                     "a latitude-band set is always resident: %s" % (
                         rows[0], rows[1], need / 1e9, max_resident_bytes / 1e9,
                         "%d ranks or more would fit" % fit if fit else "no number of ranks fits"))


def load_gcm_grid_delta_set(delta_input_dir, era_file, device="cuda"):
    """``GcmGridDeltaSet`` of the delta files of ``delta_input_dir`` still on the GCM grid (what step_02
    regridding reads), regridded on the device to the grid of ``era_file`` (an ERA5 ``ncio.Dataset``).  Its
    ``FR_LAND`` masks tos and siconc as the ``-e`` file of step_02 regridding does: the two must agree."""
    from .gcmdeltas import GcmGridDeltaSet, read_gcm_deltas
    land_fr = np.asarray(era_file[settings.var_name_map['sftlf']].data)[0]
    return GcmGridDeltaSet(read_gcm_deltas(delta_input_dir), np.asarray(era_file[settings.LAT_ERA].data),
                           np.asarray(era_file[settings.LON_ERA].data), land_fr, device=device)


MSG_GCM_BANDS = "--gcm_grid_deltas does not run with --latitude_bands"
MSG_GCM_INTERP_TIME = ("--gcm_grid_deltas does not run -D interpolate_time, which writes the time-interpolated "
                       "deltas on the grid of the delta files: regrid them with step_02 first")


def get_engine(delta_input_dir, era_file, band=None, gcm_grid_deltas=False):
    """One engine (and one resident copy of the climatology) per process and delta directory; with ``band``
    (latitude-band mode, ``Band``) one per row range, holding the deltas of those rows only.  With
    ``gcm_grid_deltas`` the delta files are on the GCM grid and regridded on the device to ``era_file``'s grid
    (``load_gcm_grid_delta_set``)."""
    import torch
    from .engine import PGWEngine
    if gcm_grid_deltas and band is not None:
        raise ValueError(MSG_GCM_BANDS)
    ak = np.asarray(era_file['ak'].data)
    bk = np.asarray(era_file['bk'].data)
    key = (os.path.abspath(delta_input_dir), torch.cuda.current_device(), ak.tobytes(), bk.tobytes())
    if band is not None:
        key += (tuple(band.rows), band.exchange)
    if gcm_grid_deltas:             # the deltas are regridded to this grid
        key += ("gcm_grid", np.asarray(era_file[settings.LAT_ERA].data).tobytes(),
                np.asarray(era_file[settings.LON_ERA].data).tobytes())
    eng = _ENGINES.get(key)
    if eng is None:
        device = torch.device("cuda", torch.cuda.current_device())
        if gcm_grid_deltas:
            ds = load_gcm_grid_delta_set(delta_input_dir, era_file, device)
        elif band is None:
            ds = load_delta_set(delta_input_dir, device=device)
        else:
            # a band that does not fit, or a delta file one rank cannot read, must stop every rank before the
            # engine's first collective
            ds, err = None, None
            try:
                ds = load_delta_set(delta_input_dir, device=device, rows=band.rows)
            except Exception as e:
                err = e
            _agree_or_raise(band, err, 0, "loading the delta climatology")
        akm = np.asarray(era_file['akm'].data) if 'akm' in era_file else None      # step_03:68-85
        bkm = np.asarray(era_file['bkm'].data) if 'bkm' in era_file else None
        soil = np.asarray(era_file[settings.SOIL_HLEV_ERA].data) if settings.SOIL_HLEV_ERA in era_file else ()
        eng = PGWEngine(ak, bk, ds, soil1=soil, akm=akm, bkm=bkm,
                        **({} if band is None else dict(group=band.group, band_exchange=band.exchange)))
        _ENGINES[key] = eng
    return eng


def pgw_for_era5(inp_era_file_path, out_era_file_path, delta_input_dir, era_step_dt,
                 ignore_top_pressure_error, debug_mode=None, gcm_grid_deltas=False):
    """Same signature as the reference's pgw_for_era5 (step_03_apply_to_era.py:44-47), plus ``gcm_grid_deltas``
    (``get_engine``)."""
    import torch
    vmap = settings.var_name_map
    if gcm_grid_deltas and debug_mode == 'interpolate_time':
        raise ValueError(MSG_GCM_INTERP_TIME)
    if settings.i_debug >= 0:
        print('Start working on input file {}'.format(inp_era_file_path))
    era_file = ncio.open_dataset(inp_era_file_path, decode_cf=False)
    eng = get_engine(delta_input_dir, era_file, gcm_grid_deltas=gcm_grid_deltas)
    names = dict(PS=vmap['ps'], FIS=vmap['zgs'], FR_LAND=vmap['sftlf'], FR_SEA_ICE=vmap['sic'],
                 T_SKIN=vmap['ts'], T_SO=vmap['st'], T=vmap['ta'], QV=vmap['hus'], U=vmap['ua'], V=vmap['va'])
    era = {k: torch.from_numpy(np.ascontiguousarray(era_file[v].data, dtype=np.float32))
           for k, v in names.items()}
    res = eng.apply(era, era_step_dt, ignore_top_pressure_error=ignore_top_pressure_error,
                    file_name=inp_era_file_path)
    host = {k: res[k].cpu().numpy() for k in ("PS", "T", "QV", "U", "V", "T_SKIN", "T_SO", "FR_SEA_ICE", "delta_ps")}

    if debug_mode == 'interpolate_full':                                       # step_03:350-361
        from . import functions as F
        ak, bk = eng.ak, eng.bk
        pa_era = (eng.akm[None, :, None, None] + era_file[vmap['ps']].data.astype(np.float64)[:, None]
                  * eng.bkm[None, :, None, None])
        rel_era = F.specific_to_relative_humidity(era_file[vmap['hus']].data.astype(np.float64), pa_era,
                                                  era_file[vmap['ta']].data.astype(np.float64))
        pa_pgw = eng.akm[None, :, None, None] + host["PS"].astype(np.float64)[:, None] * eng.bkm[None, :, None, None]
        rel_pgw = F.specific_to_relative_humidity(host["QV"].astype(np.float64), pa_pgw, host["T"].astype(np.float64))
        deltas = {'ps': host["delta_ps"], 'ta': host["T"] - era_file[vmap['ta']].data,
                  'hur': (rel_pgw - rel_era).astype(np.float32), 'ua': host["U"] - era_file[vmap['ua']].data,
                  'va': host["V"] - era_file[vmap['va']].data, 'st': host["T_SO"] - era_file[vmap['st']].data,
                  'ts': host["T_SKIN"] - era_file[vmap['ts']].data}
        for var_name, d in deltas.items():
            print(var_name)
            out_file_path = os.path.join(Path(out_era_file_path).parents[0],
                                         '{}_delta_{}'.format(vmap[var_name], Path(out_era_file_path).name))
            ref = era_file[vmap[var_name]]
            out = ncio.Dataset()
            for dname in ref.dims:
                if dname in era_file:
                    out[dname] = era_file[dname]
            out[vmap[var_name]] = ncio.Variable(ref.dims, d.reshape(ref.data.shape))
            out.to_netcdf(out_file_path, mode='w')
    else:                                                                      # step_03:367-381
        for key in ("PS", "T", "QV", "U", "V", "T_SKIN", "T_SO", "FR_SEA_ICE"):
            ref = era_file[names[key]]
            era_file[names[key]] = ncio.Variable(
                ref.dims, host[key].reshape(ref.data.shape).astype(_out_dtype(key, ref.data.dtype)), ref.attrs)
        if vmap['hur'] in era_file:
            del era_file[vmap['hur']]
        era_file.to_netcdf(out_era_file_path, mode='w')
        era_file.close()
        if settings.i_debug >= 1:
            print('Done. Saved to file {}.'.format(out_era_file_path))
    return res["n_iter"]


_ERA_NAMES = lambda vmap: dict(PS=vmap['ps'], FIS=vmap['zgs'], FR_LAND=vmap['sftlf'], FR_SEA_ICE=vmap['sic'],
                               T_SKIN=vmap['ts'], T_SO=vmap['st'], T=vmap['ta'], QV=vmap['hus'], U=vmap['ua'],
                               V=vmap['va'])


_WRITTEN = ("PS", "T", "QV", "U", "V", "T_SKIN", "T_SO", "FR_SEA_ICE")
# The reference replaces PS, T, QV, U, V by its float64 PGW state and to_netcdf keeps that dtype
# (step_03_apply_to_era.py:367-381); skin, soil and sea ice are updated in place and keep the file's dtype.
_F64_IN_REFERENCE = ("PS", "T", "QV", "U", "V")


def _out_dtype(key, file_dtype):
    """dtype a written field gets: the input file's (default, half the bytes of the reference's files), or
    with ``settings.i_reference_output_dtypes = 1`` float64 for the five fields the reference writes as float64."""
    if getattr(settings, "i_reference_output_dtypes", 0) and key in _F64_IN_REFERENCE:
        return np.float64
    return file_dtype
IO_STATS = {"raw": 0, "decoded": 0}          # files per I/O path of pgw_for_era5_files (tests, bench_files.py)


def _raw_layout(path, names, host_in, grid=None):
    """The header of ``path`` if the file can go through the pipeline without decoding: NetCDF-3, one
    record at most, every ERA5 field float32 with the size of its host buffer, no RELHUM to drop
    (step_03:371).  Else None (the decoding path is taken).  ``grid = (ny, nx)``: the host buffers hold a
    band of rows of that grid (latitude-band mode), so the fields must have ``grid`` as their last two axes
    and the buffers as many rows of every level as the band has."""
    from .nc3raw import NC_FLOAT, NotNetCDF3, RawNC3
    if os.environ.get("PGW_RAW_IO", "1") == "0" or getattr(settings, "i_reference_output_dtypes", 0):
        return None                 # float64 outputs change the layout of the file: decoding path
    try:
        raw = RawNC3(path)
    except (NotNetCDF3, OSError):
        return None
    if raw.numrecs > 1 or settings.var_name_map['hur'] in raw.vars:
        return None
    for key, name in names.items():
        v = raw.vars.get(name)
        if v is None or v.nc_type != NC_FLOAT or (v.is_record and raw.numrecs != 1):
            return None
        if grid is None:
            if v.nbytes != host_in[key].numel() * 4:
                return None
        elif tuple(v.record_shape[-2:]) != tuple(grid) or \
                v.nbytes // (grid[0] * grid[1]) * host_in[key].shape[-2] * grid[1] != host_in[key].numel() * 4 or \
                host_in[key].shape[-1] != grid[1]:
            return None
    return raw


def _copy_range(fd_in, fd_out, off, count):
    """Bytes [off, off+count) of fd_in to the same place in fd_out, in the kernel where possible."""
    while count > 0:
        try:
            n = os.copy_file_range(fd_in, fd_out, count, off, off)
        except (OSError, AttributeError):
            n = os.pwrite(fd_out, os.pread(fd_in, min(count, 1 << 24), off), off)
        if n <= 0:
            raise IOError("short copy")
        off += n
        count -= n


_WRITE_PIECE = 64 << 20


def _write_raw(raw, names, inp_path, out_path, host_out, pool=None):
    """The output file = the input file with the eight updated fields replaced (step_03:367-378): the
    bytes in between are copied file to file, the fields come straight from the (big-endian) host buffers.
    All writes are positional, so ``pool`` (a ThreadPoolExecutor) may run them side by side.  ``host_out = None``:
    the file gets the input's size and every byte outside the eight fields, whose rows the ranks of a
    latitude-band run then write (``RawNC3.write_rows``)."""
    segs = sorted((raw.offset(names[k]), raw.vars[names[k]].nbytes, k) for k in _WRITTEN)
    fd_in = os.open(inp_path, os.O_RDONLY)
    fd_out = os.open(out_path, os.O_WRONLY | os.O_CREAT | os.O_TRUNC, 0o644)

    def put(off, nbytes, key, lo=0, hi=None):
        mv = memoryview(host_out[key].numpy()).cast("B")
        done, end = lo, nbytes if hi is None else hi
        while done < end:
            done += os.pwrite(fd_out, mv[done:end], off + done)

    try:
        size = os.fstat(fd_in).st_size
        os.ftruncate(fd_out, size)
        jobs, pos = [], 0
        for off, nbytes, key in segs:
            jobs.append((_copy_range, (fd_in, fd_out, pos, off - pos)))
            if host_out is not None:
                # a 3-D field of a global file is 570 MB: cut into pieces so that all writer threads stay busy
                for lo in range(0, nbytes, _WRITE_PIECE):
                    jobs.append((put, (off, nbytes, key, lo, min(nbytes, lo + _WRITE_PIECE))))
            pos = off + nbytes
        jobs.append((_copy_range, (fd_in, fd_out, pos, size - pos)))
        if pool is None:
            for fn, args in jobs:
                fn(*args)
        else:
            for fut in [pool.submit(fn, *args) for fn, args in jobs]:
                fut.result()
    finally:
        os.close(fd_in)
        os.close(fd_out)


def _write_band(raw, names, out_path, host_out, rows, pool=None):
    """Rows [r0, r1) of the eight written fields from the (big-endian) band buffers ``host_out`` into the output
    file that rank 0 prepared (``_write_raw`` without buffers)."""
    fd = os.open(out_path, os.O_WRONLY)
    try:
        jobs = [(raw.write_rows, (fd, names[k], host_out[k].numpy(), rows[0], rows[1])) for k in _WRITTEN]
        if pool is None:
            for fn, args in jobs:
                fn(*args)
        else:
            for fut in [pool.submit(fn, *args) for fn, args in jobs]:
                fut.result()
    finally:
        os.close(fd)


class Band(namedtuple("Band", "group host_group rows exchange")):
    """This rank's share of a latitude-band run: ``group`` the (NCCL) process group the engine merges its status
    block over, ``host_group`` a gloo group of the same ranks for the host-side agreement (it waits on no CUDA
    stream), ``rows = (r0, r1)`` the latitude rows of this rank (None: ``split_rows(ny, world)[rank]`` of the
    files' grid), ``exchange`` the engine's ``band_exchange``."""
    __slots__ = ()

    def __new__(cls, group, host_group, rows=None, exchange="auto"):
        return super().__new__(cls, group, host_group, None if rows is None else tuple(rows), exchange)


def _agree_or_raise(band, err, fingerprint, what):
    """Every rank of ``band`` learns whether any rank failed (``err``) at this point, and whether all of them saw
    the same ``fingerprint``: one all-reduce (MAX) on the gloo group.  A failure raises on every rank -- its own
    exception on the rank that failed, RuntimeError on the others -- so that no rank is left waiting in a
    collective its peers never reach."""
    import torch
    import torch.distributed as dist
    world, rank = dist.get_world_size(band.host_group), dist.get_rank(band.host_group)
    v = torch.zeros(world + 2, dtype=torch.int64)
    v[rank] = int(err is not None)
    v[world], v[world + 1] = int(fingerprint), -int(fingerprint)
    dist.all_reduce(v, op=dist.ReduceOp.MAX, group=band.host_group)
    failed = [r for r in range(world) if int(v[r])]
    if err is not None:
        raise err
    if failed:
        raise RuntimeError("latitude bands: rank(s) %s failed while %s" % (failed, what))
    if int(v[world]) != -int(v[world + 1]):
        raise ValueError("latitude bands: the ranks disagree while %s (different files or headers)" % what)


def _fingerprint(*parts):
    """A 31-bit digest of ``parts`` (their repr) for ``_agree_or_raise``."""
    import zlib
    return zlib.crc32(repr(parts).encode()) & 0x7FFFFFFF


def _layout_key(raw, names):
    return tuple((names[k], raw.offset(names[k]), raw.vars[names[k]].shape) for k in sorted(names))


MSG_BAND_FILES = ("latitude bands read and write ERA5 files in place: they need NetCDF-3 files with one record, "
                  "float32 fields of one grid and no {} variable, and an output path other than the input")


def _band_refusal(debug_mode):
    """Why band mode cannot run the current settings (None if it can)."""
    from .engine import fused_refusal
    if debug_mode is not None:
        return "latitude bands do not run the debug modes (-D)"
    if getattr(settings, "i_reference_output_dtypes", 0):
        return "latitude bands write the input file's layout: i_reference_output_dtypes = 1 is not supported"
    if os.environ.get("PGW_RAW_IO", "1") == "0":
        return "latitude bands need the raw NetCDF-3 path (PGW_RAW_IO=0 is set)"
    return fused_refusal()


def _level_tables(path, names):
    """What the engine needs from the first ERA5 file -- ak, bk (akm, bkm and the soil depths where present) --
    as an ``ncio.Dataset`` read from the NetCDF-3 header and those small variables, and the grid (ny, nx) from
    the header of PS.  No field is read."""
    from .nc3raw import NotNetCDF3, RawNC3
    try:
        raw = RawNC3(path)
    except (NotNetCDF3, OSError) as e:
        raise ValueError("%s: %s (%s)" % (path, MSG_BAND_FILES.format(settings.var_name_map['hur']), e))
    if names["PS"] not in raw.vars or "ak" not in raw.vars or "bk" not in raw.vars:
        raise ValueError("%s: %s" % (path, MSG_BAND_FILES.format(settings.var_name_map['hur'])))
    out = ncio.Dataset()
    with open(path, "rb", buffering=0) as f:
        for name in ("ak", "bk", "akm", "bkm", settings.SOIL_HLEV_ERA):
            if name in raw.vars:
                v = raw.vars[name]
                out[name] = ncio.Variable(v.dims, raw.read_variable(f, name), v.attrs)
    ny, nx = raw.vars[names["PS"]].record_shape[-2:]
    return out, (int(ny), int(nx))


def _band_start(steps, names, band):
    """Latitude-band mode before any GPU work: the grid and this rank's rows from the first file, every input
    file checked on every rank, the output files created by rank 0 (the input's bytes outside the eight written
    fields), then the start barrier -- an agreement on the gloo group.  Every rank reads headers and level tables
    only, never a whole field.  Returns (level tables of the first file, (ny, nx), rows)."""
    import torch
    import torch.distributed as dist
    from .parallel import split_rows
    vmap = settings.var_name_map
    err, fp, first, grid, rows = None, 0, None, None, band.rows
    try:
        first, grid = _level_tables(steps[0]["inp_era_file_path"], names)
        nx = grid[1]
        if rows is None:
            rows = split_rows(grid[0], dist.get_world_size(band.group))[dist.get_rank(band.group)]
        nlev = len(first["ak"].data) - 1
        nsoil = len(first[settings.SOIL_HLEV_ERA].data) if settings.SOIL_HLEV_ERA in first else 0
        lev = dict(T_SO=nsoil, T=nlev, QV=nlev, U=nlev, V=nlev)
        shapes = {k: torch.empty((1, lev.get(k, 1), rows[1] - rows[0], nx), device="meta") for k in names}
        layouts = []
        for st in steps:
            inp, out = st["inp_era_file_path"], st["out_era_file_path"]
            raw = _raw_layout(inp, names, shapes, grid=grid)
            if raw is None or os.path.realpath(inp) == os.path.realpath(out):
                raise ValueError("%s: %s" % (inp, MSG_BAND_FILES.format(vmap['hur'])))
            layouts.append(_layout_key(raw, names))
            if dist.get_rank(band.host_group) == 0:
                _write_raw(raw, names, inp, out, None)
        fp = _fingerprint(grid, [(st["inp_era_file_path"], st["out_era_file_path"], str(st["era_step_dt"]))
                                 for st in steps], layouts)
    except Exception as e:
        err = e
    _agree_or_raise(band, err, fp, "checking the input files and creating the output files")
    return first, grid, tuple(rows)


def pgw_for_era5_files(steps, delta_input_dir, ignore_top_pressure_error, debug_mode=None, band=None,
                       gcm_grid_deltas=False):
    """
    The production mode of ``pgw_for_era5`` for a LIST of files on one GPU, as a three-stage
    pipeline (SURVEY.md 8f rank 1): a reader thread decodes file i+1 into pinned host buffers and
    a writer thread stores file i-1 while the GPU works on file i (``hostpipe.HostPipeline``:
    H2D, fused pass and D2H of consecutive files overlap on two CUDA streams).  NetCDF-3 files with
    float32 fields are not decoded at all: the reader moves the raw big-endian bytes of the fields into
    pinned memory (``nc3raw``), the GPU swaps the byte order next to the copies (``pgw_byteswap32``) and
    the writer assembles the output from the input file and the result buffers.  Results are
    identical to calling ``pgw_for_era5`` file by file.  ``steps``: dicts with inp_era_file_path,
    out_era_file_path, era_step_dt.  Returns the iteration counts.

    ``band`` (a ``Band``): latitude-band mode, every rank of ``band.group`` runs this with the same ``steps``.
    Rank 0 creates the output files first; each rank then reads its rows of every field (``RawNC3.read_rows``),
    runs them through an engine over its rows of the deltas whose status block is merged over the ranks, and
    writes its rows into the shared output files (``RawNC3.write_rows``).  The ranks agree on the gloo group
    before the start, before each file's submit and at the end, so a failure on one rank raises on all of them.
    Band mode runs whatever ``PGWEngine.submit`` runs (not the staged path, whose convergence test is per rank)
    on NetCDF-3 files; other settings and files raise ValueError before any GPU work.

    ``gcm_grid_deltas``: the delta files are on the GCM grid and are regridded on the device to the grid of the
    first file (``get_engine``); not with ``band`` nor with ``debug_mode = 'interpolate_time'`` (ValueError).
    """
    import queue
    import threading
    from concurrent.futures import ThreadPoolExecutor
    from .hostpipe import HostPipeline, IN_FIELDS
    if gcm_grid_deltas and band is not None:
        raise ValueError(MSG_GCM_BANDS)
    if gcm_grid_deltas and debug_mode == 'interpolate_time':
        raise ValueError(MSG_GCM_INTERP_TIME)
    if not steps:
        return []
    if band is not None:
        msg = _band_refusal(debug_mode)
        if msg is not None:
            raise ValueError(msg)
    elif debug_mode is not None or settings.i_reinterp or settings.p_ref_inp is None:
        return [pgw_for_era5(delta_input_dir=delta_input_dir,
                             ignore_top_pressure_error=ignore_top_pressure_error, debug_mode=debug_mode,
                             gcm_grid_deltas=gcm_grid_deltas, **st)
                for st in steps]
    vmap = settings.var_name_map
    names = _ERA_NAMES(vmap)
    if band is None:
        first = ncio.open_dataset(steps[0]["inp_era_file_path"], decode_cf=False)
        ny, nx = first[names["PS"]].data.shape[-2:]
        rows = (0, ny)
    else:
        first, (ny, nx), rows = _band_start(steps, names, band)
        band = band._replace(rows=rows)
    eng = get_engine(delta_input_dir, first, band, gcm_grid_deltas=gcm_grid_deltas)
    pipe = HostPipeline(eng, rows[1] - rows[0], nx)
    n_in_buf, n_out_buf = 3, 4
    free_in, free_out = queue.Queue(), queue.Queue()
    for _ in range(n_in_buf):
        free_in.put(pipe.alloc_host_inputs())
    for _ in range(n_out_buf):
        free_out.put(pipe.alloc_host_outputs())
    loaded, to_write = queue.Queue(maxsize=n_in_buf), queue.Queue()
    failure = []
    stop = threading.Event()         # set on any failure (or at the end): every blocking get/put below polls it

    def q_get(q):
        """q.get() that gives up (returns None) once the pipeline has been stopped."""
        while True:
            try:
                return q.get(timeout=0.2)
            except queue.Empty:
                if stop.is_set():
                    return None

    def q_put(q, item):
        while True:
            try:
                q.put(item, timeout=0.2)
                return True
            except queue.Full:
                if stop.is_set():
                    return False
    # the raw path is a copy between the page cache and pinned memory: a few threads per direction
    # (pread / pwrite release the GIL) move the fields of one file side by side
    n_io = max(1, min(8, (os.cpu_count() or 2) // 2))
    rpool, wpool = ThreadPoolExecutor(n_io), ThreadPoolExecutor(n_io)

    def reader():
        try:
            for k, st in enumerate(steps):
                if settings.i_debug >= 0:
                    print('Start working on input file {}'.format(st["inp_era_file_path"]))
                h = q_get(free_in)
                if h is None:
                    return
                raw = _raw_layout(st["inp_era_file_path"], names, h, grid=None if band is None else (ny, nx))
                if band is not None and raw is None:
                    raise ValueError("%s: %s" % (st["inp_era_file_path"], MSG_BAND_FILES.format(vmap['hur'])))
                if raw is not None and os.path.realpath(st["inp_era_file_path"]) != \
                        os.path.realpath(st["out_era_file_path"]):
                    read = raw.read_into if band is None else (lambda f, n, b: raw.read_rows(f, n, b, *rows))
                    with open(st["inp_era_file_path"], "rb", buffering=0) as f:
                        for fut in [rpool.submit(read, f, names[key], h[key].numpy()) for key in IN_FIELDS]:
                            fut.result()
                    IO_STATS["raw"] += 1
                    if not q_put(loaded, (st, raw, h)):
                        return
                    continue
                IO_STATS["decoded"] += 1
                era_file = first if k == 0 else ncio.open_dataset(st["inp_era_file_path"], decode_cf=False)
                for key in IN_FIELDS:
                    h[key].numpy()[...] = np.asarray(era_file[names[key]].data, dtype=np.float32).reshape(h[key].shape)
                if not q_put(loaded, (st, era_file, h)):
                    return
        except BaseException as e:          # surfaced by the main thread
            failure.append(e)
            stop.set()
        finally:
            q_put(loaded, None)

    def writer():
        try:
            while True:
                item = to_write.get()
                if item is None:
                    return
                st, era_file, host = item
                if band is not None:                                  # this rank's rows of the prepared file
                    _write_band(era_file, names, st["out_era_file_path"], host, rows, wpool)
                    free_out.put(host)
                    if settings.i_debug >= 1:
                        print('Done. Saved rows {}..{} to file {}.'.format(rows[0], rows[1], st["out_era_file_path"]))
                    continue
                if not isinstance(era_file, ncio.Dataset):           # raw layout
                    _write_raw(era_file, names, st["inp_era_file_path"], st["out_era_file_path"], host, wpool)
                    free_out.put(host)
                    if settings.i_debug >= 1:
                        print('Done. Saved to file {}.'.format(st["out_era_file_path"]))
                    continue
                for key in _WRITTEN:
                    ref = era_file[names[key]]
                    era_file[names[key]] = ncio.Variable(
                        ref.dims, host[key].numpy().reshape(ref.data.shape).astype(_out_dtype(key, ref.data.dtype)),
                        ref.attrs)
                if vmap['hur'] in era_file:
                    del era_file[vmap['hur']]
                era_file.to_netcdf(st["out_era_file_path"], mode='w')
                era_file.close()
                free_out.put(host)
                if settings.i_debug >= 1:
                    print('Done. Saved to file {}.'.format(st["out_era_file_path"]))
        except BaseException as e:
            # disk full, permission, to_netcdf error ...: the main thread must not keep waiting for the output
            # buffers only this thread hands back
            failure.append(e)
            stop.set()

    tr, tw = threading.Thread(target=reader, daemon=True), threading.Thread(target=writer, daemon=True)
    tr.start(); tw.start()
    in_flight, n_iters = [], []          # FIFO of (step, era_file, host_in, host_out) per pipeline slot use

    def retire(done):
        st, era_file, h_in, h_out = in_flight.pop(0)
        free_in.put(h_in)
        n_iters.append(done["n_iter"])
        to_write.put((st, era_file, h_out))

    try:
        for k in range(len(steps)):
            item = q_get(loaded)
            h_out = q_get(free_out) if item is not None else None
            if band is not None:
                # every rank read its band of file k (or none submits it): no column kernel or band exchange is
                # launched that a peer would wait for in vain
                ok = item is not None and h_out is not None and not failure
                err = None if ok else (failure[0] if failure else RuntimeError("the file pipeline stopped"))
                _agree_or_raise(band, err, _fingerprint(k, _layout_key(item[1], names)) if ok else 0,
                                "reading %s" % steps[k]["inp_era_file_path"])
            if item is None or h_out is None:
                break
            st, era_file, h_in = item
            done = pipe.run(h_in, st["era_step_dt"], h_out, raw=not isinstance(era_file, ncio.Dataset),
                            ignore_top_pressure_error=ignore_top_pressure_error, file_name=st["inp_era_file_path"])
            in_flight.append((st, era_file, h_in, h_out))
            if done is not None:
                retire(done)
        # band mode: every rank got here with every file submitted (the agreements above), and a rerun while
        # draining is an exchange all ranks take part in, so a rank whose writer failed drains too
        if band is not None or not stop.is_set():
            for done in pipe.drain():
                if done is not None:
                    retire(done)
    except BaseException:
        stop.set()                   # the reader must not stay blocked on its queues
        raise
    finally:
        to_write.put(None)
        tw.join()
        stop.set()
        tr.join(timeout=5)
        rpool.shutdown(wait=False)
        wpool.shutdown(wait=False)
    if band is not None:            # every output file is complete on every rank before any rank returns
        _agree_or_raise(band, failure[0] if failure else None, len(n_iters), "writing the output files")
    if failure:
        raise failure[0]
    return n_iters


def _run_file_group(steps, **fargs):
    return pgw_for_era5_files(steps, **fargs)


def debug_interpolate_time(inp_era_file_path, out_era_file_path, delta_input_dir, era_step_dt,
                           ignore_top_pressure_error, debug_mode=None, gcm_grid_deltas=False):
    """step_03_apply_to_era.py:387-414: write the deltas interpolated in time only."""
    from . import functions as F
    if gcm_grid_deltas:
        raise ValueError(MSG_GCM_INTERP_TIME)
    era_file = ncio.open_dataset(inp_era_file_path, decode_cf=False)
    for var_name in ['tos', 'tas', 'hurs', 'ps', 'ta', 'hur', 'ua', 'va', 'zg']:
        print(var_name)
        out_file_path = os.path.join(Path(out_era_file_path).parents[0],
                                     '{}_{}_{}'.format("delta", var_name, Path(out_era_file_path).name))
        delta = F.load_delta(delta_input_dir, var_name, era_file[settings.TIME_ERA].data,
                             target_date_time=era_step_dt)
        out = ncio.Dataset()
        for d in delta.dims:
            if d == settings.TIME_GCM:
                out[d] = era_file[settings.TIME_ERA]
            elif d in delta.coords:
                out[d] = ncio.Variable((d,), delta.coords[d])
        out[var_name] = ncio.Variable(delta.dims, delta.values)
        out.to_netcdf(out_file_path, mode='w')
    era_file.close()


def build_parser():
    parser = argparse.ArgumentParser(
        description="Perturb ERA5 with PGW climate deltas on B200 GPUs. Settings can be made in "
                    "settings.py (or a copy named by the PGW_SETTINGS environment variable). "
                    "Adds the climate change signal for ua, va, ta (with tas near the surface), hus "
                    "(from hur and hurs), skin/SST and soil temperature and sea ice, and iteratively "
                    "updates ps so that the geopotential at the reference pressure changes by the zg "
                    "climate delta.  See the reference's step_03_apply_to_era.py for the method.",
        formatter_class=RawDescriptionHelpFormatter)
    parser.add_argument('-i', '--input_dir', type=str, default=None,
                        help='Directory with ERA5 input files to process (not overwritten).')
    parser.add_argument('-o', '--output_dir', type=str, default=None,
                        help='Directory to store processed ERA5 files.')
    parser.add_argument('-f', '--first_era_step', type=str, default='2006080200',
                        help='Date of first ERA5 time step to process. Format YYYYMMDDHH.')
    parser.add_argument('-l', '--last_era_step', type=str, default='2006080300',
                        help='Date of last ERA5 time step to process. Format YYYYMMDDHH.')
    parser.add_argument('-H', '--hour_inc_step', type=int, default=3,
                        help='Hourly increment of the ERA5 time steps to process.')
    parser.add_argument('-d', '--delta_input_dir', type=str, default=None,
                        help='Directory with GCM climate deltas (SCEN-HIST) for ta,hur,ua,va,zg,tas,hurs,'
                             'ts,tos,siconc and the HIST climatology of ps, all on the ERA5 grid.')
    parser.add_argument('-p', '--n_par', type=int, default=1,
                        help='Number of parallel worker processes (one GPU each, round robin).')
    parser.add_argument('-t', '--ignore_top_pressure_error', action='store_true',
                        help='Ignore the error raised when the climate deltas reach up less far than ERA5.')
    parser.add_argument('-D', '--debug_mode', type=str, default=None,
                        help='"interpolate_time": store the deltas interpolated in time only; '
                             '"interpolate_full": store the final deltas instead of the modified files.')
    parser.add_argument('--latitude_bands', action='store_true',
                        help='Run under torchrun, one rank per GPU: every rank reads, computes and writes its own '
                             'latitude rows of each file, holding only those rows of the climate deltas '
                             '(NetCDF-3 ERA5 files; not in the reference).')
    parser.add_argument('--gcm_grid_deltas', action='store_true',
                        help='The delta files in -d are still on the GCM grid (the input of step_02 regridding, '
                             'normally the output of step_02 smoothing): regrid them on the GPU as step_02 '
                             'regridding would, to the grid of the first ERA5 file, whose FR_LAND masks tos and '
                             'siconc.  Not with --latitude_bands nor -D interpolate_time (not in the reference).')
    return parser


def _check_band_args(args):
    if args.n_par != 1:
        raise ValueError('--latitude_bands runs one rank per GPU under torchrun: -p must be 1.')
    if args.debug_mode is not None:
        raise ValueError('--latitude_bands does not run the debug modes (-D).')
    missing = [k for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK") if k not in os.environ]
    if missing:
        raise ValueError('--latitude_bands needs the environment of torchrun (%s not set): start it as '
                         'torchrun --nproc-per-node N -m pgw4era5_b200.step_03_apply_to_era ... --latitude_bands'
                         % ", ".join(missing))


def _main_bands(step_args, **fargs):
    """``--latitude_bands``: this process is one rank of a torchrun job; it binds its GPU, sets up NCCL (the
    engine's status exchange) and a gloo group (the host-side agreement) and runs the band pipeline over every
    file."""
    import torch
    import torch.distributed as dist
    from .parallel import bind_to_gpu_numa
    local = int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    bind_to_gpu_numa(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    try:
        return pgw_for_era5_files(step_args, band=Band(dist.group.WORLD, dist.new_group(backend="gloo")), **fargs)
    finally:
        dist.destroy_process_group()


def main(argv=None):
    args = build_parser().parse_args(argv)
    if args.input_dir is None:
        raise ValueError('Input directory (-i) is required.')
    if args.output_dir is None:
        raise ValueError('Output directory (-o) is required.')
    if args.delta_input_dir is None:
        raise ValueError('Delta input directory (-d) is required.')
    if args.debug_mode is not None and args.debug_mode not in ['interpolate_time', 'interpolate_full']:
        raise ValueError('Invalid input for argument --debug_mode! Valid arguments are: '
                         '"interpolate_time" or "interpolate_full"')
    first_era_step = datetime.strptime(args.first_era_step, '%Y%m%d%H')
    last_era_step = datetime.strptime(args.last_era_step, '%Y%m%d%H')
    era_step_dts = np.arange(first_era_step, last_era_step + timedelta(hours=args.hour_inc_step),
                             timedelta(hours=args.hour_inc_step)).tolist()
    if args.gcm_grid_deltas and args.latitude_bands:
        raise ValueError(MSG_GCM_BANDS)
    if args.gcm_grid_deltas and args.debug_mode == 'interpolate_time':
        raise ValueError(MSG_GCM_INTERP_TIME)
    if args.latitude_bands:
        _check_band_args(args)
    Path(args.output_dir).mkdir(parents=True, exist_ok=True)
    IMP = None if args.latitude_bands else IterMP(njobs=args.n_par, run_async=True)
    fargs = dict(delta_input_dir=args.delta_input_dir,
                 ignore_top_pressure_error=args.ignore_top_pressure_error, debug_mode=args.debug_mode)
    if args.gcm_grid_deltas:
        fargs["gcm_grid_deltas"] = True
    step_args = []
    for era_step_dt in era_step_dts:
        print(era_step_dt)
        name = settings.era5_file_name_base.format(era_step_dt)
        step_args.append(dict(inp_era_file_path=os.path.join(args.input_dir, name),
                              out_era_file_path=os.path.join(args.output_dir, name),
                              era_step_dt=era_step_dt))
    if args.latitude_bands:
        return _main_bands(step_args, **fargs)
    if args.debug_mode is None:
        # production mode: every worker (GPU) gets its share of the files and pipelines reading,
        # the CUDA pass and writing (the reference hands single files to its pool, :601-638)
        groups = [dict(steps=step_args[w::IMP.njobs]) for w in range(IMP.njobs)]
        IMP.run(_run_file_group, fargs, groups)
        out = [None] * len(step_args)
        for w, res in enumerate(IMP.output):
            out[w::IMP.njobs] = res
        IMP.output = out
        return IMP.output
    if args.debug_mode == 'interpolate_full':
        run_function = pgw_for_era5
    else:
        run_function = debug_interpolate_time
    IMP.run(run_function, fargs, step_args)
    return IMP.output


if __name__ == "__main__":
    main()

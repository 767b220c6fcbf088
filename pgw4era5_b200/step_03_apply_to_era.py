#!/usr/bin/python
# -*- coding: utf-8 -*-
"""
PGW for ERA5, main routine: drop-in for the reference's ``step_03_apply_to_era.py``.

Same command line (``-i -o -f -l -H -d -p -t -D``), same ``settings.py`` names, same file
naming; the per-file work (step_03_apply_to_era.py:44-381 of the reference) runs as one fused
CUDA pass per ERA5 file on a B200 through ``PGWEngine``.  ``-p N`` starts N worker processes,
worker i bound to GPU i % device_count (the reference's pool of CPU workers, parallel.py).

    python -m pgw4era5_b200.step_03_apply_to_era -i era_in -o era_out -d deltas \\
           -f 2006080200 -l 2006080300 -H 3 -t
"""
import argparse
import os
from argparse import RawDescriptionHelpFormatter
from datetime import datetime, timedelta
from pathlib import Path

import numpy as np

from . import ncio, settings
from .parallel import IterMP

_ENGINES = {}


def load_delta_set(delta_input_dir, device="cuda", max_resident_bytes=None):
    """Read every delta file the path needs (ta, hur, ua, va, zg, tas, hurs, ts, tos, siconc as
    SCEN-HIST, ps as HIST; step_03_apply_to_era.py:533-539) into one device-resident DeltaSet, or, when
    that set and the staging copy of one variable would take more than ``max_resident_bytes`` (default:
    half of the device's free memory), into a ``StreamedDeltaSet`` that reads the 3-D deltas of NetCDF-3
    files stamp by stamp.  Only the headers and coordinates of the 3-D files are read to decide."""
    from . import deltastream
    from .engine import DeltaSet, VARS_2D, VARS_3D
    headers = deltastream.read_3d_headers(delta_input_dir)
    if deltastream.should_stream(headers, device, max_resident_bytes):
        return deltastream.open_streamed(delta_input_dir, headers, device=device)
    deltas = {}
    for name in VARS_3D + VARS_2D:
        path, var_name = deltastream.delta_file(delta_input_dir, name)
        ds = ncio.open_dataset(path)
        var = ds[var_name]
        plev = None
        if settings.PLEV_GCM in var.dims:
            plev = np.asarray(ds[settings.PLEV_GCM].data, dtype=np.float64)
        deltas[name] = dict(time=ncio.decode_time(ds[settings.TIME_GCM]), plev=plev, data=var.data)
    return DeltaSet(deltas, device=device)


def get_engine(delta_input_dir, era_file):
    """One engine (and one resident copy of the climatology) per process and delta directory."""
    import torch
    from .engine import PGWEngine
    ak = np.asarray(era_file['ak'].data)
    bk = np.asarray(era_file['bk'].data)
    key = (os.path.abspath(delta_input_dir), torch.cuda.current_device(), ak.tobytes(), bk.tobytes())
    eng = _ENGINES.get(key)
    if eng is None:
        ds = load_delta_set(delta_input_dir, device=torch.device("cuda", torch.cuda.current_device()))
        akm = np.asarray(era_file['akm'].data) if 'akm' in era_file else None      # step_03:68-85
        bkm = np.asarray(era_file['bkm'].data) if 'bkm' in era_file else None
        soil = np.asarray(era_file[settings.SOIL_HLEV_ERA].data) if settings.SOIL_HLEV_ERA in era_file else ()
        eng = PGWEngine(ak, bk, ds, soil1=soil, akm=akm, bkm=bkm)
        _ENGINES[key] = eng
    return eng


def pgw_for_era5(inp_era_file_path, out_era_file_path, delta_input_dir, era_step_dt,
                 ignore_top_pressure_error, debug_mode=None):
    """Same signature as the reference's pgw_for_era5 (step_03_apply_to_era.py:44-47)."""
    import torch
    vmap = settings.var_name_map
    if settings.i_debug >= 0:
        print('Start working on input file {}'.format(inp_era_file_path))
    era_file = ncio.open_dataset(inp_era_file_path, decode_cf=False)
    eng = get_engine(delta_input_dir, era_file)
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


def _raw_layout(path, names, host_in):
    """The header of ``path`` if the file can go through the pipeline without decoding: NetCDF-3, one
    record at most, every ERA5 field float32 with the size of its host buffer, no RELHUM to drop
    (step_03:371).  Else None (the decoding path is taken)."""
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
        if v is None or v.nc_type != NC_FLOAT or (v.is_record and raw.numrecs != 1) or \
                v.nbytes != host_in[key].numel() * 4:
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
    All writes are positional, so ``pool`` (a ThreadPoolExecutor) may run them side by side."""
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


def pgw_for_era5_files(steps, delta_input_dir, ignore_top_pressure_error, debug_mode=None):
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
    """
    import queue
    import threading
    from concurrent.futures import ThreadPoolExecutor
    from .hostpipe import HostPipeline, IN_FIELDS
    if not steps:
        return []
    if debug_mode is not None or settings.i_reinterp or settings.p_ref_inp is None:
        return [pgw_for_era5(delta_input_dir=delta_input_dir,
                             ignore_top_pressure_error=ignore_top_pressure_error, debug_mode=debug_mode, **st)
                for st in steps]
    vmap = settings.var_name_map
    names = _ERA_NAMES(vmap)
    first = ncio.open_dataset(steps[0]["inp_era_file_path"], decode_cf=False)
    eng = get_engine(delta_input_dir, first)
    ny, nx = first[names["PS"]].data.shape[-2:]
    pipe = HostPipeline(eng, ny, nx)
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
                raw = _raw_layout(st["inp_era_file_path"], names, h)
                if raw is not None and os.path.realpath(st["inp_era_file_path"]) != \
                        os.path.realpath(st["out_era_file_path"]):
                    with open(st["inp_era_file_path"], "rb", buffering=0) as f:
                        for fut in [rpool.submit(raw.read_into, f, names[key], h[key].numpy()) for key in IN_FIELDS]:
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
        while True:
            item = q_get(loaded)
            if item is None:
                break
            st, era_file, h_in = item
            h_out = q_get(free_out)
            if h_out is None:
                break
            done = pipe.run(h_in, st["era_step_dt"], h_out, raw=not isinstance(era_file, ncio.Dataset),
                            ignore_top_pressure_error=ignore_top_pressure_error, file_name=st["inp_era_file_path"])
            in_flight.append((st, era_file, h_in, h_out))
            if done is not None:
                retire(done)
        if not stop.is_set():
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
    if failure:
        raise failure[0]
    return n_iters


def _run_file_group(steps, **fargs):
    return pgw_for_era5_files(steps, **fargs)


def debug_interpolate_time(inp_era_file_path, out_era_file_path, delta_input_dir, era_step_dt,
                           ignore_top_pressure_error, debug_mode=None):
    """step_03_apply_to_era.py:387-414: write the deltas interpolated in time only."""
    from . import functions as F
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
    return parser


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
    Path(args.output_dir).mkdir(parents=True, exist_ok=True)
    IMP = IterMP(njobs=args.n_par, run_async=True)
    fargs = dict(delta_input_dir=args.delta_input_dir,
                 ignore_top_pressure_error=args.ignore_top_pressure_error, debug_mode=args.debug_mode)
    step_args = []
    for era_step_dt in era_step_dts:
        print(era_step_dt)
        name = settings.era5_file_name_base.format(era_step_dt)
        step_args.append(dict(inp_era_file_path=os.path.join(args.input_dir, name),
                              out_era_file_path=os.path.join(args.output_dir, name),
                              era_step_dt=era_step_dt))
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

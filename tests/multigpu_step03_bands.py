"""step_03 file to file in latitude bands (``pgw_for_era5_files(band=...)``, the CLI's ``--latitude_bands``) against
the single-GPU file pipeline; run under torchrun, one rank per GPU (not collected by pytest):

    torchrun --standalone --nproc-per-node 8 tests/multigpu_step03_bands.py

Rank 0 writes NetCDF-3 ERA5 files and delta files from a seed (37 x 48 grid: uneven bands, nx a multiple of 4 so
that every band takes the column-kernel flavour of the whole grid) and computes the single-GPU reference; then
every rank runs its band and rank 0 compares the output files:
  (a) default settings, four files, monthly plev19 deltas: byte-identical to the single-GPU pipeline, with the
      band exchange picked automatically and with its NCCL form;
  (b) p_ref_inp = None and i_reinterp = 1: bit-identical to whole-grid PGWEngine.submit driven through
      HostPipeline in the same order; within tests/cases.TOL of the single-GPU CLI (which runs these settings
      through the staged path), with the same iteration counts;
  (c) BASELINE configs[4] settings (plev37 deltas, threshold 1e-3): byte-identical;
  (d) (2 ranks or more) daily deltas under a device-memory limit that makes the single-GPU set stream while
      every band stays resident: byte-identical.
"""
import os
import shutil
import sys
import tempfile
from datetime import datetime, timedelta

import numpy as np
import torch
import torch.distributed as dist

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(HERE))

from cases import TOL, make_case  # noqa: E402
from test_cli_gpu import _write_deltas, _write_era  # noqa: E402
from pgw4era5_b200 import ncio, settings, synthetic as S  # noqa: E402
from pgw4era5_b200 import step_03_apply_to_era as S3  # noqa: E402

NY, NX = 37, 48
T0 = datetime(2006, 8, 2, 0)


def _settings(**kw):
    old = {k: getattr(settings, k) for k in kw}
    for k, v in kw.items():
        setattr(settings, k, v)
    return old


def _steps(root, sub, whens):
    name = settings.era5_file_name_base.format
    return [dict(inp_era_file_path=os.path.join(root, "in", name(w)),
                 out_era_file_path=os.path.join(root, sub, name(w)), era_step_dt=w) for w in whens]


def _make_case(root, seed, n_files, plev=S.PLEV19, daily=False):
    """ERA5 files and deltas under ``root`` (rank 0 only)."""
    for sub in ("in", "deltas", "ref", "cli", "band", "band_nccl"):
        os.makedirs(os.path.join(root, sub))
    era0, deltas = make_case(NY, NX, seed, plev=plev, region="GL")
    if daily:
        deltas = S.make_deltas(era0, seed, ntime=366, plev=plev)
        stamps = np.datetime64("2000-01-01T12:00", "ns") + np.arange(366) * np.timedelta64(86400 * 10 ** 9, "ns")
        for d in deltas.values():
            d["time"] = stamps
    _write_deltas(os.path.join(root, "deltas"), deltas, era0["lat"], era0["lon"])
    whens = [T0 + timedelta(hours=6 * i) for i in range(n_files)]
    for i, w in enumerate(whens):
        era = S.make_era5(NY, NX, 10 * seed + i, lat=era0["lat"], lon=era0["lon"], orog_seed=seed)
        _write_era(os.path.join(root, "in", settings.era5_file_name_base.format(w)), era, w)
    return whens


def _bits(a):
    a = np.ascontiguousarray(a, dtype=np.float32)
    return a.view(np.int32)


def _submit_reference(steps, dd):
    """The whole grid through PGWEngine.submit, driven by HostPipeline in the order the file pipeline submits."""
    from pgw4era5_b200.hostpipe import HostPipeline, IN_FIELDS
    names = S3._ERA_NAMES(settings.var_name_map)
    files = [ncio.open_dataset(st["inp_era_file_path"], decode_cf=False) for st in steps]
    from pgw4era5_b200.engine import PGWEngine
    f0 = files[0]
    eng = PGWEngine(f0["ak"].data, f0["bk"].data, S3.load_delta_set(dd, device=torch.device("cuda")),
                    soil1=f0[settings.SOIL_HLEV_ERA].data)
    pipe = HostPipeline(eng, NY, NX)
    outs, res = [], []
    for st, f in zip(steps, files):
        h = pipe.alloc_host_inputs()
        for key in IN_FIELDS:
            h[key].numpy()[...] = np.asarray(f[names[key]].data, dtype=np.float32).reshape(h[key].shape)
        o = pipe.alloc_host_outputs()
        outs.append(o)
        done = pipe.run(h, st["era_step_dt"], o, ignore_top_pressure_error=True, file_name=st["inp_era_file_path"])
        if done is not None:
            res.append(done)
    res += [d for d in pipe.drain() if d is not None]
    return [r["n_iter"] for r in res], outs


def _compare_files(steps_a, steps_b, label):
    for a, b in zip(steps_a, steps_b):
        with open(a["out_era_file_path"], "rb") as fa, open(b["out_era_file_path"], "rb") as fb:
            assert fa.read() == fb.read(), (label, a["out_era_file_path"])


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    host = dist.new_group(backend="gloo")
    band = S3.Band(dist.group.WORLD, host)
    settings.i_debug = -1
    box = [tempfile.mkdtemp(prefix="pgw_bands_") if rank == 0 else None]
    dist.broadcast_object_list(box, src=0, group=host)
    top = box[0]
    names = S3._ERA_NAMES(settings.var_name_map)
    try:
        # ---- (a) default settings, several files
        root = os.path.join(top, "a")
        whens = _make_case(root, 61, 4) if rank == 0 else None
        whens = _bcast(whens, host)
        if rank == 0:
            n_ref = S3.pgw_for_era5_files(_steps(root, "ref", whens), os.path.join(root, "deltas"), True)
        # both forms of the band exchange under HostPipeline's two streams: "auto" (peer memory where it can be
        # mapped) and the NCCL all-reduce
        for sub, b in (("band", band), ("band_nccl", band._replace(exchange="nccl"))):
            n_band = S3.pgw_for_era5_files(_steps(root, sub, whens), os.path.join(root, "deltas"), True, band=b)
            if rank == 0:
                assert n_band == n_ref, (sub, n_band, n_ref)
                _compare_files(_steps(root, sub, whens), _steps(root, "ref", whens), "a " + sub)
                print("(a) default settings, exchange %s: %d files byte-identical to the single-GPU pipeline, "
                      "n_iter %s" % (b.exchange, len(whens), n_band), flush=True)

        # ---- (b) p_ref_inp = None, i_reinterp = 1
        for setting in (dict(p_ref_inp=None), dict(i_reinterp=1)):
            old = _settings(**setting)
            try:
                root = os.path.join(top, "b_%s" % "_".join(setting))
                whens = _bcast(_make_case(root, 62, 3) if rank == 0 else None, host)
                dd = os.path.join(root, "deltas")
                if rank == 0:
                    n_sub, outs = _submit_reference(_steps(root, "x", whens), dd)
                    n_cli = S3.pgw_for_era5_files(_steps(root, "cli", whens), dd, True)   # staged path
                n_band = S3.pgw_for_era5_files(_steps(root, "band", whens), dd, True, band=band)
                if rank == 0:
                    assert n_band == n_sub == n_cli, (setting, n_band, n_sub, n_cli)
                    worst = {}
                    for st, o, stc in zip(_steps(root, "band", whens), outs, _steps(root, "cli", whens)):
                        got = ncio.open_dataset(st["out_era_file_path"])
                        cli = ncio.open_dataset(stc["out_era_file_path"])
                        for key in S3._WRITTEN:
                            g = got[names[key]].data
                            assert np.array_equal(_bits(g), _bits(o[key].numpy().reshape(g.shape))), (setting, key)
                            c = cli[names[key]].data.astype(np.float64)
                            assert np.array_equal(np.isnan(g), np.isnan(c)), (setting, key)
                            err = float(np.nanmax(np.abs(g.astype(np.float64) - c))) if g.size else 0.0
                            assert err <= TOL.get(key, 1e-4), (setting, key, err)
                            worst[key] = max(worst.get(key, 0.0), err)
                    print("(b) %s: bit-identical to whole-grid submit, n_iter %s; vs staged CLI max|diff| %s"
                          % (setting, n_band, {k: "%.1e" % v for k, v in worst.items()}), flush=True)
            finally:
                _settings(**old)

        # ---- (c) BASELINE configs[4]: plev37 deltas, threshold 1e-3
        old = _settings(thresh_phi_ref_max_error=1e-3)
        try:
            root = os.path.join(top, "c")
            whens = _bcast(_make_case(root, 63, 2, plev=S.PLEV37) if rank == 0 else None, host)
            if rank == 0:
                n_ref = S3.pgw_for_era5_files(_steps(root, "ref", whens), os.path.join(root, "deltas"), True)
            n_band = S3.pgw_for_era5_files(_steps(root, "band", whens), os.path.join(root, "deltas"), True, band=band)
            if rank == 0:
                assert n_band == n_ref, (n_band, n_ref)
                _compare_files(_steps(root, "band", whens), _steps(root, "ref", whens), "c")
                print("(c) configs[4] settings: byte-identical, n_iter %s" % n_band, flush=True)
        finally:
            _settings(**old)

        # ---- (d) daily deltas that stream on one GPU and fit per band
        if world > 1:
            from pgw4era5_b200 import deltastream
            from pgw4era5_b200.parallel import split_rows
            root = os.path.join(top, "d")
            whens = _bcast(_make_case(root, 64, 3, daily=True) if rank == 0 else None, host)
            dd = os.path.join(root, "deltas")
            need = deltastream.resident_bytes(deltastream.read_3d_headers(dd))
            limit = need * max(b - a for a, b in split_rows(NY, world)) // NY + 1
            assert limit < need
            load = S3.load_delta_set
            S3.load_delta_set = lambda d, device="cuda", rows=None: load(d, device, max_resident_bytes=limit, rows=rows)
            try:
                S3._ENGINES.clear()
                if rank == 0:
                    n_ref = S3.pgw_for_era5_files(_steps(root, "ref", whens), dd, True)
                    assert any(getattr(e.deltas, "streamed", False) for e in S3._ENGINES.values())
                n_band = S3.pgw_for_era5_files(_steps(root, "band", whens), dd, True, band=band)
                assert not any(getattr(e.deltas, "streamed", False) for e in S3._ENGINES.values()
                               if e.group is not None)
            finally:
                S3.load_delta_set = load
            if rank == 0:
                assert n_band == n_ref
                _compare_files(_steps(root, "band", whens), _steps(root, "ref", whens), "d")
                print("(d) daily deltas: streamed on one GPU (%.1f MB), resident per band (limit %.1f MB): "
                      "byte-identical" % (need / 1e6, limit / 1e6), flush=True)
        elif rank == 0:
            print("(d) skipped: one rank (the band is the whole grid)", flush=True)
        dist.barrier(group=host)
        if rank == 0:
            print("multigpu_step03_bands: all checks passed on %d rank(s)" % world, flush=True)
    finally:
        if rank == 0:
            shutil.rmtree(top, ignore_errors=True)
        dist.destroy_process_group()


def _bcast(obj, group):
    box = [obj]
    dist.broadcast_object_list(box, src=0, group=group)
    return box[0]


if __name__ == "__main__":
    main()

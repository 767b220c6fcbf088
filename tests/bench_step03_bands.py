#!/usr/bin/env python
"""
File -> file wall time of step_03 in latitude bands (``--latitude_bands``) next to the single-GPU command line, on
global 721 x 1440 x 137 NetCDF-3 snapshots generated on local disk (2.3 GB per file in, as much out) with monthly
plev19 deltas.  Run under torchrun, one rank per GPU; prints one JSON line on rank 0 (and writes it to --out):

    torchrun --standalone --nproc-per-node 8 tests/bench_step03_bands.py --files 2 --out profiles/r3_step03_bands.json

  * ``cli_one_gpu_s_per_file``: the existing command line's pipeline on rank 0's GPU (measured at every W);
  * ``bands_s_per_file``: the band pipeline over all W ranks, rank 0 creating the output files included;
  * ``per_rank``: one band, stage by stage on the first file (page cache warm): read rows -> pinned buffers,
    H2D + kernels + band exchange + D2H, write rows -> output file, and the device memory of the delta band;
  * the GPU's name and power limit, read in the same run; with ``--bench-json`` (a bench.py result line) its
    ``e2e.link_bound`` next to the band path's host<->device bytes per second.
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import time
from datetime import datetime, timedelta

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def _gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        return q[0] if q else None
    except (OSError, subprocess.SubprocessError):
        return None


def _make_files(a, inp, dd, whens):
    import numpy as np
    import torch
    from pgw4era5_b200 import settings, synthetic as S
    from test_cli_gpu import _write_deltas, _write_era
    lat, lon = np.linspace(-90.0, 90.0, a.ny), 0.25 * np.arange(a.nx)
    era0 = S.make_era5(a.ny, a.nx, 1, device="cuda", lat=lat, lon=lon)
    _write_deltas(dd, S.to_numpy(S.make_deltas(era0, 1, device="cuda")), lat, lon)
    del era0
    for i, w in enumerate(whens):
        _write_era(os.path.join(inp, settings.era5_file_name_base.format(w)),
                   S.to_numpy(S.make_era5(a.ny, a.nx, 100 + i, device="cuda", lat=lat, lon=lon, orog_seed=1)), w)
        torch.cuda.empty_cache()


def _stages(steps, dd, band):
    """One band stage by stage on the first file: read, GPU (H2D, kernels, exchange, D2H), write."""
    import torch
    import torch.distributed as dist
    from concurrent.futures import ThreadPoolExecutor
    from pgw4era5_b200 import ncio, settings, step_03_apply_to_era as S3
    from pgw4era5_b200.hostpipe import HostPipeline, IN_FIELDS
    names = S3._ERA_NAMES(settings.var_name_map)
    st = steps[0]
    first = ncio.open_dataset(st["inp_era_file_path"], decode_cf=False)
    eng = S3.get_engine(dd, first, band)
    r0, r1 = band.rows
    ny, nx = first[names["PS"]].data.shape[-2:]
    pipe = HostPipeline(eng, r1 - r0, nx)
    h_in, h_out = pipe.alloc_host_inputs(), pipe.alloc_host_outputs()
    raw = S3._raw_layout(st["inp_era_file_path"], names, h_in, grid=(ny, nx))
    pool = ThreadPoolExecutor(max(1, min(8, (os.cpu_count() or 2) // 2)))

    def best(fn, reps=3):
        ts = []
        for _ in range(reps):
            dist.barrier(group=band.host_group)
            t = time.perf_counter(); fn(); ts.append(time.perf_counter() - t)
        return min(ts)

    def read():
        with open(st["inp_era_file_path"], "rb", buffering=0) as f:
            for fut in [pool.submit(raw.read_rows, f, names[k], h_in[k].numpy(), r0, r1) for k in IN_FIELDS]:
                fut.result()

    def gpu():
        pipe.run(h_in, st["era_step_dt"], h_out, raw=True, ignore_top_pressure_error=True)
        pipe.drain()
        torch.cuda.synchronize()
    out = dict(rows=[r0, r1], read_rows_s=best(read))
    gpu()
    out["h2d_kernels_exchange_d2h_s"] = best(gpu)
    out["write_rows_s"] = best(lambda: S3._write_band(raw, names, st["out_era_file_path"], h_out, (r0, r1), pool))
    out["h2d_plus_d2h_bytes"] = pipe.h2d_bytes + pipe.d2h_bytes
    out["delta_set_device_bytes"] = sum(t.numel() * t.element_size() for t in eng.deltas.tensors())
    out["band_exchange"] = eng.band_exchange
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--files", type=int, default=2)
    ap.add_argument("--dir", default="/tmp/pgw_bands_bench")
    ap.add_argument("--ny", type=int, default=721)
    ap.add_argument("--nx", type=int, default=1440)
    ap.add_argument("--out", default=None)
    ap.add_argument("--bench-json", default=None, help="a result line of bench.py, for its e2e.link_bound")
    a = ap.parse_args()
    import torch
    import torch.distributed as dist
    from pgw4era5_b200 import settings, step_03_apply_to_era as S3
    from pgw4era5_b200.parallel import bind_to_gpu_numa
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    bind_to_gpu_numa(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    host = dist.new_group(backend="gloo")
    settings.i_debug = -1
    inp, dd = os.path.join(a.dir, "in"), os.path.join(a.dir, "deltas")
    whens = [datetime(2006, 8, 1, 0) + timedelta(hours=6 * i) for i in range(a.files)]
    name = settings.era5_file_name_base.format
    steps = lambda out: [dict(inp_era_file_path=os.path.join(inp, name(w)),
                              out_era_file_path=os.path.join(a.dir, out, name(w)), era_step_dt=w) for w in whens]
    res = {}
    try:
        if rank == 0:
            shutil.rmtree(a.dir, ignore_errors=True)
            for p in (inp, dd, os.path.join(a.dir, "cli"), os.path.join(a.dir, "band"), os.path.join(a.dir, "warm")):
                os.makedirs(p)
            t = time.perf_counter()
            _make_files(a, inp, dd, whens)
            res["generate_s"] = time.perf_counter() - t
            fbytes = os.path.getsize(steps("x")[0]["inp_era_file_path"])
            # the single-GPU command line's pipeline: once to load the climatology and warm the page cache
            S3.pgw_for_era5_files(steps("warm"), dd, True)
            torch.cuda.synchronize()
            t = time.perf_counter()
            S3.pgw_for_era5_files(steps("cli"), dd, True)
            res["cli_one_gpu_s_per_file"] = (time.perf_counter() - t) / a.files
            S3._ENGINES.clear()
            torch.cuda.empty_cache()
            res["file_bytes"] = fbytes
            res["disk_bytes_used"] = sum(os.path.getsize(os.path.join(dp, f)) for dp, _, fs in os.walk(a.dir)
                                         for f in fs)
        dist.barrier(group=host)
        band = S3.Band(dist.group.WORLD, host)
        torch.cuda.reset_peak_memory_stats()
        S3.pgw_for_era5_files(steps("band"), dd, True, band=band)      # warm: band deltas, engine, page cache
        dist.barrier(group=host)
        t = time.perf_counter()
        S3.pgw_for_era5_files(steps("band"), dd, True, band=band)
        t_band = (time.perf_counter() - t) / a.files
        rows = next(k[-2] for k in S3._ENGINES if len(k) > 4)
        stages = _stages(steps("band"), dd, band._replace(rows=rows))
        stages["peak_device_bytes"] = torch.cuda.max_memory_allocated()
        gathered = [None] * world
        dist.all_gather_object(gathered, stages, group=host)
        if rank == 0:
            import filecmp
            same = all(filecmp.cmp(s["out_era_file_path"], c["out_era_file_path"], shallow=False)
                       for s, c in zip(steps("band"), steps("cli")))
            res.update(workload="%d global %dx%dx137 NetCDF-3 snapshots (%.2f GB each), monthly plev19 deltas, "
                                "file to file" % (a.files, a.ny, a.nx, res["file_bytes"] / 1e9),
                       gpu=_gpu_info(), n_gpus=world, bands_s_per_file=t_band,
                       band_outputs_byte_identical_to_cli=same, per_rank=gathered,
                       speedup_vs_one_gpu=res["cli_one_gpu_s_per_file"] / t_band)
            if a.bench_json:
                with open(a.bench_json) as f:
                    line = [ln for ln in f.read().splitlines() if ln.startswith("{")][-1]
                e2e = json.loads(line).get("e2e", {})
                res["bench_e2e_link_bound"] = e2e.get("link_bound")
                res["bench_e2e"] = {k: v for k, v in e2e.items() if k != "link_bound"}
            res["h2d_plus_d2h_GBps_per_rank_of_gpu_stage"] = [
                s["h2d_plus_d2h_bytes"] / s["h2d_kernels_exchange_d2h_s"] / 1e9 for s in gathered]
            line = json.dumps(res)
            print(line, flush=True)
            if a.out:
                with open(a.out, "w") as f:
                    f.write(line + "\n")
    finally:
        dist.barrier(group=host)
        if rank == 0:
            shutil.rmtree(a.dir, ignore_errors=True)
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

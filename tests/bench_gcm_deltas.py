"""
Cost of regridding the climatology on the device (gcmdeltas.GcmGridDeltaSet: plev19 daily deltas on a 192 x 384
GCM grid, ERA5-grid stamps produced when a timestep first needs them) next to the two sets that read deltas
already on the ERA5 grid, on the global 721 x 1440 x 137 grid, one GPU, in one process:

  resident   the regridded climatology in HBM (DeltaSet, a slice of 30 daily stamps)
  streamed   the same regridded deltas from host memory (StreamedDeltaSet, in-memory source)
  gcm_grid   the GCM-grid deltas in HBM, each stamp regridded on the copy stream (GcmGridDeltaSet)

    python tests/bench_gcm_deltas.py --steps 200 --warmup 8 --out profiles/r3_gcm_deltas.json

The loop is that of bench_delta_stream.py: ERA5 inputs cycle through a ring of 4 resident timesteps (2.3 GB each,
>> 126 MB L2) with 3-hourly dates, PGWEngine.submit with 2 timesteps in flight, so a new daily stamp is needed
every 8 timesteps.  Reported: ms per timestep of each set; per load of the GCM-grid set the time of the d4
regrid-pack and of the zg regrid (CUDA events on the copy stream after its wait for the slot's last reader); the
d4 kernel alone over repeated launches, fused and as four regrids plus a pack, with its bytes (stamp written once
plus source read once, from the shapes) per second and share of the 7.7 TB/s HBM peak; the device memory of each
set; and whether every output of every timestep of the GCM-grid set is bit-identical to the resident one.
"""
import argparse
import ctypes as C
import json
import os
import sys
import time
from datetime import datetime, timedelta

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)

from bench_reinterp import gpu_info          # noqa: E402

DAY = np.timedelta64(86400 * 10 ** 9, "ns")
HBM_PEAK = 7.7e12                            # bytes/s, HGX B200 data sheet, one GPU
OUTS = ("PS", "delta_ps", "T", "QV", "U", "V", "T_SKIN", "T_SO", "FR_SEA_ICE")


def kernel_times(ds, reps):
    """ms per launch of the d4 load kernels alone on stamp 0: pgw_regrid_pack_d4_f32, and regrid_arrays' kernel on
    each of the four variables into a scratch followed by pgw_pack_d4_f32 (what step_02 + the streamed set do)."""
    from pgw4era5_b200 import _native as N
    r = ds.rings["d4"]
    g, st = r.grid, C.c_void_p(torch.cuda.current_stream().cuda_stream)
    dst = r.bufs[0]
    n = r.n
    scratch = torch.empty(4 * n, device=dst.device, dtype=torch.float32)
    p = lambda t: C.c_void_p(t.data_ptr())
    field = g.ny_s * g.nx_s * r.K

    def fused():
        N.check(N.lib.pgw_regrid_pack_d4_f32(p(r.src[0]), p(dst), p(r.pm[0]), r.K, g.ny_s, g.nx_s, *g.args(),
                                             C.c_void_p(0), st), "pgw_regrid_pack_d4_f32")

    def unfused():
        for v in range(4):
            N.check(N.lib.pgw_regrid_bilinear_band_f32(
                C.c_void_p(r.src[0].data_ptr() + 4 * v * field), C.c_void_p(scratch.data_ptr() + 4 * v * n),
                C.c_void_p(r.pm[0].data_ptr() + 8 * v * r.K), r.K, g.ny_s, g.nx_s, *g.args(), st), "regrid")
        N.check(N.lib.pgw_pack_d4_f32(*[C.c_void_p(scratch.data_ptr() + 4 * v * n) for v in range(4)], p(dst), n, 0,
                                      st), "pack")
    out = {}
    for name, fn in (("fused", fused), ("regrid_then_pack", unfused)):
        for _ in range(5):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        out[name + "_ms"] = e0.elapsed_time(e1) / reps
    fused()
    torch.cuda.synchronize()
    nbytes = n * 16 + r.src[0].numel() * 4
    t = out["fused_ms"] * 1e-3
    out.update(launches=reps, bytes_per_launch=nbytes, stamp_store_bytes=n * 16, source_read_bytes=r.src[0].numel() * 4,
               bytes_per_s=nbytes / t, share_of_hbm_peak=nbytes / t / HBM_PEAK,
               bound="memory: 16 B stored per node and column against 12 float64 operations and 8 shared-memory "
                     "loads of the blended rows; the 22 MB source is read from L2 after the first pass")
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--days", type=int, default=30)
    ap.add_argument("--slots", type=int, default=4)
    ap.add_argument("--ring", type=int, default=4)
    ap.add_argument("--kernel-reps", type=int, default=50)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_gcm_deltas.py measures on the GPU; no CUDA device found")
    from pgw4era5_b200 import functions as F
    from pgw4era5_b200 import settings, synthetic as S
    from pgw4era5_b200.deltastream import StreamedDeltaSet
    from pgw4era5_b200.engine import DeltaSet, PGWEngine
    from pgw4era5_b200.gcmdeltas import OCEAN_VARS, GcmGridDeltaSet
    settings.i_debug = 0
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    ny, nx = 721, 1440
    era0 = S.make_era5(ny, nx, 2, device=dev, orog_seed=2)
    ring = [era0] + [S.make_era5(ny, nx, 100 + i, device=dev, orog_seed=2) for i in range(1, a.ring)]
    glat, glon = np.linspace(-89.28, 89.28, 192), np.arange(384) * 0.9375
    t0 = time.perf_counter()
    gera = S.make_era5(len(glat), len(glon), 2, device=dev, lat=glat, lon=glon)
    gcm = S.make_deltas(gera, 2, plev=S.PLEV19, device=dev, ntime=a.days)
    stamps = np.datetime64("2001-01-01T12:00", "ns") + np.arange(a.days) * DAY
    olat, olon = np.meshgrid(glat, glon, indexing="ij")
    for name, d in gcm.items():
        d["time"] = stamps
        d["data"] = d["data"].cpu().numpy()
        d["lat"], d["lon"] = (olat, olon) if name in OCEAN_VARS else (glat, glon)
    del gera
    land = era0["FR_LAND"][0].cpu().numpy()
    lat, lon = era0["lat"], era0["lon"]
    # the regridded climatology step_02 would write, in host memory
    era_grid = {}
    for name, d in gcm.items():
        if name in OCEAN_VARS:
            data = F.nan_ignoring_interp_arrays(land, lat, lon, d["data"], d["lat"], d["lon"],
                                                settings.nan_interp_kernel_radius, settings.nan_interp_sharpness)
        else:
            data = F.regrid_arrays(d["data"], d["lat"], d["lon"], lat, lon)
        era_grid[name] = dict(time=stamps, plev=d["plev"], data=torch.from_numpy(np.asarray(data)))
    torch.cuda.empty_cache()
    gen_s = time.perf_counter() - t0
    base = datetime(2001, 1, 1, 12)
    when = lambda i: base + timedelta(hours=3 * i)
    assert a.warmup + a.steps <= 8 * (a.days - 1), "the dates must stay inside the stamps"

    def run(eng, steps, first, outs, collect=None):
        pend = []
        for k in range(steps):
            i = first + k
            pend.append(eng.submit(ring[i % a.ring], when(i), out=outs[i % 2], ignore_top_pressure_error=True,
                                   slot=i % 2))
            if len(pend) >= 2:
                r = pend.pop(0).result()
                if collect is not None:
                    collect(r)
        for p in pend:
            r = p.result()
            if collect is not None:
                collect(r)

    def leg(ds):
        eng = PGWEngine(era0["ak"], era0["bk"], ds, soil1=era0["soil1"])
        outs = [eng.alloc_outputs(ny, nx, len(era0["soil1"])) for _ in range(2)]
        run(eng, a.warmup, 0, outs)
        torch.cuda.synchronize()
        streamed = getattr(ds, "streamed", False)
        if streamed:
            ds.load_events = []
            loads0 = {k: r.loads for k, r in ds.rings.items()}
        n_iter = []
        h0 = time.perf_counter()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        run(eng, a.steps, a.warmup, outs, lambda r: n_iter.append(r["n_iter"]))
        e1.record()
        torch.cuda.synchronize()
        r = dict(ms_per_timestep=e0.elapsed_time(e1) / a.steps, host_s=time.perf_counter() - h0, steps=a.steps,
                 warmup=a.warmup, n_iter_mean=float(np.mean(n_iter)), reruns=eng.stats["reruns"],
                 device_bytes=ds.device_bytes() if streamed else ds.arena.numel() * 4)
        if streamed:
            r["loads_timed"] = {k: ring_.loads - loads0[k] for k, ring_ in ds.rings.items()}
            for name in ds.rings:
                ev = [x for x in ds.load_events if x["ring"] == name]
                r["load_" + name] = dict(
                    n=len(ev), host_fill_ms_mean=1e3 * float(np.mean([x["fill_s"] for x in ev])),
                    first_interval_ms_mean=float(np.mean([x["events"][0].elapsed_time(x["events"][1]) for x in ev])),
                    second_interval_ms_mean=float(np.mean([x["events"][1].elapsed_time(x["events"][2]) for x in ev])),
                    second_interval_ms_max=float(np.max([x["events"][1].elapsed_time(x["events"][2]) for x in ev])))
            ds.load_events = None
        return r

    out = dict(workload="global %dx%dx137, plev19 daily deltas (%d stamps) on a 192x384 GCM grid, 3-hourly dates, "
                        "ring of %d resident ERA5 timesteps, 2 in flight" % (ny, nx, a.days, a.ring),
               gpu=gpu_info(0), generate_s=gen_s, slots=a.slots,
               load_intervals="streamed: first = H2D, second = waits for the slot's readers + pack; gcm_grid: first "
                              "= waits for the slot's readers, second = the regrid kernel (d4: "
                              "pgw_regrid_pack_d4_f32, zg: pgw_regrid_bilinear_band_f32)")
    t0 = time.perf_counter()
    gset = GcmGridDeltaSet(gcm, lat, lon, land, device=dev, slots=a.slots)
    torch.cuda.synchronize()
    out["gcm_grid_construct_s"] = time.perf_counter() - t0
    out["d4_kernel"] = kernel_times(gset, a.kernel_reps)
    resident = DeltaSet(era_grid, device=dev)
    out["resident"] = leg(resident)
    out["streamed"] = leg(StreamedDeltaSet(era_grid, device=dev, slots=a.slots))
    out["gcm_grid"] = leg(gset)
    for k in ("streamed", "gcm_grid"):
        out[k + "_over_resident"] = out[k]["ms_per_timestep"] / out["resident"]["ms_per_timestep"]
    # every output of every timestep, resident and GCM-grid sets in lockstep on fresh engines
    ea = PGWEngine(era0["ak"], era0["bk"], resident, soil1=era0["soil1"])
    eb = PGWEngine(era0["ak"], era0["bk"], gset, soil1=era0["soil1"])
    same, n = True, a.warmup + a.steps
    for i in range(n):
        x = ea.submit(ring[i % a.ring], when(i), ignore_top_pressure_error=True).result()
        y = eb.submit(ring[i % a.ring], when(i), ignore_top_pressure_error=True).result()
        for k in OUTS:
            same &= bool(torch.equal(x[k].view(torch.int32), y[k].view(torch.int32)))
        same &= x["n_iter"] == y["n_iter"]
    out["bit_identical"] = dict(timesteps=n, all_outputs_equal=same)
    text = json.dumps(out, indent=1)
    print(text, flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()

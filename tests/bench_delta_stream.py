"""
Cost of streaming a daily climatology (deltastream.StreamedDeltaSet, a ring of 4 stamps per ring) next to the
resident DeltaSet, on the global 721 x 1440 x 137 grid with plev19 deltas, one GPU, in one process:

  resident   the whole climatology in HBM (DeltaSet), PGWEngine.submit, 2 timesteps in flight
  streamed   the same deltas from host memory (in-memory source), same loop

    python tests/bench_delta_stream.py --steps 200 --warmup 8 --out profiles/r3_delta_stream.json

ERA5 inputs cycle through a ring of 4 resident timesteps (2.3 GB each, >> 126 MB L2) with 3-hourly dates, so a
new daily stamp is needed every 8 timesteps.  Reported: ms per timestep, per stamp load the host fill time, the
H2D time and the pack time (CUDA events on the copy stream; the pack interval also holds the wait for the
timestep that last read the slot), the device memory of each set, and whether every output of every timestep
is bit-identical between the two.  --days 365 times the streamed set alone: the generated days are tiled to a
year (stamp i holds day i % 30), which moves the same bytes without 150 GB of host memory.
"""
import argparse
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

GEN_DAYS = 30
DAY = np.timedelta64(86400 * 10 ** 9, "ns")


class TiledSource:
    """Stamp i of a year made of the generated days: day i % len(days)."""
    swap = 0

    def __init__(self, t, days):
        self.t, self.shape = t, (days,) + tuple(t.shape[1:])

    def read(self, i, out):
        out.copy_(self.t[i % self.t.shape[0]].reshape(-1))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--days", type=int, default=30)
    ap.add_argument("--slots", type=int, default=4)
    ap.add_argument("--ring", type=int, default=4)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_delta_stream.py measures on the GPU; no CUDA device found")
    from pgw4era5_b200 import settings, synthetic as S
    from pgw4era5_b200.deltastream import StreamedDeltaSet
    from pgw4era5_b200.engine import VARS_3D, DeltaSet, PGWEngine
    settings.i_debug = 0
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    ny, nx = 721, 1440
    era0 = S.make_era5(ny, nx, 2, device=dev, orog_seed=2)
    ring = [era0] + [S.make_era5(ny, nx, 100 + i, device=dev, orog_seed=2) for i in range(1, a.ring)]
    gen = min(a.days, GEN_DAYS)
    t0 = time.perf_counter()
    deltas = S.make_deltas(era0, 2, plev=S.PLEV19, device=dev, ntime=gen)
    stamps = np.datetime64("2001-01-01T12:00", "ns") + np.arange(a.days) * DAY
    for name, d in deltas.items():
        d["time"] = stamps
        d["data"] = d["data"].cpu()
        if a.days > gen:
            d["data"] = TiledSource(d["data"], a.days) if name in VARS_3D else \
                d["data"].repeat((a.days + gen - 1) // gen, 1, 1)[:a.days]
    torch.cuda.empty_cache()
    gen_s = time.perf_counter() - t0
    host_bytes = sum(d["data"].t.numel() * 4 if isinstance(d["data"], TiledSource) else d["data"].numel() * 4
                     for d in deltas.values())
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
        if getattr(ds, "streamed", False):
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
                 warmup=a.warmup, n_iter_mean=float(np.mean(n_iter)), reruns=eng.stats["reruns"])
        if getattr(ds, "streamed", False):
            r["device_bytes"] = ds.device_bytes()
            r["loads_timed"] = {k: ring_.loads - loads0[k] for k, ring_ in ds.rings.items()}
            for name in ds.rings:
                ev = [x for x in ds.load_events if x["ring"] == name]
                r["load_" + name] = dict(
                    n=len(ev), fill_ms_mean=1e3 * float(np.mean([x["fill_s"] for x in ev])),
                    h2d_ms_mean=float(np.mean([x["events"][0].elapsed_time(x["events"][1]) for x in ev])),
                    pack_ms_mean=float(np.mean([x["events"][1].elapsed_time(x["events"][2]) for x in ev])),
                    stamp_bytes=ds.rings[name].n * 4 * len(ds.rings[name].sources))
            ds.load_events = None
        else:
            r["device_bytes"] = ds.arena.numel() * 4
        return r, eng

    tiled = ", the %d generated days tiled" % gen if a.days > gen else ""
    out = dict(workload="global %dx%dx137, plev19 daily deltas (%d stamps%s, in-memory source), 3-hourly dates, "
                        "ring of %d resident ERA5 timesteps, 2 in flight" % (ny, nx, a.days, tiled, a.ring),
               gpu=gpu_info(0), host_delta_bytes=host_bytes, generate_s=gen_s, slots=a.slots)
    streamed = StreamedDeltaSet(deltas, device=dev, slots=a.slots)
    if a.days <= GEN_DAYS:
        resident = DeltaSet(deltas, device=dev)
        out["resident"], eng_r = leg(resident)
    out["streamed"], eng_s = leg(streamed)
    if a.days <= GEN_DAYS:
        out["streamed_over_resident"] = out["streamed"]["ms_per_timestep"] / out["resident"]["ms_per_timestep"]
        # every output of every timestep, both sets in lockstep on fresh engines
        ea = PGWEngine(era0["ak"], era0["bk"], resident, soil1=era0["soil1"])
        eb = PGWEngine(era0["ak"], era0["bk"], streamed, soil1=era0["soil1"])
        same, n = True, a.warmup + a.steps
        for i in range(n):
            x = ea.submit(ring[i % a.ring], when(i), ignore_top_pressure_error=True).result()
            y = eb.submit(ring[i % a.ring], when(i), ignore_top_pressure_error=True).result()
            for k in ("PS", "delta_ps", "T", "QV", "U", "V", "T_SKIN", "T_SO", "FR_SEA_ICE"):
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

#!/usr/bin/env python
"""
Benchmark of the PGW4ERA5 per-timestep path on B200 (contract: see DESIGN.md "Measurement").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Metric (BASELINE.json): global 0.25 degree ERA5 timesteps/s.  One "step" is one
full ERA5 timestep (721x1440 columns x 137 levels, plev19 deltas) through the
fused CUDA pass.  N > 1: every rank processes its own timesteps (the
reference's own parallelism: one file = one task), so `value` = N*K / max-over-
ranks time, scaling "weak"; the delta climatology is NCCL-broadcast once before
the timed region.  Inputs cycle through a ring of distinct device-resident
synthetic timesteps (each 2.3 GB, far larger than the 126 MB L2); up to four
timesteps are in flight (the host reads a timestep's status while the next ones
are queued) and consecutive timesteps alternate between two CUDA streams.
Further legs of the same line: `e2e` (host buffers, copies inside the timing)
with the platform's measured link bound, `roofline`, `cpu_baseline` (N = 1),
`config.broadcast` and `config.latband` (N > 1: one global snapshot of BASELINE
configs[4] in latitude bands).  `--impl reference`: the reference path's CPU
implementation on all host cores.  `--dump-outputs DIR`: what the last timed
step returned, as .npy files (see `dump_outputs`); the inputs depend only on
the arguments, so two builds can be compared output for output.

Prints ONE JSON line (rank 0).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time
from datetime import datetime, timedelta

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "global 0.25deg ERA5 timesteps/s"
GRIDS = {"GL": (721, 1440), "EU": (201, 281)}
DUMP_COLUMNS = 8192


def algorithmic_bytes(ncol, nlev=137, nplev=19, nsoil=4):
    """SURVEY.md 8(d): every input read once, every output written once, fp32."""
    n4 = ncol * 4
    reads = 4 * nlev * n4 + 4 * 2 * nplev * n4 + 7 * 2 * n4 + n4 + 5 * n4 + nsoil * n4
    writes = 4 * nlev * n4 + 3 * n4 + nsoil * n4
    return reads + writes


def measured_peak_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md): one
    `nvidia-smi -lms 100` process runs across the region; samples are kept by wall-clock time."""
    Q = ("timestamp,index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_indices):
        """One nvidia-smi process for all the GPUs of the job, started by rank 0 only: a poller per rank (eight
        of them on eight GPUs, each taking driver locks every 100 ms) disturbs the launch path it observes."""
        self.gpu, self.proc, self.t0, self.t1 = gpu_indices, None, None, None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", ",".join(str(g) for g in gpu_indices),
                                          "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms",
                                          "20" if len(gpu_indices) <= 2 else "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def mark_start(self):
        self.t0 = time.time()

    def mark_stop(self):
        """End of a timed region; may be called again: the window then extends to the end of the later region
        (device-resident steps first, the e2e leg after it), the first end is kept for `samples_in_region`."""
        if self.t1 is not None and not hasattr(self, "t1_first"):
            self.t1_first = self.t1
        self.t1 = time.time()

    def summary(self):
        rows = []
        if self.proc is not None:
            time.sleep(0.25)
            self.proc.terminate()
            try:
                out, _ = self.proc.communicate(timeout=5)
            except Exception:
                out = ""
            for line in out.splitlines():
                r = [x.strip() for x in line.split(",")]
                if len(r) < 10:
                    continue
                try:
                    ts = datetime.strptime(r[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                except ValueError:
                    continue
                rows.append((ts, r))
        inside = [r for ts, r in rows if self.t0 is not None and self.t0 - 0.05 <= ts <= self.t1 + 0.15]
        t1a = getattr(self, "t1_first", self.t1)
        first = [r for ts, r in rows if self.t0 is not None and self.t0 - 0.05 <= ts <= t1a + 0.15]
        use = inside if inside else [r for _, r in rows]
        num = lambda x: float(x) if x.replace(".", "", 1).isdigit() else None
        sm = [num(r[2]) for r in use if num(r[2]) is not None]
        mx = [num(r[3]) for r in use if num(r[3]) is not None]
        reasons = set()
        for r in use:
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"),
                                 r[6:10]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(use), "samples_in_region": len(first),
                "samples_in_timed_regions": len(inside),
                "window": "device-resident timed region + e2e timed region" if hasattr(self, "t1_first")
                          else "device-resident timed region"}


# --------------------------------------------------------------------------- CPU arm
def _cpu_band(seed, j0, j1, ny=721, nx=1440):
    """One task of the CPU arm: rows j0..j1 of a global 0.25 degree timestep through the oracle port of the
    reference path, on one host core.  Returns (pid, seconds in the reference path, columns, n_iter); the
    synthetic band is generated outside the timed part (it stands in for reading the file)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import torch
    torch.set_num_threads(1)
    from pgw4era5_b200 import synthetic as S
    from oracle import pgw_oracle as O
    lat = np.linspace(-90.0, 90.0, ny)[j0:j1]
    era = S.make_era5(j1 - j0, nx, seed, lat=lat, lon=np.arange(nx) * (360.0 / nx))
    deltas = S.make_deltas(era, seed)
    e, d = S.to_numpy(era), S.to_numpy(deltas)
    t0 = time.perf_counter()
    out = O.pgw_for_era5(e, d, datetime(2006, 8, 2, 6), ignore_top_pressure_error=True)
    return os.getpid(), time.perf_counter() - t0, (j1 - j0) * nx, out["n_iter"]


def cpu_arm(procs, rows_total, band_rows=8, seed0=1000):
    """`rows_total` rows of the global grid (bands of `band_rows` x 1440 columns taken evenly from pole to pole),
    one band per task, spread over `procs` worker processes by the package's IterMP -- the same interface and
    the same one-task-per-file scheme as the reference's parallel.IterMP (parallel.py:36-68; /root/reference
    itself does not exist on the GPU box).  The time of a step is the largest per-worker sum of the seconds
    spent inside the reference path.  Returns (timesteps/s, seconds, columns)."""
    from pgw4era5_b200.parallel import IterMP
    ny = GRIDS["GL"][0]
    nb = max(1, rows_total // band_rows)
    starts = np.linspace(0, ny - band_rows, nb).astype(int)
    step_args = [dict(seed=seed0 + i, j0=int(j), j1=int(j) + band_rows) for i, j in enumerate(starts)]
    os.environ["PGW_ITERMP_NO_GPU"] = "1"           # CPU workers: no CUDA context per process
    try:
        pool = IterMP(njobs=procs, run_async=True, start_method="fork", quiet=True)
        pool.run(_cpu_band, fargs={}, step_args=step_args)
    finally:
        os.environ.pop("PGW_ITERMP_NO_GPU", None)
    per_pid = {}
    for pid, sec, cols, _ in pool.output:
        per_pid[pid] = per_pid.get(pid, 0.0) + sec
    wall = max(per_pid.values())
    cols = sum(r[2] for r in pool.output)
    return cols / float(GRIDS["GL"][0] * GRIDS["GL"][1]) / wall, wall, cols


def _cpu_sample_text(procs, cols, wall):
    return ("%d columns = %.3f of one global 721x1440x137 timestep per step, in bands of 8x1440 columns, one band "
            "per task over %d worker processes driven by pgw4era5_b200.parallel.IterMP (the reference's "
            "parallel.IterMP interface, parallel.py:36-68; /root/reference is absent on the GPU box); fp64 "
            "oracle port of the reference path (numpy + C column loops; the verbatim reference needs xarray, "
            "absent in this image); %.1f s per step" % (cols, cols / 1038240.0, procs, wall))


def run_reference(a):
    """--impl reference: the reference path's CPU implementation (oracle port) on all host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import build as ob
    ob.build()
    procs = min(max(1, os.cpu_count() or 1), 64)
    steps = max(1, a.steps)
    # bounded sample: a calibration step of one band per worker sizes the rows per step so that the whole
    # --steps/--warmup run stays within about three minutes; at most one whole global timestep per step
    t_cal = time.perf_counter()
    _, w_cal, c_cal = cpu_arm(procs, 8 * procs)
    t_cal = time.perf_counter() - t_cal
    budget = 100.0 / (steps + max(a.warmup, 0))
    rows = int(8 * procs * max(1.0, (budget - 1.0) / max(t_cal, 1e-3)))
    rows = max(8 * procs, min(rows // 8 * 8, 720))
    vals, walls, cols = [], [], 0
    for i in range(max(a.warmup, 0) + steps):
        v, w, cols = cpu_arm(procs, rows, seed0=2000 + 100 * i)
        if i >= max(a.warmup, 0):
            vals.append(v); walls.append(w)
    value = float(np.mean(vals))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "timesteps/s", "n_gpus": a.gpus,
        "steps": steps, "warmup": a.warmup, "ms_per_step": 1000.0 * float(np.mean(walls)),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "global 721x1440x137 single timestep, plev19 monthly deltas (BASELINE configs[1])",
                   "sampled_fraction_of_timestep": cols / 1038240.0},
        "cpu_baseline": {"value": value, "unit": "timesteps/s", "cores": procs, "kind": "port",
                         "sample": _cpu_sample_text(procs, cols, float(np.mean(walls)))},
        "e2e": {"value": value, "unit": "timesteps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------- GPU arm
def bare_link_test(dev, nbytes, world, barrier, reps=3):
    """Bare pinned-memory copies of the e2e step's sizes, H2D and D2H at the same time on two streams, on all
    ranks at once: the bound the platform sets for the host-buffer pipeline.  Returns GB/s per direction of
    this rank (bytes / time for one direction while the other runs)."""
    import torch
    n = nbytes // 4
    h_in = torch.empty(n, dtype=torch.float32, pin_memory=True)
    h_out = torch.empty(n, dtype=torch.float32, pin_memory=True)
    d_in = torch.empty(n, device=dev, dtype=torch.float32)
    d_out = torch.empty(n, device=dev, dtype=torch.float32)
    h_in.zero_(); h_out.zero_()
    s1, s2 = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)

    def both():
        with torch.cuda.stream(s1):
            d_in.copy_(h_in, non_blocking=True)
        with torch.cuda.stream(s2):
            h_out.copy_(d_out, non_blocking=True)
    both()
    torch.cuda.synchronize()
    barrier()
    t0 = time.perf_counter()
    for _ in range(reps):
        both()
    torch.cuda.synchronize()
    el = (time.perf_counter() - t0) / reps
    del h_in, h_out, d_in, d_out
    return nbytes / el / 1e9


def latband_leg(a, dev, rank, world, barrier):
    """Latitude-band mode on BASELINE configs[4]: ONE global snapshot (plev37 deltas, threshold 1e-3, the worst
    case iteration count), rows split over the ranks.  The stopping rule is field-global, so every snapshot
    costs one all-reduce (MAX over the packed status block) between the column kernel and finalize.  Snapshots
    are submitted back to back without host synchronisation; parity: each band against the same rows of a
    whole-grid run on this GPU (bit-identical fields and the same iteration count expected)."""
    import torch
    import torch.distributed as dist
    from pgw4era5_b200 import parallel as P, settings, synthetic as S
    from pgw4era5_b200.engine import DeltaSet, PGWEngine
    ny, nx = GRIDS[a.grid]
    old = settings.thresh_phi_ref_max_error
    settings.thresh_phi_ref_max_error = 1e-3
    try:
        era = S.make_era5(ny, nx, 5, device=dev, orog_seed=5)
        deltas = S.make_deltas(era, 5, plev=S.PLEV37, device=dev)
        when = datetime(2006, 8, 2, 6)
        whole = PGWEngine(era["ak"], era["bk"], DeltaSet(deltas, device=dev), soil1=era["soil1"])
        ref = whole.apply(era, when, ignore_top_pressure_error=True)
        r0, r1 = P.split_rows(ny, world)[rank]
        sub = {k: (v[..., r0:r1, :].contiguous() if isinstance(v, torch.Tensor) and v.dim() >= 3 else v)
               for k, v in era.items()}
        subd = {k: dict(v, data=v["data"][..., r0:r1, :].contiguous()) for k, v in deltas.items()}
        band_ds = DeltaSet(subd, device=dev)
        nslot = 4
        outs = None

        def measure(mode):
            nonlocal outs
            eng = PGWEngine(era["ak"], era["bk"], band_ds, soil1=era["soil1"], group=dist.group.WORLD,
                            band_exchange=mode)
            if outs is None:
                outs = [eng.alloc_outputs(r1 - r0, nx, len(era["soil1"])) for _ in range(nslot)]
            res = eng.apply(sub, when, out=outs[0], ignore_top_pressure_error=True)
            same = {}
            for name in ("PS", "T", "QV", "U", "V", "T_SKIN"):
                g, w = res[name], ref[name][..., r0:r1, :]
                same[name] = float((g - w).abs().nan_to_num().max())
            ok = torch.tensor([float(res["n_iter"] == ref["n_iter"]), -max(same.values())], device=dev,
                              dtype=torch.float64)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
            for i in range(3):
                eng.apply(sub, when, out=outs[i % nslot], ignore_top_pressure_error=True)
            n_snap = a.latband_snapshots
            eng.kernel_events = []
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            pend = []
            for i in range(n_snap):
                pend.append(eng.submit(sub, when, out=outs[i % nslot], ignore_top_pressure_error=True, slot=i % nslot))
                if len(pend) >= nslot:
                    pend.pop(0).result()
            n_it = [p.result()["n_iter"] for p in pend]
            e1.record()
            torch.cuda.synchronize()
            k_ms = float(np.mean([x.elapsed_time(y) for x, y in eng.kernel_events]))
            eng.kernel_events = None
            t = torch.tensor([e0.elapsed_time(e1) / n_snap, k_ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return dict(exchange=eng.band_exchange, ms_per_snapshot=float(t[0]), band_kernels_ms=float(t[1]),
                        n_iter=int(n_it[-1]), identical=bool(ok[0].item() == 1.0), max_abs_diff=float(-ok[1].item()))
        first = measure("auto")                       # the fused peer-memory exchange where the platform allows it
        second = measure("nccl") if first["exchange"] == "p2p" else None
        out = {"workload": "one global %dx%dx137 snapshot, plev37 deltas, threshold 1e-3 (BASELINE configs[4]), "
                           "%d latitude bands" % (ny, nx, world),
               "ms_per_snapshot": first["ms_per_snapshot"], "snapshots": a.latband_snapshots, "n_iter": first["n_iter"],
               "n_iter_whole_grid": int(ref["n_iter"]), "n_iter_identical_on_all_bands": first["identical"],
               "band_vs_whole_grid_max_abs_diff": first["max_abs_diff"],
               "ms_per_snapshot_band_kernels_only": first["band_kernels_ms"],
               "exchange": ("pgw_band_exchange: one kernel over peer memory (NVLink) behind the column kernel, 100 "
                            "float64 stored into every peer's inbox, flag release / acquire at system scope"
                            if first["exchange"] == "p2p" else
                            "pack, 1 NCCL all-reduce(MAX) of 100 float64, unpack (no peer mapping on this platform)"),
               "what_remains": "the exchange is serial with the band kernel of the same snapshot: "
                               "ms_per_snapshot - band_kernels_only"}
        if second is not None:
            out["nccl_form_of_the_exchange"] = {"ms_per_snapshot": second["ms_per_snapshot"],
                                                "n_iter": second["n_iter"],
                                                "n_iter_identical_on_all_bands": second["identical"],
                                                "band_vs_whole_grid_max_abs_diff": second["max_abs_diff"]}
        return out
    finally:
        settings.thresh_phi_ref_max_error = old


def dump_outputs(out_dir, res):
    """Write the output dict of one timestep (`Pending.result()`) to `out_dir` as .npy files: the surface fields
    PS, T_SKIN, FR_SEA_ICE, delta_ps whole as float32 [lat, lon]; T_SO, T, QV, U, V as float32 [levels, columns]
    at DUMP_COLUMNS columns drawn once from a fixed seed (ascending flat lat * lon indices, the same for every
    run on the same grid); n_iter and phi_max_errors as float64.  About 40 MB on the global grid.
    Sea ice is undefined (NaN) over land, as in the ERA5 files and the reference's output: FR_SEA_ICE_defined
    is 1 where FR_SEA_ICE holds a value and 0 where the path returned NaN, which FR_SEA_ICE stores as 0, so
    that every file holds finite numbers.  A NaN anywhere else is a defect and is written as it is."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    ny, nx = res["PS"].shape[-2:]
    ncol = ny * nx
    cols = np.sort(np.random.default_rng(0).choice(ncol, min(DUMP_COLUMNS, ncol), replace=False))
    idx = torch.as_tensor(cols, device=res["PS"].device)
    arrays = {name: res[name].reshape(ny, nx) for name in ("PS", "T_SKIN", "FR_SEA_ICE", "delta_ps")}
    for name in ("T_SO", "T", "QV", "U", "V"):
        arrays[name] = res[name].reshape(res[name].shape[1], ncol).index_select(1, idx)
    for name, t in arrays.items():
        a = t.cpu().numpy().astype(np.float32)
        if name == "FR_SEA_ICE":
            defined = ~np.isnan(a)
            np.save(os.path.join(out_dir, "FR_SEA_ICE_defined.npy"), defined.astype(np.float32))
            a = np.where(defined, a, np.float32(0.0))
        np.save(os.path.join(out_dir, name + ".npy"), a)
    np.save(os.path.join(out_dir, "n_iter.npy"), np.array([res["n_iter"]], dtype=np.float64))
    np.save(os.path.join(out_dir, "phi_max_errors.npy"), np.array(res["phi_max_errors"], dtype=np.float64))


def run_ours(a):
    import torch
    import torch.distributed as dist
    from pgw4era5_b200 import settings, synthetic as S
    from pgw4era5_b200.engine import DeltaSet, PGWEngine
    from pgw4era5_b200 import parallel as P

    settings.i_debug = 0
    if os.environ.get("PGW_BENCH_P_REF"):        # tuning experiments only (changes the workload; not a bench line)
        settings.p_ref_inp = float(os.environ["PGW_BENCH_P_REF"])
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    from pgw4era5_b200.parallel import bind_to_gpu_numa
    numa = None if os.environ.get("PGW_NO_NUMA_BIND") else bind_to_gpu_numa(local)    # before any pinned allocation
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    ny, nx = GRIDS[a.grid]
    ncol = ny * nx
    plev = S.PLEV19

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- inputs: climatology generated on rank 0 and broadcast (the one collective of the path)
    era0 = S.make_era5(ny, nx, 2, device=dev, orog_seed=2)
    deltas = S.make_deltas(era0, 2 if rank == 0 else 99, plev=plev, device=dev)
    ds = DeltaSet(deltas, device=dev)
    del deltas
    bcast = None
    if world > 1:
        bcast = {}
        P.broadcast_deltas(ds, src=0, info=bcast)
        t = torch.tensor([bcast["ms"]], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        bcast["ms"] = float(t.item())
        bcast["gb_per_s"] = bcast["bytes"] / bcast["ms"] / 1e6
    eng = PGWEngine(era0["ak"], era0["bk"], ds, soil1=era0["soil1"])
    # ring members: same terrain as the climatology, different weather
    ring = [era0] + [S.make_era5(ny, nx, 100 * (rank + 1) + i, device=dev, orog_seed=2)
                     for i in range(1, a.ring)]
    nslot = max(2, a.inflight)
    outs = [eng.alloc_outputs(ny, nx, len(era0["soil1"])) for _ in range(nslot)]
    base = datetime(2006, 8, 1, 0)
    when = lambda i: base + timedelta(hours=6 * ((i * world + rank) % 124))

    streams = [torch.cuda.Stream(device=dev) for _ in range(a.streams)] if a.streams > 1 else None

    def run_steps(n, collect=None):
        """n timesteps, up to `nslot` in flight: the host checks the status of a timestep (iteration count,
        error bits; may trigger a rerun) while the next ones are already queued behind it.  With --streams S > 1
        consecutive timesteps alternate between S streams (slot i always on the same stream), so the last,
        partly filled wave of one timestep's column kernel overlaps the first wave of the next."""
        pend = []
        for i in range(n):
            if streams:
                with torch.cuda.stream(streams[(i % nslot) % a.streams]):
                    pend.append(eng.submit(ring[i % a.ring], when(i), out=outs[i % nslot],
                                           ignore_top_pressure_error=True, slot=i % nslot))
            else:
                pend.append(eng.submit(ring[i % a.ring], when(i), out=outs[i % nslot], ignore_top_pressure_error=True,
                                       slot=i % nslot))
            if len(pend) >= nslot:
                r = pend.pop(0).result()
                if collect is not None:
                    collect.append(r["n_iter"])
        last = pend[-1]
        for p in pend:
            r = p.result()
            if collect is not None:
                collect.append(r["n_iter"])
        return last

    # ---- warm-up
    run_steps(a.warmup)
    n_iters = []

    # ---- timed region: device-resident inputs -> device-resident outputs
    sampler = ClockSampler(list(range(world))) if rank == 0 else None
    eng.kernel_events = []
    launches0 = eng.stats["launches"]
    barrier()
    if sampler:
        sampler.mark_start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    if streams:
        for st in streams:
            st.wait_event(ev0)
    last = run_steps(a.steps, n_iters)
    if streams:
        for st in streams:
            torch.cuda.current_stream().wait_stream(st)
    ev1.record()
    import ctypes
    from pgw4era5_b200 import _native
    kernel_name = ("pgw_column_tma_kernel" if _native.lib.pgw_timestep_uses_tma(ctypes.byref(last.args)) == 1
                   else "pgw_column_kernel")
    barrier()
    if sampler:
        sampler.mark_stop()
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, last.result())        # before the legs below reuse the output buffers
    ms = ev0.elapsed_time(ev1)
    kernel_ms = [e0.elapsed_time(e1) for e0, e1 in eng.kernel_events]
    # time the GPU spent in the column kernel per launch: the union of the launches' intervals (with several
    # streams the last wave of one launch runs next to the first wave of the following one; summing the
    # individual durations would count that time twice)
    iv = sorted((ev0.elapsed_time(e0), ev0.elapsed_time(e1)) for e0, e1 in eng.kernel_events)
    busy, cur_a, cur_b = 0.0, None, None
    for x, y in iv:
        if cur_b is None or x > cur_b:
            busy += (cur_b - cur_a) if cur_b is not None else 0.0
            cur_a, cur_b = x, y
        else:
            cur_b = max(cur_b, y)
    busy += (cur_b - cur_a) if cur_b is not None else 0.0
    kernel_busy_ms = busy / max(1, len(iv))
    eng.kernel_events = None
    launches = eng.stats["launches"] - launches0
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    value = world * a.steps / (ms / 1000.0)
    # host time per submit: the same loop with nothing to wait for would take this long per step
    t0 = time.perf_counter()
    for i in range(50):
        eng._fill_args(ring[i % a.ring], when(i), outs[i % nslot], None, i % nslot)
    host_us_fill = (time.perf_counter() - t0) / 50 * 1e6
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    ps = [eng.submit(ring[i % a.ring], when(i), out=outs[i % nslot], ignore_top_pressure_error=True, slot=i % nslot)
          for i in range(nslot)]
    host_us_submit = (time.perf_counter() - t0) / nslot * 1e6
    [p.result() for p in ps]

    # ---- end to end through the public API with HOST buffers (pinned), copies inside the timing
    e2e = None
    if a.e2e_steps > 0:
        from pgw4era5_b200.hostpipe import HostPipeline
        ns = a.e2e_slots
        pipe = HostPipeline(eng, ny, nx, nslots=ns)
        hin = [pipe.pin_inputs(ring[i % a.ring]) for i in range(ns)]
        houts = [pipe.alloc_host_outputs() for _ in range(ns)]
        for i in range(ns):
            pipe.run(hin[i % ns], when(i), houts[i % ns], ignore_top_pressure_error=True)
        pipe.drain()
        barrier()
        t0 = time.perf_counter()
        for i in range(a.e2e_steps):
            pipe.run(hin[i % ns], when(i), houts[i % ns], ignore_top_pressure_error=True)
        pipe.drain()
        torch.cuda.synchronize()
        el = time.perf_counter() - t0
        t = torch.tensor([el], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_val = world * a.e2e_steps / float(t.item())
        if sampler:
            sampler.mark_stop()
        h2d_b, d2h_b = pipe.h2d_bytes, pipe.d2h_bytes
        del pipe, hin, houts
        # the platform's bound for this pipeline: bare pinned copies of the same sizes, both directions at once,
        # on all ranks at once
        link = bare_link_test(dev, h2d_b, world, barrier)
        t = torch.tensor([link], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
        link = float(t.item())
        per_rank_gbs = (e2e_val / world) * h2d_b / 1e9
        e2e = {"value": e2e_val, "unit": "timesteps/s",
               "h2d_bytes_per_step": h2d_b, "d2h_bytes_per_step": d2h_b,
               "steps": a.e2e_steps, "slots": ns,
               "link_bound": {"gb_per_s_per_direction_per_gpu": link,
                              "timesteps_per_s": world * link * 1e9 / h2d_b,
                              "how": "bare pinned H2D + D2H copies of the step's sizes, both directions at once on "
                                     "two streams, all %d ranks at the same time (min over ranks)" % world},
               "frac_of_link": per_rank_gbs / link if link else None}

    # ---- roofline of the dominant kernel (the fused column kernel)
    peak, peak_kind = measured_peak_gbs()
    abytes = algorithmic_bytes(ncol, 137, len(plev), len(era0["soil1"]))
    k_ms = float(kernel_busy_ms) if kernel_ms else None
    achieved = abytes / (k_ms / 1000.0) / 1e9 if k_ms else None
    traffic, traffic_source = None, None
    try:
        with open(os.path.join(ROOT, "profiles", "column_kernel_traffic.json")) as f:
            tj = json.load(f)
            traffic = tj.get("dram_bytes_per_launch")
            traffic_source = ("ncu --set full capture of this kernel on another B200 of the pool (%s), not "
                              "measured during this run" % tj.get("source", "profiles/"))
    except Exception:
        pass
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": (achieved / peak) if achieved else None, "traffic": traffic,
                "traffic_source": traffic_source,
                "kernel": kernel_name, "kernel_ms": k_ms,
                "kernel_ms_how": "CUDA events around every launch (init + column kernel) inside the timed region; "
                                 "union of the launches' intervals / launches (= the mean duration with one stream)",
                "kernel_ms_mean_of_launch_durations": float(np.mean(kernel_ms)) if kernel_ms else None,
                "algorithmic_bytes": abytes,
                "peak_kind": peak_kind,
                "frac_whole_step": abytes / (ms / a.steps / 1000.0) / 1e9 / peak}

    # ---- latitude-band mode (BASELINE configs[4]) where there is more than one GPU
    latband = None
    if world > 1 and a.grid == "GL" and not a.no_latband:
        ring.clear()
        outs.clear()
        torch.cuda.empty_cache()
        latband = latband_leg(a, dev, rank, world, barrier)

    # ---- CPU baseline on a bounded sample (rank 0, N = 1 only): all host cores, IterMP-driven
    cpu = None
    if rank == 0 and world == 1 and not a.no_cpu:
        from oracle import build as ob
        ob.build()
        procs = min(max(1, os.cpu_count() or 1), 64)
        cpu_arm(procs, 8 * procs)                                   # start-up costs out of the way
        rows = max(8 * procs, min(720, 8 * procs * 6))
        v, wall, cols = cpu_arm(procs, rows)
        cpu = {"value": v, "unit": "timesteps/s", "cores": procs, "kind": "port",
               "sample": _cpu_sample_text(procs, cols, wall)}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "timesteps/s", "n_gpus": world, "steps": a.steps,
            "warmup": a.warmup, "ms_per_step": ms / a.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32 storage; f64 geopotential/ps iteration", "data": "synthetic",
            "config": {"workload": ("global %dx%dx137 single timestep per step, plev19 monthly deltas "
                                    "(BASELINE configs[1]); N>1: timesteps sharded by rank (configs[2])" % (ny, nx))
                       if a.grid == "GL" else
                       ("European subdomain %dx%dx137 single timestep per step, plev19 monthly deltas "
                        "(BASELINE configs[0], not the metric's configuration)" % (ny, nx)),
                       "grid": a.grid, "ring": a.ring,
                       "l2": "inputs cycle through %d distinct 2.3 GB timesteps (>> 126 MB L2)" % a.ring,
                       "parallelism": "timestep-sharded x%d" % world, "numa_node": numa,
                       "timesteps_in_flight": nslot, "streams": a.streams,
                       "n_iter": {"min": int(min(n_iters)), "max": int(max(n_iters)), "steps": len(n_iters)},
                       "engine": dict(eng.stats),
                       "host_us_per_submit": host_us_submit, "host_us_fill_args": host_us_fill,
                       "broadcast_ms": bcast["ms"] if bcast else None, "broadcast": bcast,
                       "latband": latband},
            "e2e": e2e, "gpu_launches": launches, "roofline": roofline, "cpu_baseline": cpu,
            "clocks": sampler.summary() if sampler else None,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=400)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--grid", default="GL", choices=sorted(GRIDS))
    ap.add_argument("--ring", type=int, default=4)
    ap.add_argument("--e2e-steps", type=int, default=48)
    ap.add_argument("--e2e-slots", type=int, default=2, help="timesteps in flight in the host-buffer pipeline")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--inflight", type=int, default=4, help="timesteps queued before the host checks the oldest")
    ap.add_argument("--streams", type=int, default=2, help="CUDA streams the timesteps alternate between")
    ap.add_argument("--no-latband", action="store_true")
    ap.add_argument("--latband-snapshots", type=int, default=100)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned (rank 0) to DIR as .npy files")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    a.warmup = max(a.warmup, 3) if a.impl == "ours" else a.warmup
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)


if __name__ == "__main__":
    main()

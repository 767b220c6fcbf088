"""
Cost of i_reinterp = 1 (the ERA state re-interpolated onto every iteration's pressures, step_03_apply_to_era.py:
202-216, :330-343) next to the default setting, on the global 721 x 1440 x 137 grid with plev19 deltas (BASELINE
configs[1]), one GPU, in one process:

  (a) default setting, PGWEngine.submit (TMA flavour of the column kernel)
  (b) default setting with PGW_COLUMN_PATH=generic (cp.async flavour, what (c) builds on)
  (c) i_reinterp = 1 through PGWEngine.submit (cp.async flavour with PGW_FLAG_REINTERP)
  (d) i_reinterp = 1 through PGWEngine.apply, i.e. the staged path (a few steps only)

    python tests/bench_reinterp.py --steps 20 --warmup 3 --out profiles/r3_reinterp.json

Inputs cycle through a ring of distinct device-resident timesteps (2.3 GB each, >> 126 MB L2) as in bench.py;
every leg uses a fresh engine, two timesteps in flight, and CUDA events around the timed steps.  Also reported:
iteration counts, reruns, replays (finalize relaunching the column kernel for N < k_spec), max |dps|, and in
how many columns the lowest level's final target lies two or more ERA levels away from its own.
"""
import argparse
import json
import os
import subprocess
import sys
from datetime import datetime, timedelta

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))


def gpu_info(idx):
    info = dict(name=torch.cuda.get_device_name(idx))
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(idx), "--query-gpu=power.limit,clocks.max.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["clocks_max_sm"] = [x.strip() for x in q.split(",")]
    except Exception as e:                  # the timings stand without it; say why it is missing
        info["power_limit"] = "not read: %r" % (e,)
    return info


def moved_levels(eng, era, res):
    """Per timestep: max |dps|, the number of columns with 2 or more ERA levels between the lowest level's final
    target and its own ERA level (dps < 0), and the number whose target lies below ERA level L-1 (dps > 0:
    constant extrapolation)."""
    PS = era["PS"].reshape(-1).double()
    ps = res["PS"].reshape(-1).double()
    akm, bkm = eng.akm_d, eng.bkm_d
    pe_low = akm[-1] + PS * bkm[-1]
    pt_low = akm[-1] + ps * bkm[-1]
    n = torch.zeros_like(PS, dtype=torch.int32)
    for l in range(len(akm) - 1):                         # ERA levels strictly between target and own level
        pe = akm[l] + PS * bkm[l]
        n += ((pe > torch.minimum(pt_low, pe_low)) & (pe < torch.maximum(pt_low, pe_low))).int()
    below = pt_low > pe_low
    return float((ps - PS).abs().max()), int((n >= 2).sum()), int(below.sum())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--staged-steps", type=int, default=2)
    ap.add_argument("--ring", type=int, default=4)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_reinterp.py measures on the GPU; no CUDA device found")
    from pgw4era5_b200 import settings, synthetic as S
    from pgw4era5_b200.engine import DeltaSet, PGWEngine
    settings.i_debug = 0
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    ny, nx = 721, 1440
    era0 = S.make_era5(ny, nx, 2, device=dev, orog_seed=2)
    ds = DeltaSet(S.make_deltas(era0, 2, plev=S.PLEV19, device=dev), device=dev)
    ring = [era0] + [S.make_era5(ny, nx, 100 + i, device=dev, orog_seed=2) for i in range(1, a.ring)]
    base = datetime(2006, 8, 1, 0)
    when = lambda i: base + timedelta(hours=6 * (i % 124))

    def engine():
        return PGWEngine(era0["ak"], era0["bk"], ds, soil1=era0["soil1"])

    def leg(i_reinterp, column_path, steps, warmup):
        if column_path:
            os.environ["PGW_COLUMN_PATH"] = column_path
        else:
            os.environ.pop("PGW_COLUMN_PATH", None)
        settings.i_reinterp = i_reinterp
        eng = engine()
        outs = [eng.alloc_outputs(ny, nx, len(era0["soil1"])) for _ in range(2)]
        n_iter = []

        def run(n, collect):
            pend = []
            for i in range(n):
                pend.append(eng.submit(ring[i % a.ring], when(i), out=outs[i % 2], ignore_top_pressure_error=True,
                                       slot=i % 2))
                if len(pend) >= 2:
                    collect.append(pend.pop(0).result()["n_iter"])
            for p in pend:
                collect.append(p.result()["n_iter"])

        run(warmup, [])
        reruns_warm = eng.stats["reruns"]
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        run(steps, n_iter)
        e1.record()
        torch.cuda.synchronize()
        r = dict(ms_per_timestep=e0.elapsed_time(e1) / steps, steps=steps, warmup=warmup, n_iter=n_iter,
                 reruns_warmup=reruns_warm, reruns_timed=eng.stats["reruns"] - reruns_warm,
                 rewrites=eng.stats["rewrites"], ps_bound=eng.ps_bound)
        if i_reinterp:
            r["max_abs_dps"], r["columns_moved_2_or_more_levels"], r["columns_below_level_L-1"] = [], [], []
            for i, era in enumerate(ring):
                res = eng.submit(era, when(i), out=outs[0], ignore_top_pressure_error=True).result()
                for k, v in zip(("max_abs_dps", "columns_moved_2_or_more_levels", "columns_below_level_L-1"),
                                moved_levels(eng, era, res)):
                    r[k].append(v)
            r["replays"] = eng.stats["rewrites"]
        return r, eng

    out = dict(workload="global %dx%dx137 single timestep, plev19 monthly deltas (BASELINE configs[1]), "
                        "ring of %d resident timesteps, 2 in flight" % (ny, nx, a.ring),
               gpu=gpu_info(0))
    out["a_default_tma"], _ = leg(0, None, a.steps, a.warmup)
    out["b_default_generic"], _ = leg(0, "generic", a.steps, a.warmup)
    out["c_reinterp_submit"], eng_c = leg(1, None, a.steps, a.warmup)
    os.environ.pop("PGW_COLUMN_PATH", None)

    # (d) the staged path: synchronous, float64 temporaries, one host synchronisation per iteration
    settings.i_reinterp = 1
    eng_d = engine()
    res_d = eng_d.apply(ring[0], when(0), ignore_top_pressure_error=True)
    times = []
    for i in range(a.staged_steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        r = eng_d.apply(ring[i % a.ring], when(i), ignore_top_pressure_error=True)
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1))
    out["d_reinterp_staged"] = dict(ms_per_timestep=float(np.mean(times)), ms=times, steps=a.staged_steps,
                                     warmup=1, n_iter=int(r["n_iter"]))
    # (c) and (d) on the same timestep: same N, fields within the parity tolerances
    res_c = eng_c.submit(ring[0], when(0), ignore_top_pressure_error=True).result()
    out["c_vs_d_ring0"] = dict(
        n_iter=[int(res_c["n_iter"]), int(res_d["n_iter"])],
        **{"max_abs_" + k: float((res_c[k].double() - res_d[k].double()).abs().max())
           for k in ("PS", "T", "QV", "U", "V")})
    c, b, d = (out[k]["ms_per_timestep"] for k in ("c_reinterp_submit", "b_default_generic", "d_reinterp_staged"))
    out["ratios"] = dict(c_over_b=c / b, d_over_c=d / c)
    text = json.dumps(out, indent=1)
    print(text, flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()

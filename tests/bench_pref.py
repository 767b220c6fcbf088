"""
Cost of p_ref_inp = None (the reference pressure picked per column and iteration, step_03_apply_to_era.py:219-251)
next to the default scalar p_ref, on the global 721 x 1440 x 137 grid with plev19 deltas (BASELINE configs[1]),
one GPU, in one process:

  (a) default setting, PGWEngine.submit (TMA flavour of the column kernel)
  (b) default setting with PGW_COLUMN_PATH=generic (cp.async flavour, what (c) builds on)
  (c) p_ref_inp = None through PGWEngine.submit (cp.async flavour with PGW_FLAG_LOCAL_PREF)
  (d) p_ref_inp = None through PGWEngine.apply, i.e. the staged path (a few steps only)

    python tests/bench_pref.py --steps 20 --warmup 3 --out profiles/r3_pref.json

Inputs cycle through a ring of distinct device-resident timesteps (2.3 GB each, >> 126 MB L2) as in bench.py;
every leg uses a fresh engine, two timesteps in flight, and CUDA events around the timed steps.  Also reported:
iteration counts, reruns (ps_bound / p_floor), and in how many columns p_ref at iteration N differs from the
first iteration's choice.
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


def first_choice(ps, plev):
    """p_ref of the first iteration (dps = 0): the first zg level, in file order, below 0.95 PS."""
    pe = 0.95 * ps.reshape(-1).double()
    out = torch.full_like(pe, float("nan"))
    for p in reversed([float(x) for x in plev]):       # the first qualifying level in file order wins
        out = torch.where(pe > p, torch.full_like(pe, p), out)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--staged-steps", type=int, default=2)
    ap.add_argument("--ring", type=int, default=4)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_pref.py measures on the GPU; no CUDA device found")
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
    plev_zg = ds.vars["zg"]["plev"]

    def engine():
        return PGWEngine(era0["ak"], era0["bk"], ds, soil1=era0["soil1"])

    def leg(p_ref_inp, column_path, steps, warmup):
        if column_path:
            os.environ["PGW_COLUMN_PATH"] = column_path
        else:
            os.environ.pop("PGW_COLUMN_PATH", None)
        settings.p_ref_inp = p_ref_inp
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
        if p_ref_inp is None:
            r["p_floor"] = eng.p_floor
            moved = []
            for i, era in enumerate(ring):
                res = eng.submit(era, when(i), out=outs[0], ignore_top_pressure_error=True).result()
                p1 = first_choice(era["PS"], plev_zg)
                moved.append(int((res["p_ref"].reshape(-1) != p1).sum()))
            r["columns_p_ref_changed_after_iteration_1"] = moved
        return r, eng

    out = dict(workload="global %dx%dx137 single timestep, plev19 monthly deltas (BASELINE configs[1]), "
                        "ring of %d resident timesteps, 2 in flight" % (ny, nx, a.ring),
               gpu=gpu_info(0))
    out["a_default_tma"], _ = leg(30000, None, a.steps, a.warmup)
    out["b_default_generic"], _ = leg(30000, "generic", a.steps, a.warmup)
    out["c_pref_none_submit"], eng_c = leg(None, None, a.steps, a.warmup)
    os.environ.pop("PGW_COLUMN_PATH", None)

    # (d) the staged path: synchronous, float64 temporaries, one host synchronisation per iteration
    settings.p_ref_inp = None
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
    out["d_pref_none_staged"] = dict(ms_per_timestep=float(np.mean(times)), ms=times, steps=a.staged_steps,
                                     warmup=1, n_iter=int(r["n_iter"]))
    # (c) and (d) on the same timestep: same N and p_ref, fields within the parity tolerances
    res_c = eng_c.submit(ring[0], when(0), ignore_top_pressure_error=True).result()
    out["c_vs_d_ring0"] = dict(
        n_iter=[int(res_c["n_iter"]), int(res_d["n_iter"])],
        p_ref_mismatches=int((res_c["p_ref"] != res_d["p_ref"]).sum()),
        **{"max_abs_" + k: float((res_c[k].double() - res_d[k].double()).abs().max())
           for k in ("PS", "T", "QV", "U", "V")})
    c, b, d = (out[k]["ms_per_timestep"] for k in ("c_pref_none_submit", "b_default_generic", "d_pref_none_staged"))
    out["ratios"] = dict(c_over_b=c / b, d_over_c=d / c)
    text = json.dumps(out, indent=1)
    print(text, flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()

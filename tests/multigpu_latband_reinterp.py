"""
Latitude-band mode with i_reinterp = 1 on real GPUs (run under torchrun, one rank per GPU; not collected by
pytest):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 \
        --master-port 29513 tests/multigpu_latband_reinterp.py

Each rank runs its latitude band of one snapshot through a band-mode engine and the whole grid through a
single-GPU engine, both with fresh speculation state.  The columns are independent and the bands agree on the
field-global iteration count, so every band must equal the matching rows of the whole-grid result bit for bit.
The first snapshot speculates past N, so its outputs come from finalize's replay of the column kernel for the
merged N.  With more ranks than GPUs (e.g. 8 ranks on one GPU) the ranks share the devices, use gloo,
and the bands agree through the pack / all-reduce / unpack form of the exchange.
"""
import os
import sys

import torch
import torch.distributed as dist

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(HERE))

from cases import ERA_DATE, make_case  # noqa: E402

FIELDS = ("PS", "delta_ps", "T", "QV", "U", "V", "T_SKIN", "T_SO", "FR_SEA_ICE")


def main():
    from pgw4era5_b200 import parallel as P, settings
    from pgw4era5_b200.engine import DeltaSet, PGWEngine
    settings.i_debug = 0
    settings.i_reinterp = 1
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    shared = world > torch.cuda.device_count()
    local = int(os.environ["LOCAL_RANK"]) % torch.cuda.device_count()
    torch.cuda.set_device(local)
    if shared:
        dist.init_process_group("gloo")
    else:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ny, nx = 48, 96
    era, deltas = make_case(ny, nx, 3, region="GL")
    dev = {k: (v.cuda() if isinstance(v, torch.Tensor) else v) for k, v in era.items()}
    whole = PGWEngine(era["ak"], era["bk"], DeltaSet(deltas, device="cuda"), soil1=era["soil1"])
    ref = whole.submit(dev, ERA_DATE, ignore_top_pressure_error=True).result()
    r0, r1 = P.split_rows(ny, world)[rank]
    sub = {k: (v[..., r0:r1, :].contiguous() if isinstance(v, torch.Tensor) and v.dim() >= 3 else v)
           for k, v in dev.items()}
    subd = {k: dict(v, data=v["data"][..., r0:r1, :].contiguous()) for k, v in deltas.items()}
    for exchange in (("nccl",) if shared else ("p2p", "nccl")):
        eng = PGWEngine(era["ak"], era["bk"], DeltaSet(subd, device="cuda"), soil1=era["soil1"],
                        group=dist.group.WORLD, band_exchange="auto" if exchange == "p2p" else "nccl")
        for rep in range(3):
            res = eng.submit(sub, ERA_DATE, ignore_top_pressure_error=True).result()
            assert res["n_iter"] == ref["n_iter"], (rank, res["n_iter"], ref["n_iter"])
            assert res["phi_max_errors"] == ref["phi_max_errors"], rank
            if rep == 0:       # later snapshots speculate k_spec = N: exact hit instead of the replay
                for name in FIELDS:          # bit for bit; NaN (sea ice over land) must sit at the same points
                    g, r = res[name], ref[name][..., r0:r1, :]
                    assert torch.equal(g.isnan(), r.isnan()) and torch.equal(g.nan_to_num(), r.nan_to_num()), \
                        (rank, name)
            if rep == 0:
                assert eng.stats["rewrites"] == 1, (rank, eng.stats)
        print("rank %d rows %d..%d on cuda:%d, exchange %s: n_iter %d, band == whole grid bit for bit, stats %s"
              % (rank, r0, r1, local, eng.band_exchange, res["n_iter"], eng.stats), flush=True)
        dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()

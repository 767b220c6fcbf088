"""The streamed delta set (deltastream.StreamedDeltaSet) against a resident DeltaSet built from the same daily
climatology: every output bit for bit, NaN payloads included, through submit, HostPipeline, reruns, the staged
apply() and the command line.  The stamps are days of the leap year 2000, so 29 February is dropped."""
import os
from contextlib import contextmanager
from datetime import datetime, timedelta

import numpy as np
import pytest
import torch

from cases import make_case
from pgw4era5_b200 import settings, synthetic as S
from pgw4era5_b200.deltastream import StreamedDeltaSet
from pgw4era5_b200.engine import DeltaSet, PGWEngine

pytestmark = pytest.mark.gpu

OUT = ("PS", "delta_ps", "T", "QV", "U", "V", "T_SKIN", "T_SO", "FR_SEA_ICE")
DAY = np.timedelta64(86400 * 10 ** 9, "ns")


def _run(start, end, hours=3):
    out, t = [], start
    while t <= end:
        out.append(t)
        t += timedelta(hours=hours)
    return out


# exact hits at 12 UTC, the days around the dropped 29 February, and 31 December -> 1 January
DATES = _run(datetime(2000, 2, 27, 9), datetime(2000, 3, 2, 12)) + _run(datetime(2000, 12, 30, 21),
                                                                         datetime(2001, 1, 1, 18))


@contextmanager
def _settings(**kw):
    old = {k: getattr(settings, k) for k in kw}
    for k, v in kw.items():
        setattr(settings, k, v)
    try:
        yield
    finally:
        for k, v in old.items():
            setattr(settings, k, v)


def daily_case(ny, nx, seed=5):
    era, _ = make_case(ny, nx, seed)
    deltas = S.make_deltas(era, seed, ntime=366)
    stamps = np.datetime64("2000-01-01T12:00", "ns") + np.arange(366) * DAY
    for d in deltas.values():
        d["time"] = stamps
    return era, deltas


def _dev(era):
    return {k: (v.cuda() if isinstance(v, torch.Tensor) else v) for k, v in era.items()}


def _engine(era, ds, **kw):
    return PGWEngine(era["ak"], era["bk"], ds, soil1=era["soil1"], **kw)


def _bits(t):
    t = t.detach().reshape(-1)
    return t.view(torch.int64 if t.dtype == torch.float64 else torch.int32).cpu()


def assert_same(got, want, names=OUT):
    for name in names:
        assert torch.equal(_bits(got[name]), _bits(want[name])), name
    assert got["n_iter"] == want["n_iter"]


def _snap(res):
    return {k: (v.clone() if isinstance(v, torch.Tensor) else v) for k, v in res.items()}


def _submit_all(eng, era, dates, **kw):
    dev = _dev(era)
    return [_snap(eng.submit(dev, when, ignore_top_pressure_error=True, **kw).result()) for when in dates]


SETTINGS = {"default": {}, "p_ref_inp=None": dict(p_ref_inp=None), "i_reinterp=1": dict(i_reinterp=1),
            "i_reference_dtypes=1": dict(i_reference_dtypes=1)}


@pytest.mark.parametrize("grid", [(8, 16), (7, 13)], ids=["tma", "cp_async"])
@pytest.mark.parametrize("slots", [2, 4])
@pytest.mark.parametrize("setting", list(SETTINGS))
def test_submit_matches_resident(grid, slots, setting):
    era, deltas = daily_case(*grid)
    names = OUT + (("p_ref",) if setting == "p_ref_inp=None" else ())
    with _settings(**SETTINGS[setting]):
        want = _submit_all(_engine(era, DeltaSet(deltas)), era, DATES)
        ds = StreamedDeltaSet(deltas, slots=slots)
        got = _submit_all(_engine(era, ds), era, DATES)
    for g, w in zip(got, want):
        assert_same(g, w, names)
    # 9 days of stamps (27 Feb .. 2 Mar without 29 Feb, 30 Dec .. 1 Jan): each loaded once
    assert ds.rings["d4"].loads == ds.rings["zg"].loads == 9


def _pipeline_all(ds, era, ny, nx):
    from pgw4era5_b200.hostpipe import HostPipeline
    pipe = HostPipeline(_engine(era, ds), ny, nx, nslots=2)
    h_in = pipe.pin_inputs(era)
    got = []
    for when in DATES:
        done = pipe.run(h_in, when, pipe.alloc_host_outputs(), ignore_top_pressure_error=True)
        if done is not None:
            got.append(done)
    return got + [d for d in pipe.drain() if d is not None]


def test_host_pipeline_matches_resident():
    """Two timesteps in flight on two streams, each new stamp evicting one the other stream may still read.  The
    reference is the same pipeline over a resident set: its k_spec schedule differs from one-at-a-time submits."""
    era, deltas = daily_case(8, 16)
    want = _pipeline_all(DeltaSet(deltas), era, 8, 16)
    got = _pipeline_all(StreamedDeltaSet(deltas, slots=2), era, 8, 16)
    assert len(got) == len(want) == len(DATES)
    for g, w in zip(got, want):
        for name in OUT:
            assert torch.equal(_bits(g[name]), _bits(w[name])), name
        assert g["n_iter"] == w["n_iter"]


def test_eviction_waits_for_the_timestep_that_reads_the_slot():
    """Timestep t is held back on its stream; t+1, on another stream, needs two other stamps and so evicts both
    of t's.  The loads must wait until t's kernels have read them."""
    era, deltas = daily_case(8, 16)
    t, t1 = datetime(2000, 3, 10, 6), datetime(2000, 6, 10, 6)
    want = _submit_all(_engine(era, DeltaSet(deltas)), era, [t, t1, t, t])[-1]      # the same k prediction
    eng = _engine(era, StreamedDeltaSet(deltas, slots=2))
    dev = _dev(era)
    _submit_all(eng, era, [t, t1])                         # warm up both workspaces and the engine's k prediction
    _submit_all(eng, era, [t])
    sa, sb = torch.cuda.Stream(), torch.cuda.Stream()
    torch.cuda.synchronize()
    with torch.cuda.stream(sa):
        torch.cuda._sleep(200_000_000)                      # ~0.1 s: a delay of t's column kernel, nothing else
        p = eng.submit(dev, t, ignore_top_pressure_error=True, slot=0)
    with torch.cuda.stream(sb):
        q = eng.submit(dev, t1, ignore_top_pressure_error=True, slot=1)
    b = eng.deltas.bracket("ta", t)
    assert b.ind_before not in eng.deltas.rings["d4"].keys and b.ind_after not in eng.deltas.rings["d4"].keys
    assert_same(_snap(p.result()), want)
    q.result()


@pytest.mark.parametrize("how", ["ps_bound", "k_spec"])
def test_rerun_after_eviction(how):
    era, deltas = daily_case(8, 16)
    t, t1 = datetime(2000, 3, 10, 6), datetime(2000, 6, 10, 6)
    kw = dict(ps_bound=float(era["PS"].min()) - 100.0) if how == "ps_bound" else {}
    sub = dict(k_spec=1) if how == "k_spec" else {}
    res = {}
    for name, ds in (("resident", DeltaSet(deltas)), ("streamed", StreamedDeltaSet(deltas, slots=2))):
        eng = _engine(era, ds, **kw)
        dev = _dev(era)
        p = eng.submit(dev, t, ignore_top_pressure_error=True, slot=0, **sub)
        q = eng.submit(dev, t1, ignore_top_pressure_error=True, slot=1, **sub)    # evicts t's stamps
        res[name] = (_snap(p.result()), _snap(q.result()), eng.stats["reruns"])
    assert res["streamed"][2] == res["resident"][2] >= 2
    assert_same(res["streamed"][0], res["resident"][0])
    assert_same(res["streamed"][1], res["resident"][1])


@pytest.mark.parametrize("setting", [dict(i_reinterp=1), dict(i_reinterp=1, p_ref_inp=None)])
def test_staged_apply_matches_resident(setting):
    era, deltas = daily_case(7, 13)
    dates = [datetime(2000, 2, 28, 18), datetime(2000, 3, 1, 12), datetime(2000, 12, 31, 21)]
    dev = _dev(era)
    with _settings(**setting):
        want = [_snap(_engine(era, DeltaSet(deltas)).apply(dev, d, ignore_top_pressure_error=True)) for d in dates]
        eng = _engine(era, StreamedDeltaSet(deltas, slots=2))
        got = [_snap(eng.apply(dev, d, ignore_top_pressure_error=True)) for d in dates]
    names = OUT + (("p_ref",) if "p_ref_inp" in setting else ())
    for g, w in zip(got, want):
        assert_same(g, w, names)


def test_latitude_bands_refuse_a_streamed_set():
    era, deltas = daily_case(7, 13)
    with pytest.raises(ValueError, match="latitude bands need a resident DeltaSet"):
        _engine(era, StreamedDeltaSet(deltas, slots=2), group=object())


@pytest.mark.parametrize("n", [1, 3, 4, 1001, 4099])
@pytest.mark.parametrize("swap", [0, 1])
@pytest.mark.parametrize("offset", [0, 1])
def test_pack_d4(n, swap, offset):
    import ctypes as C
    from pgw4era5_b200 import _native as N
    g = torch.Generator().manual_seed(n)
    words = torch.randint(-2 ** 31, 2 ** 31 - 1, (4, n + offset), generator=g, dtype=torch.int64).to(torch.int32)
    words[:, ::7] = torch.tensor([0x7FC00001, 0x7F800123, -0x5FFFEDD, 0x7FFFFFFF], dtype=torch.int32)[:, None]
    want = torch.stack([w[offset:] for w in words], dim=-1)
    src = words
    if swap:                                               # big-endian words as a NetCDF-3 record holds them
        src = torch.from_numpy(words.numpy().byteswap())
    src = src.cuda()
    ins = [C.c_void_p(src[j].data_ptr() + 4 * offset) for j in range(4)]
    out = torch.full((n, 4), -1, device="cuda", dtype=torch.int32)
    N.check(N.lib.pgw_pack_d4_f32(*ins, C.c_void_p(out.data_ptr()), n, swap,
                                  C.c_void_p(torch.cuda.current_stream().cuda_stream)), "pgw_pack_d4_f32")
    assert torch.equal(out.cpu(), want)


def test_cli_streams_daily_delta_files(tmp_path, monkeypatch):
    from test_cli_gpu import _write_deltas, _write_era
    from pgw4era5_b200 import deltastream, ncio
    from pgw4era5_b200 import step_03_apply_to_era as S3
    era, deltas = daily_case(10, 24)
    inp, dd = tmp_path / "in", tmp_path / "deltas"
    inp.mkdir(); dd.mkdir()
    dates = _run(datetime(2000, 2, 28, 6), datetime(2000, 3, 1, 18), hours=6)
    for when in dates:
        _write_era(str(inp / settings.era5_file_name_base.format(when)), era, when)
    _write_deltas(str(dd), deltas, era["lat"], era["lon"])
    files_3d = {os.path.realpath(deltastream.delta_file(str(dd), n)[0]) for n in ("ta", "hur", "ua", "va", "zg")}
    argv = lambda out: ["-i", str(inp), "-o", str(out), "-d", str(dd), "-f", dates[0].strftime("%Y%m%d%H"),
                        "-l", dates[-1].strftime("%Y%m%d%H"), "-H", "6", "-t"]
    with _settings(i_debug=0):
        monkeypatch.setattr(S3, "_ENGINES", {})
        S3.main(argv(tmp_path / "resident"))
        assert not getattr(next(iter(S3._ENGINES.values())).deltas, "streamed", False)

        load, open_dataset = S3.load_delta_set, ncio.open_dataset

        def no_3d(path, *a, **k):
            assert os.path.realpath(path) not in files_3d, path
            return open_dataset(path, *a, **k)
        monkeypatch.setattr(S3, "_ENGINES", {})
        monkeypatch.setattr(S3, "load_delta_set", lambda d, device="cuda": load(d, device, max_resident_bytes=0))
        monkeypatch.setattr(ncio, "open_dataset", no_3d)
        S3.main(argv(tmp_path / "streamed"))
        assert next(iter(S3._ENGINES.values())).deltas.streamed
    for when in dates:
        name = settings.era5_file_name_base.format(when)
        a, b = (tmp_path / "resident" / name).read_bytes(), (tmp_path / "streamed" / name).read_bytes()
        assert a == b, name

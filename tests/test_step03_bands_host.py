"""Latitude-band mode of step_03 without a GPU: row hyperslabs of NetCDF-3 files (nc3raw.RawNC3.read_rows /
write_rows) against scipy, the output file assembled from bands, the delta climatology by band, the command-line
refusals, and the host-side agreement of the ranks (gloo): a failure on one rank raises on every rank."""
import os
import socket
from datetime import datetime

import numpy as np
import pytest
import torch

from pgw4era5_b200 import ncio, settings
from pgw4era5_b200 import step_03_apply_to_era as S3
from pgw4era5_b200.nc3raw import RawNC3
from pgw4era5_b200.parallel import split_rows

NY, NX = 11, 6


def _scipy_file(path, version, nt=2):
    """A file with record and non-record variables of one to three axes in front of the rows."""
    from scipy.io import netcdf_file
    rng = np.random.default_rng(version)
    vals = dict(rec3=rng.normal(size=(nt, NY, NX)), rec4=rng.normal(size=(nt, 3, NY, NX)),
                fix2=rng.normal(size=(NY, NX)), fix4=rng.normal(size=(2, 3, NY, NX)))
    vals = {k: v.astype(np.float32) for k, v in vals.items()}
    with netcdf_file(path, "w", version=version) as f:
        f.createDimension("time", None); f.createDimension("lev", 3); f.createDimension("two", 2)
        f.createDimension("lat", NY); f.createDimension("lon", NX)
        t = f.createVariable("time", "d", ("time",)); t[:] = np.arange(nt, dtype=np.float64)
        f.createVariable("rec3", "f", ("time", "lat", "lon"))[:] = vals["rec3"]
        f.createVariable("rec4", "f", ("time", "lev", "lat", "lon"))[:] = vals["rec4"]
        f.createVariable("fix2", "f", ("lat", "lon"))[:] = vals["fix2"]
        f.createVariable("fix4", "f", ("two", "lev", "lat", "lon"))[:] = vals["fix4"]
    return vals


BANDS = [(0, 4), (4, 7), (7, 11), (5, 6), (0, 11), (10, 11)] + split_rows(NY, 3) + split_rows(NY, 4)


@pytest.mark.parametrize("version", [1, 2])
def test_read_rows_matches_scipy(tmp_path, version):
    path = str(tmp_path / "a.nc")
    vals = _scipy_file(path, version)
    raw = RawNC3(path)
    assert raw.version == version
    with open(path, "rb", buffering=0) as f:
        for name, want in vals.items():
            v = raw.vars[name]
            for r0, r1 in BANDS:
                for rec in range(raw.numrecs if v.is_record else 1):
                    whole = want[rec] if v.is_record else want
                    buf = np.empty(whole.shape[:-2] + (r1 - r0, NX), dtype=">f4")
                    raw.read_rows(f, name, buf, r0, r1, record=rec)
                    np.testing.assert_array_equal(buf.astype(np.float32), whole[..., r0:r1, :],
                                                  err_msg="%s %s %d" % (name, (r0, r1), rec))


@pytest.mark.parametrize("version", [1, 2])
def test_write_rows_matches_scipy(tmp_path, version):
    path = str(tmp_path / "b.nc")
    vals = _scipy_file(path, version)
    raw = RawNC3(path)
    want = {k: v.copy() for k, v in vals.items()}
    rng = np.random.default_rng(11)
    fd = os.open(path, os.O_RDWR)
    try:
        for name, (r0, r1) in zip(vals, [(0, 3), (3, 4), (8, 11), (2, 9)]):
            v = raw.vars[name]
            rec = 1 if v.is_record else 0
            shp = v.record_shape[:-2] + (r1 - r0, NX)
            new = rng.normal(size=shp).astype(np.float32)
            raw.write_rows(fd, name, new.astype(">f4"), r0, r1, record=rec)
            (want[name][rec] if v.is_record else want[name])[..., r0:r1, :] = new
    finally:
        os.close(fd)
    back = ncio.open_dataset(path)
    for name in vals:
        np.testing.assert_array_equal(back[name].data, want[name], err_msg=name)


def test_rows_are_checked(tmp_path):
    path = str(tmp_path / "c.nc")
    _scipy_file(path, 2)
    raw = RawNC3(path)
    with open(path, "rb", buffering=0) as f:
        with pytest.raises(ValueError):
            raw.read_rows(f, "rec4", np.empty((3, 2, NX), ">f4"), 0, 3)          # buffer of 2 rows for 3
        with pytest.raises(ValueError):
            raw.read_rows(f, "rec4", np.empty((3, 2, NX), ">f4"), 10, 12)        # beyond the last row
        with pytest.raises(ValueError):
            raw.read_rows(f, "rec4", np.empty((3, 0, NX), ">f4"), 4, 4)          # empty band
        with pytest.raises(IndexError):
            raw.read_rows(f, "rec3", np.empty((1, NX), ">f4"), 0, 1, record=2)
        with pytest.raises(ValueError):
            raw.read_rows(f, "time", np.empty(1, ">f8"), 0, 1)                   # no row axis


def _era_file(path, when, seed, ny=9, nx=8):
    from test_cli_gpu import _write_era
    from pgw4era5_b200 import synthetic as S
    _write_era(path, S.make_era5(ny, nx, seed), when)


def test_bands_written_into_the_prepared_file_equal_write_raw(tmp_path):
    """Rank 0's prepared file plus W bands of the eight fields = _write_raw of the whole grid, byte for byte."""
    ny, nx = 9, 8
    inp = str(tmp_path / "in.nc")
    _era_file(inp, datetime(2006, 8, 2, 0), 3, ny, nx)
    names = S3._ERA_NAMES(settings.var_name_map)
    raw = RawNC3(inp)
    rng = np.random.default_rng(4)
    whole = {k: torch.from_numpy(rng.normal(size=raw.vars[names[k]].shape).astype(">f4").view(np.float32))
             for k in S3._WRITTEN}
    S3._write_raw(raw, names, inp, str(tmp_path / "whole.nc"), whole)
    for world in (1, 2, 3, 4):
        out = str(tmp_path / ("bands%d.nc" % world))
        S3._write_raw(raw, names, inp, out, None)
        for r0, r1 in reversed(split_rows(ny, world)):
            band = {k: v[..., r0:r1, :].contiguous() for k, v in whole.items()}
            S3._write_band(raw, names, out, band, (r0, r1))
        assert (tmp_path / ("bands%d.nc" % world)).read_bytes() == (tmp_path / "whole.nc").read_bytes(), world


def test_band_layout_of_the_reader(tmp_path):
    ny, nx = 9, 8
    inp = str(tmp_path / "in.nc")
    _era_file(inp, datetime(2006, 8, 2, 0), 5, ny, nx)
    names = S3._ERA_NAMES(settings.var_name_map)
    lev = dict(T_SO=raw_len(inp, "soil1"), T=137, QV=137, U=137, V=137)
    band = lambda h, w=nx: {k: torch.empty((1, lev.get(k, 1), h, w), device="meta") for k in names}
    assert S3._raw_layout(inp, names, band(3), grid=(ny, nx)) is not None
    assert S3._raw_layout(inp, names, band(ny), grid=(ny, nx)) is not None
    assert S3._raw_layout(inp, names, band(3), grid=(ny + 1, nx)) is None     # another grid
    assert S3._raw_layout(inp, names, band(3, nx - 1), grid=(ny, nx - 1)) is None


def raw_len(path, dim):
    return RawNC3(path).dims[dim]


def _write_monthly_deltas(ddir, ny, nx, seed=8):
    from test_cli_gpu import _write_deltas
    from pgw4era5_b200 import synthetic as S
    era = S.make_era5(ny, nx, seed)
    deltas = S.make_deltas(era, seed)
    _write_deltas(ddir, deltas, era["lat"], era["lon"])
    return deltas


def test_band_delta_set_is_the_rows_of_the_whole(tmp_path, monkeypatch):
    """load_delta_set(rows=...) hands DeltaSet the rows of what the whole-file load hands it (the 3-D deltas read
    band by band from the NetCDF-3 files, the rest decoded and sliced), for NetCDF-3 and decoded 3-D files."""
    from pgw4era5_b200 import deltastream, engine
    ny, nx = 13, 10
    dd = tmp_path / "deltas"
    dd.mkdir()
    _write_monthly_deltas(str(dd), ny, nx)
    monkeypatch.setattr(engine, "DeltaSet", lambda deltas, device="cuda": deltas)
    whole = S3.load_delta_set(str(dd), device="cpu", max_resident_bytes=1 << 40)
    for heads in (True, False):
        if not heads:          # the decoding path for files that are not float32 NetCDF-3
            monkeypatch.setattr(deltastream, "read_3d_headers", lambda d: None)
        for r0, r1 in [(0, 4), (4, 9), (12, 13)]:
            band = S3.load_delta_set(str(dd), device="cpu", max_resident_bytes=1 << 40, rows=(r0, r1))
            assert set(band) == set(whole)
            for name, d in whole.items():
                np.testing.assert_array_equal(np.asarray(band[name]["time"]), np.asarray(d["time"]))
                if d["plev"] is None:
                    assert band[name]["plev"] is None
                else:
                    np.testing.assert_array_equal(band[name]["plev"], d["plev"])
                got = np.asarray(band[name]["data"])
                assert got.dtype.byteorder in "=|<" and got.flags.c_contiguous
                np.testing.assert_array_equal(got, np.asarray(d["data"])[..., r0:r1, :], err_msg=name)


def test_band_delta_set_too_large_names_the_ranks_that_fit(tmp_path):
    from pgw4era5_b200 import deltastream
    ny, nx = 16, 10
    dd = tmp_path / "deltas"
    dd.mkdir()
    _write_monthly_deltas(str(dd), ny, nx)
    need = deltastream.resident_bytes(deltastream.read_3d_headers(str(dd)))
    with pytest.raises(ValueError, match="4 ranks or more would fit"):
        S3.load_delta_set(str(dd), device="cpu", max_resident_bytes=need // 4, rows=(0, 8))
    with pytest.raises(ValueError, match="no number of ranks fits"):
        S3.load_delta_set(str(dd), device="cpu", max_resident_bytes=1, rows=(0, 1))


def test_decoded_band_delta_set_too_large_names_the_ranks_that_fit(tmp_path, monkeypatch):
    """Delta files that are not float32 NetCDF-3 are decoded whole and sliced; the band is sized from the decoded
    arrays before anything goes to the device, with the same message."""
    from pgw4era5_b200 import deltastream, engine
    ny, nx = 16, 10
    dd = tmp_path / "deltas"
    dd.mkdir()
    _write_monthly_deltas(str(dd), ny, nx)
    need = deltastream.resident_bytes(deltastream.read_3d_headers(str(dd)))
    monkeypatch.setattr(deltastream, "read_3d_headers", lambda d: None)
    monkeypatch.setattr(engine, "DeltaSet", lambda deltas, device="cuda": deltas)
    with pytest.raises(ValueError, match="4 ranks or more would fit"):
        S3.load_delta_set(str(dd), device="cpu", max_resident_bytes=need // 4, rows=(0, 8))
    band = S3.load_delta_set(str(dd), device="cpu", max_resident_bytes=need // 4, rows=(0, 4))
    assert band["ta"]["data"].shape[-2:] == (4, nx)


@pytest.mark.parametrize("extra, msg", [(["-p", "2"], "-p must be 1"), (["-D", "interpolate_full"], "debug modes"),
                                        ([], "environment of torchrun")])
def test_cli_refusals(tmp_path, monkeypatch, extra, msg):
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK"):
        monkeypatch.delenv(k, raising=False)
    if extra:
        monkeypatch.setenv("RANK", "0"); monkeypatch.setenv("WORLD_SIZE", "1"); monkeypatch.setenv("LOCAL_RANK", "0")
    with pytest.raises(ValueError, match=msg):
        S3.main(["-i", str(tmp_path), "-o", str(tmp_path / "out"), "-d", str(tmp_path), "-f", "2006080200",
                 "-l", "2006080200", "--latitude_bands"] + extra)
    assert not (tmp_path / "out").exists()          # refused before anything is created


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _steps(inp, out, whens):
    name = settings.era5_file_name_base.format
    return [dict(inp_era_file_path=os.path.join(inp, name(w)), out_era_file_path=os.path.join(out, name(w)),
                 era_step_dt=w) for w in whens]


def _band_worker(rank, world, port, tmp, case):
    import sys
    import traceback
    import torch.distributed as dist
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    settings.i_debug = -1
    whens = [datetime(2006, 8, 2, 0), datetime(2006, 8, 2, 6), datetime(2006, 8, 2, 12)]
    inp = os.path.join(tmp, "in_missing" if (case == "missing" and rank == 1) else "in")
    if case == "settings":
        settings.i_reference_output_dtypes = 1
    band = S3.Band(dist.group.WORLD, dist.group.WORLD)
    try:
        S3.pgw_for_era5_files(_steps(inp, os.path.join(tmp, "out"), whens), os.path.join(tmp, "deltas"), True,
                              band=band)
        res = "returned"
    except Exception as e:
        res = "%s: %s" % (type(e).__name__, e)
        if not isinstance(e, (ValueError, RuntimeError)):
            res += traceback.format_exc()
    with open(os.path.join(tmp, "rank%d.txt" % rank), "w") as f:
        f.write(res)
    dist.destroy_process_group()


def _band_case(tmp_path):
    import shutil
    inp, miss = tmp_path / "in", tmp_path / "in_missing"
    for p in (inp, miss, tmp_path / "out", tmp_path / "deltas"):
        p.mkdir()
    whens = [datetime(2006, 8, 2, 0), datetime(2006, 8, 2, 6), datetime(2006, 8, 2, 12)]
    for i, w in enumerate(whens):
        _era_file(os.path.join(str(inp), settings.era5_file_name_base.format(w)), w, 30 + i)
    for w in whens[:2]:                 # the third file is missing in this directory
        name = settings.era5_file_name_base.format(w)
        shutil.copy(str(inp / name), str(miss / name))
    _write_monthly_deltas(str(tmp_path / "deltas"), 9, 8)


@pytest.mark.timeout(240)
def test_a_missing_file_on_one_rank_raises_on_every_rank(tmp_path):
    """World 3 on gloo: rank 1 lacks the third input file.  Every rank raises at the start barrier -- rank 1 its own
    ValueError, ranks 0 and 2 a RuntimeError naming rank 1 -- and none is left waiting (mp.spawn returns)."""
    import torch.multiprocessing as mp
    _band_case(tmp_path)
    mp.spawn(_band_worker, args=(3, _free_port(), str(tmp_path), "missing"), nprocs=3, join=True)
    res = [(tmp_path / ("rank%d.txt" % r)).read_text() for r in range(3)]
    assert res[1].startswith("ValueError") and "2006080212" in res[1], res[1]
    for r in (0, 2):
        assert res[r].startswith("RuntimeError: latitude bands: rank(s) [1] failed while checking the input files"), \
            res[r]
    # rank 0 prepared the output files before the barrier; nobody wrote a band into them
    out = tmp_path / "out" / settings.era5_file_name_base.format(datetime(2006, 8, 2, 0))
    assert out.stat().st_size == (tmp_path / "in" / out.name).stat().st_size


@pytest.mark.timeout(240)
def test_settings_band_mode_cannot_run_raise_on_every_rank(tmp_path):
    import torch.multiprocessing as mp
    _band_case(tmp_path)
    mp.spawn(_band_worker, args=(2, _free_port(), str(tmp_path), "settings"), nprocs=2, join=True)
    for r in range(2):
        res = (tmp_path / ("rank%d.txt" % r)).read_text()
        assert res.startswith("ValueError: latitude bands write the input file's layout"), res
    assert not os.listdir(str(tmp_path / "out"))          # refused before any file was created


def test_band_start_reads_headers_and_level_tables_only(tmp_path, monkeypatch):
    """Before the pipeline a rank reads the headers and ak, bk, akm, bkm and the soil depths of the first file --
    no field is decoded (a global snapshot is 2.3 GB) -- and rank 0 prepares the output files."""
    import torch.distributed as dist
    from pgw4era5_b200 import ncio as N
    whens = [datetime(2006, 8, 2, 0), datetime(2006, 8, 2, 6)]
    (tmp_path / "in").mkdir(); (tmp_path / "out").mkdir()
    for i, w in enumerate(whens):
        _era_file(os.path.join(str(tmp_path / "in"), settings.era5_file_name_base.format(w)), w, 40 + i)
    steps = _steps(str(tmp_path / "in"), str(tmp_path / "out"), whens)
    want = N.open_dataset(steps[0]["inp_era_file_path"], decode_cf=False)

    def no_decoding(path, *a, **k):
        raise AssertionError("decoded %s" % path)
    monkeypatch.setattr(N, "open_dataset", no_decoding)
    dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%d" % _free_port(), rank=0, world_size=1)
    try:
        names = S3._ERA_NAMES(settings.var_name_map)
        first, grid, rows = S3._band_start(steps, names, S3.Band(dist.group.WORLD, dist.group.WORLD))
    finally:
        dist.destroy_process_group()
    assert grid == (9, 8) and rows == (0, 9)
    for name in ("ak", "bk", settings.SOIL_HLEV_ERA):
        np.testing.assert_array_equal(first[name].data, want[name].data)
    assert set(first.keys()) <= {"ak", "bk", "akm", "bkm", settings.SOIL_HLEV_ERA}
    for st in steps:
        assert os.path.getsize(st["out_era_file_path"]) == os.path.getsize(st["inp_era_file_path"])

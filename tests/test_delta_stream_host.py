"""The host side of the streamed delta set, without a GPU: which file record a bracket needs, the slot a
load evicts, the resident/streamed decision from the delta file headers, and the shared validation."""
import os
from datetime import datetime

import numpy as np
import pytest
import torch

from pgw4era5_b200 import deltastream as D
from pgw4era5_b200 import ncio, settings, timeinterp
from pgw4era5_b200.engine import VARS_2D, VARS_3D, DeltaSet, read_axes

DAY = np.timedelta64(86400 * 10 ** 9, "ns")


def daily_2000():
    """366 daily stamps at 12 UTC of the leap year 2000."""
    return np.datetime64("2000-01-01T12:00", "ns") + np.arange(366) * DAY


def needed_records(stamps, when):
    """The source entries of the two stamps that bracket ``when``."""
    kept, keep, _ = read_axes("ta", dict(time=stamps))
    b = timeinterp.bracket(kept, when)
    return D.stamp_record(keep, b.ind_before), D.stamp_record(keep, b.ind_after)


@pytest.mark.parametrize("when, records", [
    (datetime(2000, 1, 10, 12), (9, 9)),                 # exact hit
    (datetime(2000, 2, 28, 18), (58, 60)),               # 28 Feb -> 1 Mar: record 59 (29 Feb) is dropped
    (datetime(2000, 3, 1, 0), (58, 60)),
    (datetime(2000, 3, 1, 15), (60, 61)),                # after the leap day every record is one further on
    (datetime(2000, 12, 31, 15), (365, 0)),              # 31 Dec -> 1 Jan of the next year
    (datetime(2001, 1, 1, 3), (365, 0)),                 # before the first stamp: the wrap to the last one
    (datetime(2001, 3, 1, 6), (58, 60)),                 # a year without 29 Feb reads the same records
])
def test_records_across_leap_day_and_year_wrap(when, records):
    assert needed_records(daily_2000(), when) == records


def test_records_without_leap_day():
    stamps = np.datetime64("2001-01-01T12:00", "ns") + np.arange(365) * DAY
    assert needed_records(stamps, datetime(2001, 3, 1, 0)) == (58, 59)
    assert needed_records(stamps, datetime(2001, 1, 1, 0)) == (364, 0)


def test_lru_slot_choice():
    assert D.choose_slot([3, None, 5, 7], [4, 0, 2, 3], busy=set()) == 1             # an empty slot first
    assert D.choose_slot([3, 4, 5, 7], [4, 1, 2, 3], busy=set()) == 1                # else the least recently used
    assert D.choose_slot([3, 4, 5, 7], [4, 1, 2, 3], busy={1}) == 2                  # ... that is not in use
    with pytest.raises(RuntimeError, match="every slot of the delta ring is in use"):
        D.choose_slot([3, 4], [4, 1], busy={0, 1})


def _write(ddir, ny=3, nx=5, ntime=366, K=4, Kz=None, dtype=np.float32):
    """Delta files as step_02 writes them: (time, plev, lat, lon), time as the record dimension."""
    rng = np.random.default_rng(0)
    stamps = daily_2000()[:ntime]
    plev = np.array([100000.0, 85000.0, 50000.0, 20000.0])[:K]
    for name in VARS_3D + VARS_2D:
        path, var = D.delta_file(ddir, name)
        ds = ncio.Dataset()
        ds["time"] = ncio.encode_time(stamps, "days since 1850-01-01 00:00:00")
        if name in VARS_3D:
            k = Kz if (name == "zg" and Kz) else K
            ds["plev"] = ncio.Variable(("plev",), plev[:k])
            ds[var] = ncio.Variable(("time", "plev", "lat", "lon"), rng.standard_normal((ntime, k, ny, nx)).astype(dtype))
        else:
            ds[var] = ncio.Variable(("time", "lat", "lon"), rng.standard_normal((ntime, ny, nx)).astype(np.float32))
        ds.to_netcdf(path)
    return stamps, plev


def test_decision_from_headers(tmp_path):
    ny, nx, K, Kz = 3, 5, 4, 3
    _write(str(tmp_path), ny, nx, K=K, Kz=Kz)
    h = D.read_3d_headers(str(tmp_path))
    assert sorted(h) == sorted(VARS_3D)
    assert len(h["ta"][2]["time"]) == 366 and list(h["zg"][2]["plev"]) == [100000.0, 85000.0, 50000.0]
    ncol, nt = ny * nx, 365                                        # 29 February is not resident
    arena = 4 * ncol * (4 * nt * K + nt * Kz + 6 * nt)
    staged = 4 * 366 * K * ncol                                    # one variable as the constructor stages it
    assert D.resident_bytes(h) == arena + staged
    assert not D.should_stream(h, "cpu", max_resident_bytes=arena + staged)
    assert D.should_stream(h, "cpu", max_resident_bytes=arena + staged - 1)


def test_non_netcdf3_takes_the_resident_path(tmp_path):
    _write(str(tmp_path))
    path, _ = D.delta_file(str(tmp_path), "hur")
    with open(path, "wb") as f:                                    # a NetCDF-4 (HDF5) file begins like this
        f.write(b"\x89HDF\r\n\x1a\n" + bytes(64))
    assert D.read_3d_headers(str(tmp_path)) is None
    assert not D.should_stream(None, "cpu", max_resident_bytes=0)


def test_float64_deltas_take_the_resident_path(tmp_path):
    _write(str(tmp_path), dtype=np.float64)
    assert D.read_3d_headers(str(tmp_path)) is None


def test_read_stamp_of_record_and_fixed_variables(tmp_path):
    from pgw4era5_b200.nc3raw import RawNC3
    a = np.arange(5 * 2 * 3, dtype=np.float32).reshape(5, 2, 3)
    ds = ncio.Dataset()
    ds["time"] = ncio.Variable(("time",), np.arange(5.0))
    ds["rec"] = ncio.Variable(("time", "y", "x"), a)
    ds["fixed"] = ncio.Variable(("t2", "y", "x"), a + 100)          # the stamp axis is not the record dimension
    path = str(tmp_path / "f.nc")
    ds.to_netcdf(path)
    raw = RawNC3(path)
    assert raw.vars["rec"].is_record and not raw.vars["fixed"].is_record
    buf = np.empty(6, dtype=">f4")
    with open(path, "rb", buffering=0) as f:
        for i in (0, 3, 4):
            raw.read_stamp(f, "rec", buf, i)
            assert np.array_equal(buf.astype(np.float32), a[i].ravel())
            raw.read_stamp(f, "fixed", buf, i)
            assert np.array_equal(buf.astype(np.float32), a[i].ravel() + 100)
        with pytest.raises(ValueError):
            raw.read_stamp(f, "fixed", buf, 5)


def _deltas(ntime=6, K=3, ny=2, nx=3):
    stamps = daily_2000()[:ntime]
    plev = np.array([100000.0, 85000.0, 50000.0])[:K]
    d3 = lambda: dict(time=stamps, plev=plev.copy(), data=torch.zeros(ntime, K, ny, nx))
    d2 = lambda: dict(time=stamps, plev=None, data=torch.zeros(ntime, ny, nx))
    return {**{n: d3() for n in VARS_3D}, **{n: d2() for n in VARS_2D}}


@pytest.mark.parametrize("edit, message", [
    (lambda d: d["hur"].update(plev=d["hur"]["plev"][::-1].copy()), "must share their pressure levels"),
    (lambda d: [d[n].update(plev=np.array([100000.0, 50000.0, 85000.0])) for n in ("ta", "hur", "ua", "va")],
     "Source pressure values must be ascending!"),
    (lambda d: d["va"].update(time=d["va"]["time"] + DAY), "must share their time stamps"),
    (lambda d: d["ua"].update(data=torch.zeros(6, 3, 2, 4)), "must share their shape"),
])
def test_validation_messages_match_the_resident_set(edit, message):
    for cls in (DeltaSet, D.StreamedDeltaSet):
        d = _deltas()
        edit(d)
        with pytest.raises(ValueError, match=message):
            cls(d, device="cpu")
    d = _deltas()
    del d["zg"]
    with pytest.raises(KeyError, match="climate delta 'zg' missing"):
        D.StreamedDeltaSet(d, device="cpu")
    with pytest.raises(ValueError, match="at least 2 slots"):
        D.StreamedDeltaSet(_deltas(), device="cpu", slots=1)


def test_streamed_set_is_not_broadcast():
    from pgw4era5_b200 import parallel

    class Streamed:
        streamed = True
    with pytest.raises(ValueError, match="every rank reads the delta files itself"):
        parallel.broadcast_deltas(Streamed())

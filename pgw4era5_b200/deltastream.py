"""
Climate deltas that do not fit in HBM: daily climatologies at the global 0.25 degree grid (365 stamps,
153 GB resident on plev19).  A timestep only reads the two stamps that bracket its date, and consecutive
3-hourly ERA5 timesteps share them, so ``StreamedDeltaSet`` keeps a ring of a few stamps on the device and
loads a stamp from its source when a timestep needs one that is not there.  The six 2-D deltas stay resident.

Two rings, each of ``slots`` stamps: the packed ta/hur/ua/va nodes the column kernel reads (``d4``) and zg,
which may have its own time axis.  A load on a miss:

1. takes the least recently used slot that the current timestep does not need;
2. waits on the host until the ring's pinned staging buffer has been copied to the device by the previous load;
3. fills the staging buffer from the source (a NetCDF-3 record, raw big-endian bytes, or a host array);
4. on a copy stream of its own: H2D, then waits for every use of the slot recorded since it was last loaded
   (``hold``), then packs the four variables into the slot (``pgw_pack_d4_f32``; zg goes straight into its
   slot, so its H2D waits instead, followed by ``pgw_byteswap32`` for big-endian records);
5. records the slot's ready event, which the stream that asked for the stamp waits on.

The host never waits for device work other than the staging buffer's previous H2D.
"""
import ctypes as C
import os
import time

import numpy as np
import torch

from . import _native as N
from . import ncio, settings
from .engine import VARS_2D, VARS_3D, VARS_PACKED, DeltaSetBase, read_axes
from .nc3raw import NC_FLOAT, NotNetCDF3, RawNC3


class ArraySource:
    """Stamps of a host array (numpy or CPU torch, [nt, K, ny, nx]) in native byte order."""
    swap = 0

    def __init__(self, data):
        t = data if isinstance(data, torch.Tensor) else torch.from_numpy(np.asarray(data))
        if t.device.type != "cpu":
            raise ValueError("a streamed delta set reads host arrays; deltas already on the device belong in a DeltaSet")
        self.t = t.to(torch.float32).contiguous()
        self.shape = tuple(self.t.shape)

    def read(self, i, out):
        out.copy_(self.t[i].reshape(-1))


class NC3Source:
    """Stamps of a float32 variable of a NetCDF-3 file: entry ``i`` of its first axis (a record when that
    axis is the record dimension), read as raw big-endian bytes straight into pinned memory."""
    swap = 1

    def __init__(self, path, name, raw=None):
        self.raw = raw if raw is not None else RawNC3(path)
        v = self.raw.vars[name]
        if v.nc_type != NC_FLOAT:
            raise ValueError("%s in %s is not float32" % (name, path))
        self.name, self.shape = name, tuple(v.shape)
        self.f = open(path, "rb", buffering=0)

    def read(self, i, out):
        self.raw.read_stamp(self.f, self.name, out.numpy(), i)

    def close(self):
        self.f.close()


def stamp_record(keep, i):
    """Entry of the source that holds kept stamp ``i``: 29 February is not a kept stamp, and ``i = -1`` (a date
    before the first stamp of its year) is the last one."""
    return keep[i % len(keep)]


def choose_slot(keys, ticks, busy):
    """Slot to load into: an empty one, else the least recently used one outside ``busy``."""
    free = [s for s in range(len(keys)) if s not in busy]
    if not free:
        raise RuntimeError("every slot of the delta ring is in use by the current timestep: use more slots")
    empty = [s for s in free if keys[s] is None]
    return empty[0] if empty else min(free, key=lambda s: ticks[s])


class _Ring:
    """``slots`` device buffers of one stamp each (``words`` floats per variable, ``nvar`` = 4 packed variables or
    1): which slot holds which stamp, eviction and the device-side waits for the slots' users.  A subclass fills a
    slot: ``_stage`` on the host, then ``_fill`` on the set's copy stream, which must wait for ``_wait_uses`` before
    it writes the slot."""

    def __init__(self, owner, name, keep, words, nvar, slots):
        dev = owner.device
        self.owner, self.name, self.keep, self.n = owner, name, keep, words
        self.bufs = [torch.empty(words * nvar, device=dev, dtype=torch.float32) for _ in range(slots)]
        self.keys, self.ticks = [None] * slots, [0] * slots
        self.ready = [torch.cuda.Event() for _ in range(slots)]
        self.uses = [{} for _ in range(slots)]              # stream -> last use event (a stream runs in order)
        self.pending, self.clock, self.loads = set(), 0, 0

    def device_tensors(self):
        return list(self.bufs)

    def acquire(self, i, other=None):
        """Slot of kept stamp ``i`` (-1: the last, the year wrap), loaded on a miss; the slot of kept stamp
        ``other`` is not evicted.  The current stream waits until the slot is filled."""
        nt = len(self.keep)
        i %= nt
        self.clock += 1
        if i in self.keys:
            s = self.keys.index(i)
        else:
            protect = {other % nt} if other is not None else set()
            busy = self.pending | {s for s, k in enumerate(self.keys) if k in protect}
            s = choose_slot(self.keys, self.ticks, busy)
            self._load(s, i)
        self.ticks[s] = self.clock
        self.pending.add(s)
        torch.cuda.current_stream().wait_event(self.ready[s])
        return s

    def _wait_uses(self, s, stream):
        for e in self.uses[s].values():
            stream.wait_event(e)

    def _stage(self, rec):
        """Host work of a load, before anything is queued on the copy stream."""

    def _load(self, s, i):
        rec = stamp_record(self.keep, i)
        timing = self.owner.load_events
        t0 = time.perf_counter()
        self._stage(rec)
        t1 = time.perf_counter()
        cs = self.owner.copy_stream
        with torch.cuda.stream(cs):
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)] if timing is not None else None
            if ev:
                ev[0].record(cs)
            self._fill(s, rec, cs, ev)
            if ev:
                ev[2].record(cs)
            self.ready[s].record(cs)
        self.uses[s] = {}
        self.keys[s] = i
        self.loads += 1
        if ev:
            timing.append(dict(ring=self.name, fill_s=t1 - t0, events=ev))


class _HostRing(_Ring):
    """A ring loaded from ``sources`` through one pinned staging buffer: the host reads the stamp, the copy stream
    uploads it and packs it into the slot (zg: uploads it into the slot)."""

    def __init__(self, owner, name, sources, keep, words, slots):
        super().__init__(owner, name, keep, words, len(sources), slots)
        self.sources = sources
        self.packed = len(sources) == 4
        self.swap = sources[0].swap
        self.stride = (words + 3) // 4 * 4                  # 16-byte aligned pieces: vector loads in the pack
        self.host = torch.empty(len(sources) * self.stride, dtype=torch.float32, pin_memory=True)
        self.host_free = torch.cuda.Event()
        self.raw = torch.empty(4 * self.stride, device=owner.device, dtype=torch.float32) if self.packed else None

    def device_tensors(self):
        return self.bufs + ([self.raw] if self.raw is not None else [])

    def _stage(self, rec):
        self.host_free.synchronize()
        for j, src in enumerate(self.sources):
            src.read(rec, self.host[j * self.stride:j * self.stride + self.n])

    def _fill(self, s, rec, cs, ev):
        if not self.packed:
            self._wait_uses(s, cs)
        dst = self.raw if self.packed else self.bufs[s]
        dst.copy_(self.host[:dst.numel()], non_blocking=True)
        self.host_free.record(cs)
        if ev:
            ev[1].record(cs)
        st = C.c_void_p(cs.cuda_stream)
        if self.packed:
            self._wait_uses(s, cs)
            p = [C.c_void_p(self.raw.data_ptr() + 4 * j * self.stride) for j in range(4)]
            N.check(N.lib.pgw_pack_d4_f32(*p, C.c_void_p(self.bufs[s].data_ptr()), self.n, self.swap, st),
                    "pgw_pack_d4_f32")
        elif self.swap:
            N.check(N.lib.pgw_byteswap32(C.c_void_p(self.bufs[s].data_ptr()), self.n, st), "pgw_byteswap32")


class StreamedDeltaSet(DeltaSetBase):
    """
    The interface of ``engine.DeltaSet`` for climatologies that do not fit in HBM.

    ``deltas``: the dict form ``DeltaSet`` takes.  The ``data`` of ta, hur, ua, va and zg is a host array
    (numpy or CPU torch) or a source such as ``NC3Source`` (``shape``, ``swap`` and ``read(entry, out)``, which
    fills the pinned float32 tensor ``out`` with one stamp); the 2-D deltas are uploaded once.  ``slots``: stamps per ring
    (at least 2, the two a timestep reads).  A streamed set cannot be broadcast to other ranks
    (``parallel.broadcast_deltas``) nor serve an engine in latitude-band mode.
    """
    streamed = True

    def __init__(self, deltas, device="cuda", slots=4):
        if slots < 2:
            raise ValueError("a streamed delta set needs at least 2 slots per ring")
        self.device = torch.device(device)
        self.vars, sources, keeps, flat = {}, {}, {}, {}
        for name in VARS_3D + VARS_2D:
            if name not in deltas:
                raise KeyError("climate delta %r missing" % name)
            d = deltas[name]
            stamps, keep, plev = read_axes(name, d)
            self.vars[name] = dict(time=stamps, plev=plev, data=None)
            data = d["data"]
            if name in VARS_3D:
                src = data if hasattr(data, "read") else ArraySource(data)
                if len(src.shape) != 4 or src.shape[0] != len(d["time"]):
                    raise ValueError("%s delta: data of shape %s for %d time stamps" % (name, src.shape,
                                                                                       len(d["time"])))
                sources[name], keeps[name] = src, keep
                continue
            if not isinstance(data, torch.Tensor):
                data = torch.as_tensor(np.asarray(data))
            if len(keep) != len(d["time"]):
                data = data[torch.as_tensor(keep, device=data.device)]
            flat[name] = data
        self.shape2d = tuple(flat["ts"].shape[-2:])
        self.ncol = self.shape2d[0] * self.shape2d[1]
        self._check_axes({name: sources[name].shape for name in VARS_PACKED})
        for name in VARS_3D:
            if tuple(sources[name].shape[-2:]) != self.shape2d:
                raise ValueError("%s delta is on a %s grid, the 2-D deltas on %s" % (name, sources[name].shape[-2:],
                                                                                     self.shape2d))
        self._upload_2d(flat)
        self.sources = sources
        self.copy_stream = torch.cuda.Stream(device=self.device)
        # set to [] to collect every load: the host fill time and three CUDA events on the copy stream (start; upload
        # done, or the slot's users done for a regridded stamp; slot filled)
        self.load_events = None
        K, Kz = sources["ta"].shape[1], sources["zg"].shape[1]
        self.rings = dict(d4=_HostRing(self, "d4", [sources[n] for n in VARS_PACKED], keeps["ta"], K * self.ncol,
                                       slots),
                          zg=_HostRing(self, "zg", [sources["zg"]], keeps["zg"], Kz * self.ncol, slots))
        self.ts_clim = None
        self.refresh_derived()

    def _upload_2d(self, flat):
        """The 2-D deltas (name -> [nt, ny, nx] tensor, 29 February dropped) into one device arena."""
        offs, total = {}, 0
        for name in VARS_2D:
            offs[name] = total
            total += (flat[name].numel() + 3) // 4 * 4
        self.arena = torch.empty(total, device=self.device, dtype=torch.float32)
        for name in VARS_2D:
            v = self.arena[offs[name]:offs[name] + flat[name].numel()].view(flat[name].shape)
            v.copy_(flat.pop(name).to(self.device, torch.float32))
            self.vars[name]["data"] = v

    def device_bytes(self):
        """Device memory of the set: the 2-D arena, the ring slots and the packing buffer."""
        ts = [self.arena] + [t for r in self.rings.values() for t in r.device_tensors()]
        return sum(t.numel() * t.element_size() for t in ts)

    def hold(self, stream=None):
        """The stamps handed out since the last call are in use until ``stream`` (default: the current one)
        gets to this point; a load that evicts one of them waits for it on the device."""
        if not any(r.pending for r in self.rings.values()):
            return
        stream = stream if stream is not None else torch.cuda.current_stream()
        ev = torch.cuda.Event()
        ev.record(stream)
        for r in self.rings.values():
            for s in r.pending:
                r.uses[s][stream.cuda_stream] = ev
            r.pending = set()

    def _ring_of(self, name):
        return self.rings["d4"] if name in VARS_PACKED else self.rings["zg"]

    def stamp(self, name, i):
        """Kept stamp ``i`` of variable ``name`` as a device tensor ([K, ny, nx] or [ny, nx]), loaded if needed."""
        if name in VARS_2D:
            return self.vars[name]["data"][i]
        r = self._ring_of(name)
        buf = r.bufs[r.acquire(i)]
        ny, nx = self.shape2d
        if name == "zg":
            return buf.view(-1, ny, nx)
        return buf.view(-1, ny, nx, 4)[..., VARS_PACKED.index(name)]

    def _pair(self, ring, b):
        lo = ring.acquire(b.ind_before, b.ind_after)
        hi = ring.acquire(b.ind_after, b.ind_before)
        return ring.bufs[lo].data_ptr(), ring.bufs[hi].data_ptr()

    def slab(self, name, when, level=None):
        """pgw_tslab for variable ``name`` at ERA5 time ``when`` (optionally one plev)."""
        if name != "zg":
            return super().slab(name, when, level)
        b = self.bracket(name, when)
        lo, hi = self._pair(self.rings["zg"], b)
        off = 4 * self.ncol * level if level is not None else 0
        return N.TSlab(lo + off, hi + off, b.x_hi, b.x_new)

    def slab4(self, when):
        """pgw_tslab of the packed (ta, hur, ua, va) deltas at ERA5 time ``when``."""
        b = self.bracket("ta", when)
        lo, hi = self._pair(self.rings["d4"], b)
        return N.TSlab(lo, hi, b.x_hi, b.x_new)


# --------------------------------------------------------------------------- delta files
def delta_file(delta_input_dir, name):
    """(path, variable name) of delta ``name`` (step_03_apply_to_era.py:533-539: ps as HIST, the rest SCEN-HIST)."""
    var, base = ("ps", settings.file_name_bases['HIST']) if name == "ps_hist" else \
        (name, settings.file_name_bases['SCEN-HIST'])
    return os.path.join(delta_input_dir, base.format(var)), var


def read_3d_headers(delta_input_dir):
    """name -> (RawNC3 header, variable, dict(time, plev)) of the 3-D delta files, reading nothing but the
    headers and the time and plev coordinates; None if one of them is not a float32 NetCDF-3 file."""
    out = {}
    for name in VARS_3D:
        path, var = delta_file(delta_input_dir, name)
        try:
            raw = RawNC3(path)
        except NotNetCDF3:
            return None
        v = raw.vars[var]
        if v.nc_type != NC_FLOAT or len(v.shape) != 4:
            return None
        with open(path, "rb", buffering=0) as f:
            tv = raw.vars[settings.TIME_GCM]
            axes = dict(time=ncio.decode_time(ncio.Variable(tv.dims, raw.read_variable(f, tv.name), tv.attrs)),
                        plev=np.asarray(raw.read_variable(f, settings.PLEV_GCM), dtype=np.float64))
        out[name] = (raw, var, axes)
    return out


def resident_bytes(headers):
    """Device memory ``DeltaSet`` needs for the files of ``headers``: its arena (d4, zg and six 2-D deltas on
    ta's time axis) plus the largest variable, which its constructor stages on the device."""
    def kept(name):
        return len(read_axes(name, headers[name][2])[1])
    ta = headers["ta"][0].vars[headers["ta"][1]]
    zg = headers["zg"][0].vars[headers["zg"][1]]
    K, Kz, ncol = ta.shape[1], zg.shape[1], ta.shape[2] * ta.shape[3]
    arena = 4 * ncol * (4 * kept("ta") * K + kept("zg") * Kz + len(VARS_2D) * kept("ta"))
    staged = max(4 * int(np.prod(h[0].vars[h[1]].shape, dtype=np.int64)) for h in headers.values())
    return arena + staged


def should_stream(headers, device, max_resident_bytes=None):
    """Stream when the resident set would need more than ``max_resident_bytes`` (default: half of the
    device's free memory now)."""
    if headers is None:
        return False
    if max_resident_bytes is None:
        max_resident_bytes = torch.cuda.mem_get_info(torch.device(device))[0] // 2
    return resident_bytes(headers) > max_resident_bytes


def open_streamed(delta_input_dir, headers, device="cuda", slots=4):
    """StreamedDeltaSet over the delta files: 3-D deltas read stamp by stamp, 2-D deltas read whole."""
    deltas = {}
    for name in VARS_3D:
        raw, var, axes = headers[name]
        deltas[name] = dict(axes, data=NC3Source(raw.path, var, raw))
    for name in VARS_2D:
        path, var = delta_file(delta_input_dir, name)
        ds = ncio.open_dataset(path)
        deltas[name] = dict(time=ncio.decode_time(ds[settings.TIME_GCM]), plev=None, data=ds[var].data)
    return StreamedDeltaSet(deltas, device=device, slots=slots)

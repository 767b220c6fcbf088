"""
Raw access to NetCDF-3 files (classic, 64-bit offset and CDF-5) for the file pipeline of the
step_03 drop-in: the header is parsed here (it is a few hundred bytes), so that the big fields can
be moved between the file and pinned host memory with ``readinto`` / ``pwrite`` -- no decoding, no
intermediate numpy copies.  NetCDF-3 stores big-endian numbers; the byte order of the float32
fields is swapped on the GPU (``pgw_byteswap32``), next to the H2D / D2H copies.

Only what the pipeline needs: locate a variable (offset, shape, type) and read or overwrite the
values of one record, or of a band of its rows (latitude-band mode).  Everything else (coordinates,
attributes, the engine's level tables) goes through ``ncio``.  File format: NetCDF Classic Format
Specification (Unidata), all integers big-endian:
    header  = magic numrecs dim_list gatt_list var_list
    var     = name nelems [dimid ...] vatt_list nc_type vsize begin
"""
import os
import struct

import numpy as np

NC_DIMENSION, NC_VARIABLE, NC_ATTRIBUTE = 0x0A, 0x0B, 0x0C
_TYPES = {1: ("i1", 1), 2: ("S1", 1), 3: (">i2", 2), 4: (">i4", 4), 5: (">f4", 4), 6: (">f8", 8),
          7: ("u1", 1), 8: (">u2", 2), 9: (">u4", 4), 10: (">i8", 8), 11: (">u8", 8)}
NC_FLOAT = 5


class NotNetCDF3(ValueError):
    pass


class _Reader:
    def __init__(self, buf, version):
        self.b, self.p, self.v = buf, 0, version

    def u32(self):
        (x,) = struct.unpack_from(">I", self.b, self.p)
        self.p += 4
        return x

    def u64(self):
        (x,) = struct.unpack_from(">Q", self.b, self.p)
        self.p += 8
        return x

    def size(self):                      # NON_NEG: 64 bit in CDF-5
        return self.u64() if self.v == 5 else self.u32()

    def name(self):
        n = self.size()
        s = bytes(self.b[self.p:self.p + n]).decode("utf-8")
        self.p += (n + 3) & ~3
        return s

    def values(self, nc_type, nelems):
        """``nelems`` values of ``nc_type`` (padded to four bytes): str for NC_CHAR, else a native numpy
        array, a python scalar if there is exactly one."""
        dt, size = _TYPES[nc_type]
        raw = bytes(self.b[self.p:self.p + size * nelems])
        self.p += ((size * nelems) + 3) & ~3
        if nc_type == 2:
            return raw.rstrip(b"\x00").decode("utf-8", "replace")
        a = np.frombuffer(raw, dtype=dt).astype(np.dtype(dt).newbyteorder("="))
        return a.reshape(()).item() if a.size == 1 else a

    def att_list(self):
        tag = self.u32()
        n = self.size()
        out = {}
        if tag == 0:
            return out
        if tag != NC_ATTRIBUTE:
            raise NotNetCDF3("attribute list expected")
        for _ in range(n):
            name = self.name()
            t = self.u32()
            out[name] = self.values(t, self.size())
        return out


class RawVar:
    __slots__ = ("name", "dims", "shape", "nc_type", "dtype", "vsize", "begin", "is_record", "attrs")

    def __init__(self, name, dims, shape, nc_type, vsize, begin, is_record, attrs=None):
        self.name, self.dims, self.shape, self.nc_type = name, dims, shape, nc_type
        self.dtype, self.vsize, self.begin, self.is_record = np.dtype(_TYPES[nc_type][0]), vsize, begin, is_record
        self.attrs = dict(attrs or {})

    @property
    def record_shape(self):
        """Shape of the values of one record (record variables) or of the whole variable."""
        return self.shape[1:] if self.is_record else self.shape

    @property
    def nbytes(self):
        return int(np.prod(self.record_shape, dtype=np.int64)) * self.dtype.itemsize


class RawNC3:
    """Header of a NetCDF-3 file: ``dims`` (name -> length, record dimension -> numrecs), ``vars``."""

    def __init__(self, path, header_bytes=1 << 20):
        self.path = path
        with open(path, "rb") as f:
            head = f.read(header_bytes)
            if len(head) < 8 or head[:3] != b"CDF" or head[3] not in (1, 2, 5):
                raise NotNetCDF3("%s is not a NetCDF-3 file" % path)
            while True:
                try:
                    self._parse(head)
                    break
                except (struct.error, IndexError):
                    if len(head) < header_bytes:
                        raise NotNetCDF3("truncated header in %s" % path)
                    header_bytes *= 8
                    f.seek(0)
                    head = f.read(header_bytes)

    def _parse(self, head):
        version = head[3]
        r = _Reader(memoryview(head), version)
        r.p = 4
        numrecs = r.size()
        streaming = numrecs == (0xFFFFFFFFFFFFFFFF if version == 5 else 0xFFFFFFFF)
        tag, n = r.u32(), r.size()
        dims = []
        if tag == NC_DIMENSION:
            for _ in range(n):
                name = r.name()
                dims.append((name, r.size()))
        elif tag != 0:
            raise NotNetCDF3("dimension list expected")
        self.attrs = r.att_list()
        tag, n = r.u32(), r.size()
        self.vars, rec_vars = {}, []
        if tag == NC_VARIABLE:
            for _ in range(n):
                name = r.name()
                nd = r.size()
                dimids = [r.size() for _ in range(nd)]
                vattrs = r.att_list()
                nc_type = r.u32()
                vsize = r.size()
                begin = r.u64() if version in (2, 5) else r.u32()
                is_rec = nd > 0 and dims[dimids[0]][1] == 0
                shape = tuple(dims[d][1] for d in dimids)
                v = RawVar(name, tuple(dims[d][0] for d in dimids), shape, nc_type, vsize, begin, is_rec, vattrs)
                self.vars[name] = v
                if is_rec:
                    rec_vars.append(v)
        elif tag != 0:
            raise NotNetCDF3("variable list expected")
        self.version, self.header_size = version, r.p
        # record size: sum of the per-record sizes padded to four bytes (computed here: the 32-bit vsize of the
        # header saturates for huge variables); a single record variable is not padded
        per_rec = [int(np.prod(v.shape[1:], dtype=np.int64)) * v.dtype.itemsize for v in rec_vars]
        self.recsize = per_rec[0] if len(rec_vars) == 1 else sum((b + 3) & ~3 for b in per_rec)
        if streaming:
            size = os.path.getsize(self.path)
            first = min((v.begin for v in rec_vars), default=size)
            numrecs = (size - first) // self.recsize if rec_vars and self.recsize else 0
        self.numrecs = int(numrecs)
        self.dims = {name: (self.numrecs if length == 0 else length) for name, length in dims}
        for v in rec_vars:
            v.shape = (self.numrecs,) + v.shape[1:]

    def read_variable(self, fobj, name):
        """All values of ``name`` as a native-endian numpy array (record variables: every record).  Reads go
        through ``preadv`` in pieces, so variables and records beyond 2 GiB are fine."""
        v = self.vars[name]
        out = np.empty(v.shape, dtype=v.dtype)
        if v.is_record:
            for rec in range(self.numrecs):
                if out[rec:rec + 1].nbytes:
                    self.read_into(fobj, name, out[rec:rec + 1], record=rec)
        elif out.nbytes:
            self.read_into(fobj, name, out)
        if v.dtype.byteorder == ">":
            return out.byteswap(inplace=True).view(v.dtype.newbyteorder("="))
        return out

    def offset(self, name, record=0):
        v = self.vars[name]
        if v.is_record:
            if not 0 <= record < self.numrecs:
                raise IndexError("record %d of %d" % (record, self.numrecs))
            return v.begin + record * self.recsize
        return v.begin

    def read_into(self, fobj, name, buf, record=0):
        """Fill ``buf`` (writable buffer of exactly the variable's record size) with the raw
        big-endian bytes of ``name``; ``fobj`` is the file opened 'rb' (unbuffered is best)."""
        v = self.vars[name]
        mv = memoryview(buf).cast("B")
        if mv.nbytes != v.nbytes:
            raise ValueError("%s: buffer has %d bytes, variable %d" % (name, mv.nbytes, v.nbytes))
        off, done = self.offset(name, record), 0
        while done < mv.nbytes:                      # os.preadv may return short counts on large reads
            n = os.preadv(fobj.fileno(), [mv[done:]], off + done)
            if n <= 0:
                raise IOError("unexpected end of %s while reading %s" % (self.path, name))
            done += n

    def read_stamp(self, fobj, name, buf, i):
        """Raw big-endian bytes of entry ``i`` of the first axis of ``name`` into ``buf``: record ``i`` of a
        record variable, else the slice at ``begin + i * bytes per entry``."""
        v = self.vars[name]
        if v.is_record:
            return self.read_into(fobj, name, buf, record=i)
        mv = memoryview(buf).cast("B")
        step = int(np.prod(v.shape[1:], dtype=np.int64)) * v.dtype.itemsize
        if mv.nbytes != step or not 0 <= i < v.shape[0]:
            raise ValueError("%s: entry %d of %d, buffer has %d bytes, entry %d" % (name, i, v.shape[0], mv.nbytes,
                                                                                  step))
        off, done = v.begin + i * step, 0
        while done < mv.nbytes:
            n = os.preadv(fobj.fileno(), [mv[done:]], off + done)
            if n <= 0:
                raise IOError("unexpected end of %s while reading %s" % (self.path, name))
            done += n

    def write_from(self, fd, name, buf, record=0):
        """Overwrite the values of ``name`` in the file open as descriptor ``fd`` with raw big-endian bytes."""
        v = self.vars[name]
        mv = memoryview(buf).cast("B")
        if mv.nbytes != v.nbytes:
            raise ValueError("%s: buffer has %d bytes, variable %d" % (name, mv.nbytes, v.nbytes))
        off, done = self.offset(name, record), 0
        while done < mv.nbytes:
            done += os.pwrite(fd, mv[done:], off + done)

    def _row_pieces(self, name, nbytes, r0, r1, record):
        """(file offset, buffer offset, bytes) of every contiguous piece of rows [r0, r1) of the second-to-last
        axis of ``name``, for every index of the axes in front of it; the buffer holds the band as
        [..., r1 - r0, nx]."""
        v = self.vars[name]
        shp = v.record_shape
        if len(shp) < 2:
            raise ValueError("%s has no row axis" % name)
        ny, row = shp[-2], shp[-1] * v.dtype.itemsize
        lead = int(np.prod(shp[:-2], dtype=np.int64))
        if not 0 <= r0 < r1 <= ny:
            raise ValueError("%s: rows %d..%d of %d" % (name, r0, r1, ny))
        if not v.is_record and record != 0:
            raise IndexError("%s is not a record variable" % name)
        band = (r1 - r0) * row
        if nbytes != lead * band:
            raise ValueError("%s: buffer has %d bytes, rows %d..%d %d" % (name, nbytes, r0, r1, lead * band))
        base = self.offset(name, record)
        if r1 - r0 == ny:                            # whole rows of every level: one piece
            return [(base, 0, lead * band)]
        return [(base + (i * ny + r0) * row, i * band, band) for i in range(lead)]

    def read_rows(self, fobj, name, buf, r0, r1, record=0):
        """Fill ``buf`` with the raw big-endian bytes of rows [r0, r1) of ``name`` (the second-to-last axis; every
        index of the axes in front of it, e.g. levels), stored contiguously as [..., r1 - r0, nx]."""
        pieces = self._row_pieces(name, memoryview(buf).nbytes, r0, r1, record)
        mv = memoryview(buf).cast("B")
        for off, pos, count in pieces:
            done = 0
            while done < count:
                n = os.preadv(fobj.fileno(), [mv[pos + done:pos + count]], off + done)
                if n <= 0:
                    raise IOError("unexpected end of %s while reading %s" % (self.path, name))
                done += n

    def write_rows(self, fd, name, buf, r0, r1, record=0):
        """Overwrite rows [r0, r1) of ``name`` in the file open as descriptor ``fd`` with the raw big-endian bytes
        of ``buf`` (laid out as ``read_rows`` fills it); the other rows are left as they are."""
        pieces = self._row_pieces(name, memoryview(buf).nbytes, r0, r1, record)
        mv = memoryview(buf).cast("B")
        for off, pos, count in pieces:
            done = 0
            while done < count:
                n = os.pwrite(fd, mv[pos + done:pos + count], off + done)
                if n <= 0:
                    raise IOError("short write of %s to %s" % (name, self.path))
                done += n

"""
Device-resident PGW engine: the host side of the fused per-timestep pass.

``DeltaSet`` keeps the GCM climate-delta climatology in HBM (uploaded or
NCCL-broadcast once; it is time invariant), ``PGWEngine`` applies it to one
ERA5 timestep per call through ``pgw_timestep`` / ``pgw_timestep_finalize`` of
libpgw_b200.so.  This replaces the body of the reference's ``pgw_for_era5``
(step_03_apply_to_era.py:44-381) between reading and writing the file; names
of fields follow ``settings.var_name_map``.

The reference's stopping rule is field-global (step_03_apply_to_era.py:189,308).
The kernel runs a speculative number of iterations ``k_spec`` for every column
and records max|error| per iteration; ``finalize`` finds the reference's count N
on the device.  N == k_spec: nothing to do.  N < k_spec: PS/QV are rewritten for
iteration N.  Not converged within k_spec: the timestep is rerun with
``max_n_iter - 1`` iterations (the reference raises once ``it > max_n_iter``).
``k_spec`` follows the last N, which is stable from one timestep to the next.
"""
import ctypes as C

import numpy as np
import torch

from . import _native as N
from . import settings, timeinterp

VARS_3D = ("ta", "hur", "ua", "va", "zg")
VARS_PACKED = ("ta", "hur", "ua", "va")       # one float4 per pressure node and column on the device
VARS_2D = ("tas", "hurs", "ps_hist", "ts", "tos", "siconc")

_STATUS_BYTES = C.sizeof(N.TimestepStatus)

MSG_TOP = ("ERA5 top pressure is lower than climate delta top pressure. If you are certain that "
           "you do not need the data beyond to upper-most pressure level of the climate delta, "
           "you can set the flag --ignore_top_pressure_error and re-run the script.")
MSG_PREF = ("p_ref locally lies below the surface. Please set a lower reference pressue "
            "(p_ref_inp) in settings.py")
MSG_NOCONV = ('ERROR! Pressure adjustment did not converge for file {}. Consider increasing the '
              'value for "max_n_iter" in settings.py')


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def fused_refusal():
    """Why ``PGWEngine.submit`` cannot run the current settings in the fused pass (None if it can)."""
    ref_dtypes = getattr(settings, "i_reference_dtypes", 0)
    if (settings.i_reinterp and settings.p_ref_inp is None) or \
            ((settings.i_reinterp or settings.p_ref_inp is None) and ref_dtypes):
        return ("i_reinterp = 1 with p_ref_inp = None, and either of them with i_reference_dtypes = 1, "
                "run through the staged path: use apply()")
    return None


def read_axes(name, d):
    """(kept stamps, indices of the kept stamps in the source, plev or None) of one delta variable in the dict
    form ``DeltaSet`` takes; 29 February is dropped (functions.py:224-230)."""
    stamps = np.asarray(d["time"]).astype("datetime64[ns]")
    keep = timeinterp.drop_leap_day(stamps)
    plev = None if d.get("plev") is None else np.asarray(d["plev"], dtype=np.float64)
    return stamps[keep], keep, plev


class DeltaSetBase:
    """What the resident and the streamed delta set share: the pressure axis of the packed deltas and its checks,
    which two stamps bracket an ERA5 date, the slabs of resident variables and ``ts_clim``.  Subclasses fill
    ``vars`` (name -> dict(time, plev, data)) and call ``_check_axes`` with the shapes of ta, hur, ua, va."""

    def _check_axes(self, shapes):
        plev = self.vars["ta"]["plev"]
        for name in ("hur", "ua", "va"):
            if not np.array_equal(self.vars[name]["plev"], plev):
                raise ValueError("ta, hur, ua, va deltas must share their pressure levels")
        self.plev = plev
        desc = bool(plev[0] > plev[-1])
        mono = np.all(np.diff(plev) < 0) if desc else np.all(np.diff(plev) > 0)
        if not mono:
            raise ValueError("Source pressure values must be ascending!")
        self.plev_descending = desc
        self.plev_dev = torch.as_tensor(plev, device=self.device, dtype=torch.float64)
        stamps = self.vars["ta"]["time"]
        for name in ("hur", "ua", "va"):
            if not np.array_equal(self.vars[name]["time"], stamps):
                raise ValueError("ta, hur, ua, va deltas must share their time stamps")
            if tuple(shapes[name]) != tuple(shapes["ta"]):
                raise ValueError("ta, hur, ua, va deltas must share their shape")
        self._brackets, self._moved, self._time_group, self._time_ids, self._lay = {}, {}, {}, {}, {}

    def refresh_derived(self):
        """Annual mean of the ts delta (step_03_apply_to_era.py:134-136), computed once."""
        ts = self.vars["ts"]["data"]
        if self.ts_clim is None or tuple(self.ts_clim.shape) != tuple(ts.shape[1:]):     # else in place: its address
            self.ts_clim = torch.empty(ts.shape[1:], device=self.device, dtype=torch.float32)   # is cached in args
        N.check(N.lib.pgw_time_mean_f32(_ptr(ts), ts.shape[0], _ptr(self.ts_clim), self.ncol, _stream()),
                "pgw_time_mean_f32")
        # the pipelines run on their own streams, which do not wait for the stream the arena was filled on
        torch.cuda.current_stream().synchronize()

    def bracket(self, name, when):
        """TimeBracket of variable ``name`` for the ERA5 date ``when``; variables that share their time axis
        (normally all of them) share the result, and the year-shifted stamps are kept per year."""
        gid = self._time_group.get(name)
        if gid is None:
            stamps = self.vars[name]["time"]
            gid = self._time_group[name] = self._time_ids.setdefault(stamps.tobytes(), len(self._time_ids))
        key = (gid, when)
        b = self._brackets.get(key)
        if b is None:
            if len(self._brackets) > 4096:
                self._brackets.clear()
            stamps = self.vars[name]["time"]
            mk = (gid, when.year)
            moved = self._moved.get(mk)
            if moved is None:
                if len(self._moved) > 64:
                    self._moved.clear()
                moved = self._moved[mk] = timeinterp.moved_to_year(stamps, when.year)
            b = timeinterp.bracket(stamps, when, moved=moved)
            self._brackets[key] = b
        return b

    def _layout(self, name):
        """(address of the first time slab, bytes per time slab, bytes per level) of a variable."""
        lay = self._lay.get(name)
        if lay is None:
            t = self.d4 if name == "d4" else self.vars[name]["data"]
            lay = (t.data_ptr(), t.stride(0) * 4, (t.stride(1) * 4) if t.dim() == 4 else 0)
            self._lay[name] = lay
        return lay

    def slab(self, name, when, level=None):
        """pgw_tslab for variable ``name`` at ERA5 time ``when`` (optionally one plev)."""
        b = self.bracket(name, when)
        base, st, sl = self._layout(name)
        off = base + (sl * level if level is not None else 0)
        nt = len(self.vars[name]["time"])
        return N.TSlab(off + st * (b.ind_before % nt), off + st * (b.ind_after % nt), b.x_hi, b.x_new)


class DeltaSet(DeltaSetBase):
    """
    Climate deltas resident on one GPU.

    ``deltas``: var -> dict(time=datetime64[nt], plev=[K] or None, data=[nt,(K),ny,nx])
    for ta, hur, ua, va, zg, tas, hurs, ts, tos, siconc (SCEN-HIST) and ``ps_hist``
    (the HIST ps climatology, functions.py:330-332).  29 February is dropped
    once here (functions.py:224-230).

    Layout in HBM: ta, hur, ua, va are interleaved per pressure node and column as
    ``d4[nt, K, ny, nx, 4]`` (one 16-byte load per node, month and column in the column
    kernel); ``vars[name]["data"]`` of these four are strided views of ``d4``.  zg and
    the 2-D deltas stay separate, contiguous fields.
    """

    def __init__(self, deltas, device="cuda"):
        self.device = torch.device(device)
        self.vars = {}
        staged = {}
        for name in VARS_3D + VARS_2D:
            if name not in deltas:
                raise KeyError("climate delta %r missing" % name)
            d = deltas[name]
            stamps, keep, plev = read_axes(name, d)
            data = d["data"]
            if not isinstance(data, torch.Tensor):
                data = torch.as_tensor(np.asarray(data))
            if len(keep) != len(d["time"]):
                data = data[torch.as_tensor(keep, device=data.device)]
            self.vars[name] = dict(time=stamps, plev=plev, data=None)
            staged[name] = data
        self.shape2d = tuple(staged["ts"].shape[-2:])
        self.ncol = self.shape2d[0] * self.shape2d[1]
        self._check_axes({name: staged[name].shape for name in VARS_PACKED})
        # ONE arena holds the whole climatology (the packed float4 nodes first: 16-byte aligned), so that
        # replicating it to the other GPUs is one NCCL broadcast (parallel.broadcast_deltas)
        shapes = [("d4", tuple(staged["ta"].shape) + (4,))] + \
                 [(n, tuple(staged[n].shape)) for n in ("zg",) + VARS_2D]
        offs, total = {}, 0
        for name, shp in shapes:
            offs[name] = total
            total += (int(np.prod(shp)) + 3) // 4 * 4
        self.arena = torch.empty(total, device=self.device, dtype=torch.float32)
        view = lambda name, shp: self.arena[offs[name]:offs[name] + int(np.prod(shp))].view(shp)
        self.d4 = view(*shapes[0])
        for i, name in enumerate(VARS_PACKED):
            self.d4[..., i].copy_(staged.pop(name).to(self.device, torch.float32))
            self.vars[name]["data"] = self.d4[..., i]
        for name, shp in shapes[1:]:
            v = view(name, shp)
            v.copy_(staged.pop(name).to(self.device, torch.float32))
            self.vars[name]["data"] = v
        self.ts_clim = None
        self.refresh_derived()

    def tensors(self):
        """The device memory that holds the climatology (for the NCCL broadcast): one arena."""
        return [self.arena]

    def hold(self, stream=None):
        """The stamps handed out since the last call stay in use until ``stream`` gets here.  Every stamp is
        resident, so there is nothing to record."""

    def stamp(self, name, i):
        """Kept stamp ``i`` of variable ``name`` as a device tensor ([K, ny, nx] or [ny, nx])."""
        return self.vars[name]["data"][i]

    def slab4(self, when):
        """pgw_tslab of the packed (ta, hur, ua, va) deltas at ERA5 time ``when``."""
        b = self.bracket("ta", when)
        base, st, _ = self._layout("d4")
        nt = len(self.vars["ta"]["time"])
        return N.TSlab(base + st * (b.ind_before % nt), base + st * (b.ind_after % nt), b.x_hi, b.x_new)


class Pending:
    """A submitted timestep; ``result()`` waits for it and applies the host-side checks."""

    def __init__(self, engine, args, out, ws, ctx):
        self.engine, self.args, self.out = engine, args, out
        self.ws, self.ctx = ws, ctx
        self.status = None              # private copy of the status block once the timestep has finished
        self._done = None

    def snapshot(self):
        """Wait for the timestep and take its status block out of the slot's pinned buffer (which the
        next submit on the same slot overwrites)."""
        if self.status is None:
            self.ws["event"].synchronize()
            self.status = N.TimestepStatus.from_buffer_copy(self.ws["status_host"].numpy())
            if self.ws.get("inflight") is self:
                self.ws["inflight"] = None
        return self.status

    def result(self):
        if self._done is None:
            self._done = self.engine._complete(self)
        return self._done


class PGWEngine:
    """
    ak, bk: half-level hybrid coefficients [L+1] (index 0 = model top); akm/bkm
    optional full-level coefficients (else the reference's mid-point rule,
    step_03_apply_to_era.py:68-85); soil1: soil depths [S].  ``ps_bound`` and, with
    ``p_ref_inp = None``, ``p_floor`` (the lowest per-column reference pressure) size the
    column stash; a timestep that leaves that range is rerun with a wider one.  The default
    floor of 300 hPa is a lower pressure than the ~400 hPa the highest ERA5 terrain selects.
    """

    def __init__(self, ak, bk, deltas, soil1=(), akm=None, bkm=None, ps_bound=110000.0, group=None,
                 band_exchange="auto", p_floor=30000.0):
        if not torch.cuda.is_available():
            raise RuntimeError("PGWEngine needs a CUDA device (B200, sm_100a); there is no CPU path")
        self.deltas = deltas
        self.device = deltas.device
        ak = np.asarray(ak)
        bk = np.asarray(bk)
        if akm is None:
            akm = 0.5 * np.diff(ak) + ak[:-1]
            bkm = 0.5 * np.diff(bk) + bk[:-1]
        self.ak = np.ascontiguousarray(ak, dtype=np.float64)
        self.bk = np.ascontiguousarray(bk, dtype=np.float64)
        self.akm = np.ascontiguousarray(akm, dtype=np.float64)
        self.bkm = np.ascontiguousarray(bkm, dtype=np.float64)
        self.nlev = len(self.akm)
        dev = lambda a: torch.as_tensor(a, device=self.device, dtype=torch.float64)
        self.ak_d, self.bk_d, self.akm_d, self.bkm_d = dev(self.ak), dev(self.bk), dev(self.akm), dev(self.bkm)
        soil1 = np.asarray(soil1)
        if len(soil1) > N.PGW_MAX_SOIL:
            raise ValueError("at most %d soil levels" % N.PGW_MAX_SOIL)
        self.soil_decay = np.exp(-soil1 / 2.8).astype(np.float64)     # step_03:140
        self.ps_bound = float(ps_bound)
        self.p_floor = float(p_floor)
        self._zg_tables = None
        self.group = group
        if group is not None and getattr(deltas, "streamed", False):
            raise ValueError("latitude bands need a resident DeltaSet: a streamed delta set is not supported")
        # latitude-band mode: how the bands agree on the iteration count.  "p2p": pgw_band_exchange, one kernel over
        # peer memory behind the column kernel (inboxes in torch symmetric memory); "nccl": pack, all-reduce(MAX),
        # unpack; "auto": p2p where the peer mapping can be set up, else nccl.
        self.band_exchange = None
        self._xseq = 0
        if group is not None:
            self.band_exchange = self._setup_band_exchange(band_exchange)
        self.k_pred = 8
        self._n_hist = []               # iteration counts of the last few timesteps
        self._ws = {}
        self._zg_level = {}
        self.stats = dict(timesteps=0, rewrites=0, reruns=0, launches=0)
        self.kernel_events = None       # set to [] to collect CUDA events around the column kernel

    def _setup_band_exchange(self, mode):
        import torch.distributed as dist
        if mode not in ("auto", "p2p", "nccl"):
            raise ValueError("band_exchange must be 'auto', 'p2p' or 'nccl'")
        if mode == "nccl":
            return "nccl"
        world, rank = dist.get_world_size(self.group), dist.get_rank(self.group)
        ok, err = 1, None
        try:
            import torch.distributed._symmetric_memory as symm
            n = N.BAND_PARITIES * world * N.BAND_SLOT
            box = symm.empty(n, dtype=torch.float64, device=self.device)
            box.zero_()
            hdl = symm.rendezvous(box, self.group)
            ptrs = [int(p) for p in hdl.buffer_ptrs]
            if len(ptrs) != world or not all(ptrs):
                raise RuntimeError("symmetric memory returned no peer pointers")
            self._inbox, self._inbox_hdl = box, hdl
            self._inbox_ptrs = torch.tensor(ptrs, dtype=torch.int64, device=self.device)
            self._xrank, self._xworld = rank, world
        except Exception as e:           # no peer mapping on this platform: the NCCL form of the same exchange
            ok, err = 0, e
        flag = torch.tensor([ok], device=self.device, dtype=torch.int32)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=self.group)       # all ranks take the same path
        torch.cuda.synchronize()
        if int(flag.item()) == 1:
            return "p2p"
        if mode == "p2p":
            raise RuntimeError("peer-memory band exchange not available: %r" % (err,))
        return "nccl"

    # ------------------------------------------------------------------ workspace
    def _workspace(self, ncol, max_iter, slot=0):
        """Per-slot scratch: iteration trajectory, the status block on the device and its pinned host
        copy, one event.  Timesteps in flight on different streams must use different slots."""
        key = (ncol, max_iter, slot)
        ws = self._ws.get(key)
        if ws is None:
            self._ws = {k: v for k, v in self._ws.items() if k[:2] == (ncol, max_iter)}
            ws = dict(
                traj=torch.empty((max_iter, ncol), device=self.device, dtype=torch.float32),
                status=torch.zeros(_STATUS_BYTES, device=self.device, dtype=torch.uint8),
                status_host=torch.zeros(_STATUS_BYTES, dtype=torch.uint8, pin_memory=True),
                event=torch.cuda.Event(), inflight=None,
            )
            if self.group is not None:
                ws["band_words"] = torch.zeros(N.BAND_WORDS, device=self.device, dtype=torch.float64)
            self._ws[key] = ws
        return ws

    def alloc_outputs(self, ny, nx, nsoil):
        e = lambda *s: torch.empty(s, device=self.device, dtype=torch.float32)
        L = self.nlev
        return dict(PS=e(1, ny, nx), T_SKIN=e(1, ny, nx), FR_SEA_ICE=e(1, ny, nx), T_SO=e(1, nsoil, ny, nx),
                    T=e(1, L, ny, nx), QV=e(1, L, ny, nx), U=e(1, L, ny, nx), V=e(1, L, ny, nx),
                    delta_ps=e(1, ny, nx))

    # ------------------------------------------------------------------ submit
    def submit(self, era, era_step_dt, out=None, ignore_top_pressure_error=False, k_spec=None,
               file_name="<memory>", slot=0, direct=False):
        """
        Enqueue one timestep on the current CUDA stream.  ``era``: float32 CUDA
        tensors PS, FIS, FR_LAND, FR_SEA_ICE, T_SKIN [1,ny,nx], T_SO [1,S,ny,nx],
        T, QV, U, V [1,L,ny,nx] (the names of settings.var_name_map).  Returns a
        ``Pending``; nothing is synchronised here.
        """
        msg = fused_refusal()
        if msg is not None:
            raise ValueError(msg)
        a, f, out, ws, k_spec, k_max = self._fill_args(era, era_step_dt, out, k_spec, slot)
        if direct:
            a.flags |= N.FLAG_DIRECT          # every parked level integrated in every iteration
        if ws["inflight"] is not None:        # the slot's pinned status block is about to be reused
            ws["inflight"].snapshot()
        st = _stream()
        sdev, shost = C.c_void_p(ws["status"].data_ptr()), C.c_void_p(ws["status_host"].data_ptr())
        if self.kernel_events is not None:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
        if self.group is None and self.kernel_events is None:
            # init, column kernel, convergence scan, rewrite and the status copy in one call
            N.check(N.lib.pgw_timestep_run(C.byref(a), sdev, shost, 0, st), "pgw_timestep_run")
        else:
            N.check(N.lib.pgw_timestep_run(C.byref(a), sdev, None, N.RUN_NO_FINALIZE, st), "pgw_timestep_run")
            if self.kernel_events is not None:
                e1.record()
                self.kernel_events.append((e0, e1))
            if self.group is not None:
                # latitude-band mode: the stopping rule is global over all bands (step_03:189,308).  ONE
                # collective merges the whole status block: max error per iteration, error bits, minima.
                if self.band_exchange == "p2p":
                    self._xseq += 1
                    N.check(N.lib.pgw_band_exchange(sdev, C.c_void_p(self._inbox_ptrs.data_ptr()), self._xrank,
                                                    self._xworld, self._xseq, 20.0, st), "pgw_band_exchange")
                    self.stats["launches"] += 1
                else:
                    import torch.distributed as dist
                    w = ws["band_words"]
                    N.check(N.lib.pgw_band_pack(sdev, C.c_void_p(w.data_ptr()), st), "pgw_band_pack")
                    dist.all_reduce(w, op=dist.ReduceOp.MAX, group=self.group)
                    N.check(N.lib.pgw_band_unpack(C.c_void_p(w.data_ptr()), sdev, st), "pgw_band_unpack")
                    self.stats["launches"] += 2
            N.check(N.lib.pgw_timestep_finish(C.byref(a), sdev, shost, st), "pgw_timestep_finish")
        self.stats["launches"] += 4
        ws["event"].record()
        self.deltas.hold(torch.cuda.current_stream())      # a streamed set keeps this timestep's stamps until here
        ctx = dict(era=era, when=era_step_dt, ignore_top=ignore_top_pressure_error, k_spec=k_spec,
                   k_max=k_max, keep=(f, a), file_name=file_name, slot=slot, direct=direct,
                   stream=torch.cuda.current_stream(), local_pref=bool(a.flags & N.FLAG_LOCAL_PREF))
        p = Pending(self, a, out, ws, ctx)
        ws["inflight"] = p
        return p

    def _fill_args(self, era, era_step_dt, out=None, k_spec=None, slot=0):
        """Validate the ERA5 fields and fill a ``pgw_timestep_args`` for them.  Returns
        (args, input tensors, outputs, workspace, k_spec, k_max)."""
        ds = self.deltas
        ny, nx = era["PS"].shape[-2:]
        ncol = ny * nx
        if ncol != ds.ncol:
            raise ValueError("Lat dimension of input files is inconsistent!" if ny != ds.shape2d[0]
                             else "Lon dimension of input files is inconsistent!")
        L = self.nlev
        nsoil = len(self.soil_decay)
        f = {}
        for name, lev in (("PS", 1), ("FIS", 1), ("FR_LAND", 1), ("FR_SEA_ICE", 1), ("T_SKIN", 1),
                          ("T_SO", nsoil), ("T", L), ("QV", L), ("U", L), ("V", L)):
            if lev == 0:
                continue
            t = era[name]
            if t.device != self.device or t.dtype != torch.float32 or not t.is_contiguous():
                t = t.to(self.device, torch.float32).contiguous()
            if t.numel() != lev * ncol:
                raise ValueError("field %s has %d values, expected %d" % (name, t.numel(), lev * ncol))
            f[name] = t
        if out is None:
            out = self.alloc_outputs(ny, nx, nsoil)
        max_iter = int(settings.max_n_iter)
        k_max = max(1, min(max_iter - 1, N.PGW_MAX_ITER))
        if k_spec is None:
            k_spec = self.k_pred
        k_spec = max(1, min(int(k_spec), k_max))
        ws = self._workspace(ncol, k_max, slot)

        zg = ds.vars["zg"]
        local = settings.p_ref_inp is None                                # level picked per column and iteration
        if local:
            sel0, p_ref_scalar = 0, float(zg["plev"][0])
            if "p_ref" not in out:
                out["p_ref"] = torch.empty((1, ny, nx), device=self.device, dtype=torch.float64)
        else:
            p_ref_scalar = float(settings.p_ref_inp)
            sel0 = self._zg_level.get(p_ref_scalar)
            if sel0 is None:
                sel = np.nonzero(zg["plev"] == p_ref_scalar)[0]           # .sel(plev=p_ref), step_03:294
                if len(sel) != 1:
                    raise KeyError(p_ref_scalar)
                sel0 = self._zg_level[p_ref_scalar] = int(sel[0])

        # everything that does not change from one timestep to the next on this slot is filled once
        in_names = ("PS", "FIS", "FR_LAND", "FR_SEA_ICE", "T_SKIN", "T", "QV", "U", "V")
        out_names = ("PS", "T_SKIN", "FR_SEA_ICE", "T", "QV", "U", "V")
        key = (tuple(f[n].data_ptr() for n in in_names), f["T_SO"].data_ptr() if nsoil else 0,
               tuple(out[n].data_ptr() for n in out_names), out["T_SO"].data_ptr() if nsoil else 0,
               out["delta_ps"].data_ptr(), ncol)
        if ws.get("args_key") != key:
            t = N.TimestepArgs()
            t.ncol, t.nlev, t.nplev, t.nsoil = ncol, L, len(ds.plev), nsoil
            t.plev_descending = int(ds.plev_descending)
            t.ak, t.bk, t.akm, t.bkm = (self.ak_d.data_ptr(), self.bk_d.data_ptr(), self.akm_d.data_ptr(),
                                        self.bkm_d.data_ptr())
            t.plev = ds.plev_dev.data_ptr()
            t.ak_host, t.bk_host = self.ak.ctypes.data, self.bk.ctypes.data
            t.akm_host, t.bkm_host = self.akm.ctypes.data, self.bkm.ctypes.data
            for name in in_names:
                setattr(t, name, f[name].data_ptr())
            t.T_SO = f["T_SO"].data_ptr() if nsoil else 0
            t.ts_clim = ds.ts_clim.data_ptr()
            for i, v in enumerate(self.soil_decay):
                t.soil_decay[i] = float(v)
            t.PS_out, t.T_SKIN_out, t.FR_SEA_ICE_out = (out["PS"].data_ptr(), out["T_SKIN"].data_ptr(),
                                                        out["FR_SEA_ICE"].data_ptr())
            t.T_SO_out = out["T_SO"].data_ptr() if nsoil else 0
            t.T_out, t.QV_out, t.U_out, t.V_out = (out["T"].data_ptr(), out["QV"].data_ptr(),
                                                   out["U"].data_ptr(), out["V"].data_ptr())
            t.dps_out = out["delta_ps"].data_ptr()
            t.dps_traj = ws["traj"].data_ptr()
            base = ws["status"].data_ptr()
            S = N.TimestepStatus
            t.maxerr = base + S.maxerr.offset
            t.stats = base + S.stats.offset
            t.err = base + S.err.offset
            t.first_k = base + S.first_k.offset
            t.poly_fallback = base + S.poly_fallback.offset
            ws["args_key"], ws["args"] = key, t
        a = N.TimestepArgs.from_buffer_copy(ws["args"])
        a.d4 = ds.slab4(era_step_dt)
        for name in ("tas", "hurs", "ps_hist", "ts", "tos", "siconc"):
            setattr(a, name, ds.slab(name, era_step_dt))
        a.zg_ref = ds.slab("zg", era_step_dt, level=sel0)
        a.p_ref = p_ref_scalar
        a.adj_factor = float(settings.adj_factor)
        a.thresh_phi_ref_max_error = float(settings.thresh_phi_ref_max_error)
        a.k_spec = k_spec
        a.ps_bound = self.ps_bound
        a.flags = N.FLAG_REF_DTYPES if getattr(settings, "i_reference_dtypes", 0) else 0
        if settings.i_reinterp:
            a.flags |= N.FLAG_REINTERP        # re-interpolate the ERA state every iteration (step_03:202-216)
        if local:
            if self._zg_tables is None:
                plev = np.ascontiguousarray(zg["plev"], dtype=np.float64)
                if len(np.unique(plev)) != len(plev):
                    raise ValueError("zg pressure levels must be distinct")
                self._zg_tables = (plev, torch.as_tensor(plev, device=self.device))
            plev, plev_d = self._zg_tables
            a.flags |= N.FLAG_LOCAL_PREF
            a.zg = ds.slab("zg", era_step_dt)
            a.zg_plev, a.zg_plev_host, a.nzg = plev_d.data_ptr(), plev.ctypes.data, len(plev)
            a.p_floor = self.p_floor
            if "pref_traj" not in ws:
                ws["pref_traj"] = torch.empty(ws["traj"].shape, device=self.device, dtype=torch.uint8)
            a.pref_traj = ws["pref_traj"].data_ptr()
            a.p_ref_out = out["p_ref"].data_ptr()
        return a, f, out, ws, k_spec, k_max

    # ------------------------------------------------------------------ completion
    def _complete(self, p):
        st = p.snapshot()
        maxerr = np.frombuffer(st.maxerr, dtype=np.float64)
        n_iter, converged, rewritten = st.result.n_iter, st.result.converged, st.result.rewritten
        min_targ_p, min_src_p = float(st.stats[0]), float(st.stats[1])
        err = int(st.err)
        ctx = p.ctx
        # The kernel runs k_spec iterations for every column; the reference stops after N.  A ps-dependent
        # condition that only fired in an iteration the reference never ran did not happen there.
        n_ran = int(n_iter) if converged else ctx["k_spec"]
        if (err & N.ERR_PREF_BELOW_SFC) and st.first_k[0] >= n_ran:
            err &= ~N.ERR_PREF_BELOW_SFC
        if (err & N.ERR_PS_BOUND) and st.first_k[1] >= n_ran:
            err &= ~N.ERR_PS_BOUND
        if (err & N.ERR_NO_PREF) and st.first_k[2] >= n_ran:
            err &= ~N.ERR_NO_PREF
        if (err & N.ERR_PREF_FLOOR) and st.first_k[3] >= n_ran:
            err &= ~N.ERR_PREF_FLOOR
        # a column that left the stash computes garbage from then on, which can end in NO_PREF later: rerun first
        k_stash = min(st.first_k[1] if err & N.ERR_PS_BOUND else N.INT32_MAX,
                      st.first_k[3] if err & N.ERR_PREF_FLOOR else N.INT32_MAX)
        if (err & N.ERR_NO_PREF) and st.first_k[2] > k_stash:
            err &= ~N.ERR_NO_PREF
        if err & N.ERR_BAND_TIMEOUT:
            raise RuntimeError("latitude-band exchange: the status block of a peer rank did not arrive")
        if err & N.ERR_PS_HIST_RANGE:
            raise ValueError()                                           # functions.py:360-361
        if (min_targ_p < min_src_p or min_targ_p < float(np.min(self.deltas.plev))) \
                and not ctx["ignore_top"]:
            raise ValueError(MSG_TOP)                                    # functions.py:417-425
        if err & N.ERR_NO_PREF:
            from .staged import MSG_NO_PREF
            raise ValueError(MSG_NO_PREF)                                # step_03:245-251
        if err & N.ERR_PREF_BELOW_SFC:
            raise ValueError(MSG_PREF)                                   # functions.py:162-165
        if err & (N.ERR_PS_BOUND | N.ERR_PREF_FLOOR):
            if err & N.ERR_PS_BOUND:
                self.ps_bound *= 1.25
            if err & N.ERR_PREF_FLOOR:                                   # one more zg level into the stash
                below = self._zg_tables[0][self._zg_tables[0] < self.p_floor]
                self.p_floor = float(below.max()) if len(below) else 0.8 * self.p_floor
            self.stats["reruns"] += 1
            with torch.cuda.stream(ctx["stream"]):       # a rerun goes where the timestep was submitted
                return self.submit(ctx["era"], ctx["when"], out=p.out, ignore_top_pressure_error=ctx["ignore_top"],
                               k_spec=ctx["k_spec"], file_name=ctx["file_name"], slot=ctx["slot"],
                               direct=ctx["direct"]).result()
        if not converged:
            if ctx["k_spec"] >= ctx["k_max"]:
                raise ValueError(MSG_NOCONV.format(ctx["file_name"]))   # step_03:315-319
            self.stats["reruns"] += 1
            with torch.cuda.stream(ctx["stream"]):
                return self.submit(ctx["era"], ctx["when"], out=p.out, ignore_top_pressure_error=ctx["ignore_top"],
                               k_spec=ctx["k_max"], file_name=ctx["file_name"], slot=ctx["slot"],
                               direct=ctx["direct"]).result()
        # predict the largest recent count: one iteration too many costs a cheap rewrite
        # (+13 % traffic), one too few a full rerun
        self._n_hist = (self._n_hist + [int(n_iter)])[-4:]
        self.k_pred = max(self._n_hist)
        self.stats["timesteps"] += 1
        self.stats["rewrites"] += int(rewritten)
        res = dict(p.out)
        res["n_iter"] = int(n_iter)
        res["phi_max_errors"] = [float(x) for x in maxerr[:int(n_iter)]]
        res["poly_fallback"] = int(st.poly_fallback)
        if not ctx.get("local_pref"):
            res.pop("p_ref", None)
        if settings.i_debug >= 2:
            for it, e in enumerate(res["phi_max_errors"], 1):
                print("### iteration {:03d}, phi max error: {}".format(it, e))
        return res

    def apply(self, era, era_step_dt, **kw):
        """Synchronous form of ``submit``: returns the output dict (device tensors).  i_reinterp = 1 and
        p_ref_inp = None take the staged path (``submit`` runs each of them, though not both together, in
        the fused pass)."""
        if settings.i_reinterp or settings.p_ref_inp is None:
            from . import staged
            kw.pop("k_spec", None)
            kw.pop("slot", None)
            return staged.apply_staged(self, era, era_step_dt, **kw)
        return self.submit(era, era_step_dt, **kw).result()

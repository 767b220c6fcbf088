"""
Work partitioning over GPUs and the reference-compatible ``IterMP`` driver.

The reference parallelises over ERA5 files with a process pool (parallel.py:12-68,
one file = one timestep = one task).  Here one process drives one B200:
  * many timesteps: rank r takes timesteps r, r+W, ... (``timesteps_for_rank``);
    the only collective is one NCCL broadcast of the delta climatology
    (``broadcast_deltas``);
  * a single snapshot: contiguous latitude bands (``split_rows``); the
    field-global stopping rule of the ps iteration then needs a MAX all-reduce of
    the per-iteration error vector (done inside ``PGWEngine.submit`` when the
    engine is given a process group).
``IterMP`` keeps the reference's call signature; tasks run in this process on
the current GPU (njobs == 1) or in ``njobs`` spawned workers, worker i bound to
GPU i % device_count.
"""
import multiprocessing as mp
import os


def split_rows(ny, world):
    """Contiguous latitude bands: the first ``world-1`` ranks get ny // world rows,
    the last one the remainder (721 rows on 8 ranks -> 7 x 90 + 91)."""
    base = ny // world
    bounds = []
    for r in range(world):
        start = r * base
        stop = ny if r == world - 1 else (r + 1) * base
        bounds.append((start, stop))
    return bounds


def timesteps_for_rank(n_steps, rank, world):
    """Round-robin assignment of independent timesteps to ranks."""
    return list(range(rank, n_steps, world))


def decide_n_iter(maxerr, thresh):
    """First iteration count N with max|phi error| <= thresh (step_03_apply_to_era.py:189,308),
    or 0 if none of the recorded iterations converged.  Host mirror of the device-side scan,
    used on the merged (all-reduced) error vector."""
    for k, e in enumerate(maxerr):
        if not (e > thresh):
            return k + 1
    return 0


def broadcast_deltas(deltas, src=0, group=None, info=None):
    """NCCL-broadcast the climatology of a ``DeltaSet`` from ``src`` -- ONE collective over its arena, after a
    one-element collective that makes NCCL set up its communicator and channels outside the timing.  Returns
    the elapsed ms of the broadcast itself; ``info`` (a dict) also receives bytes and GB/s."""
    import torch
    import torch.distributed as dist
    if getattr(deltas, "streamed", False):
        raise ValueError("a streamed delta set cannot be broadcast: every rank reads the delta files itself")
    warm = torch.zeros(1, device=deltas.device)
    dist.broadcast(warm, src=src, group=group)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    nbytes = 0
    for t in deltas.tensors():
        dist.broadcast(t, src=src, group=group)
        nbytes += t.numel() * t.element_size()
    e1.record()
    torch.cuda.synchronize()
    deltas.refresh_derived()
    ms = e0.elapsed_time(e1)
    if info is not None:
        info.update(bytes=nbytes, ms=ms, gb_per_s=nbytes / ms / 1e6 if ms > 0 else None, collectives=len(deltas.tensors()))
    return ms


def regrid_banded(data, lat_gcm, lon_gcm, targ_lat, targ_lon, group=None, src=0, gather=True, smooth=False,
                  device=None, regrid_fn=None):
    """
    step_02 for ONE variable on all GPUs of ``group`` (SURVEY.md 8e, third row): the source field on the GCM grid
    is replicated (NCCL broadcast from ``src``: 1.8 GB for a daily 3-D variable), every rank regrids its own band
    of TARGET latitudes (``split_rows``; the tables are those of the whole grid, the pole-row zonal means are
    computed on every rank) and, with ``smooth``, first smooths the annual cycle of the whole source field
    itself (1 ms on one B200: replicating that work is cheaper than any exchange of its result).  Returns
    ``(band, (r0, r1), whole)``: this rank's rows [.., r1 - r0, nx] as a CUDA tensor, its row range, and -- with
    ``gather`` -- the whole regridded field on rank ``src`` (None elsewhere), collected with one NCCL gather
    of the bands.  ``data``: array / tensor holding the field on ``src``; on the other ranks anything of the same
    shape (the broadcast overwrites it).  ``device`` / ``regrid_fn`` exist for the CPU (gloo) test of the
    exchange logic; the product path is CUDA + ``functions.regrid_arrays``.
    """
    import torch
    import torch.distributed as dist
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
    if regrid_fn is None:
        from . import functions as F
        regrid_fn = F.regrid_arrays
    d = torch.as_tensor(data).to(dev, torch.float32).contiguous() if not isinstance(data, torch.Tensor) \
        else data.to(dev, torch.float32).contiguous()
    dist.broadcast(d, src=src, group=group)
    if smooth:
        from . import functions as F
        d = F.smooth_annual_cycle(d)
        if not isinstance(d, torch.Tensor):
            d = torch.as_tensor(d, device=dev)
    ny_t = len(targ_lat)
    bounds = split_rows(ny_t, world)
    r0, r1 = bounds[rank]
    band = regrid_fn(d, lat_gcm, lon_gcm, targ_lat, targ_lon, rows=(r0, r1))
    whole = None
    if gather:
        lead, nx_t = tuple(band.shape[:-2]), band.shape[-1]
        # bands differ in their number of rows (721 = 7 x 90 + 91): gather equal-sized, row-major-in-band pieces
        hmax = max(b - a for a, b in bounds)
        piece = torch.zeros((hmax,) + lead + (nx_t,), device=dev, dtype=torch.float32)
        piece[:r1 - r0] = band.movedim(-2, 0)
        pieces = [torch.empty_like(piece) for _ in range(world)] if rank == src else None
        dist.gather(piece, pieces, dst=src, group=group)
        if rank == src:
            whole = torch.empty(lead + (ny_t, nx_t), device=dev, dtype=torch.float32)
            for (a, b), pc in zip(bounds, pieces):
                whole[..., a:b, :] = pc[:b - a].movedim(0, -2)
    return band, (r0, r1), whole


def _parse_cpulist(text):
    cpus = set()
    for part in text.strip().split(","):
        if not part:
            continue
        lo, _, hi = part.partition("-")
        cpus.update(range(int(lo), int(hi or lo) + 1))
    return cpus


def bind_to_gpu_numa(device_index):
    """Pin this process to the CPUs of the NUMA node the GPU hangs off, BEFORE any pinned host buffer is
    allocated: the staging buffers of the host pipeline are then node-local to the GPU's PCIe root, which is
    what lets N processes stream over N PCIe links without meeting on the inter-socket link.  Returns the
    node (or None when the topology is not exposed; nothing is changed then)."""
    try:
        import torch
        p = torch.cuda.get_device_properties(device_index)
        bdf = "%04x:%02x:%02x.0" % (p.pci_domain_id, p.pci_bus_id, p.pci_device_id)
        with open("/sys/bus/pci/devices/%s/numa_node" % bdf) as f:
            node = int(f.read().strip())
        if node < 0:
            return None
        with open("/sys/devices/system/node/node%d/cpulist" % node) as f:
            cpus = _parse_cpulist(f.read())
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return node
    except (OSError, AttributeError, ValueError, RuntimeError):
        return None


def _init_worker(counter):
    """Pool initializer: every worker process takes ONE GPU (worker index % device_count) for its whole
    lifetime -- whichever tasks the pool hands it later -- and binds to that GPU's NUMA node."""
    with counter.get_lock():
        idx = counter.value
        counter.value += 1
    if os.environ.get("PGW_ITERMP_NO_GPU"):       # CPU-only tasks (bench.py's reference arm)
        return
    try:
        import torch
        if torch.cuda.is_available():
            dev = idx % torch.cuda.device_count()
            torch.cuda.set_device(dev)
            bind_to_gpu_numa(dev)
    except ImportError:
        pass


def _worker(payload):
    func, kwargs = payload
    return func(**kwargs)


class IterMP:
    """Same interface as the reference's ``IterMP`` (parallel.py:36-68):
    ``IterMP(njobs, run_async).run(func, fargs, step_args)`` then ``.output``."""

    def __init__(self, njobs=None, run_async=False, start_method="spawn", quiet=False):
        """``start_method``/``quiet`` are not in the reference: workers that use a GPU must be spawned (a forked
        child cannot use CUDA); CPU-only tasks may fork."""
        self.run_async = run_async
        self.njobs = 1 if njobs is None else int(njobs)
        self.start_method = start_method
        if not quiet:
            print('IterMP: njobs = ' + str(self.njobs))
        self.output = None

    def run(self, func, fargs={}, step_args=None):
        tasks = []
        for i in range(len(step_args)):
            kw = dict(fargs)
            kw.update(step_args[i])
            tasks.append(kw)
        if self.njobs > 1:
            ctx = mp.get_context(self.start_method)
            with ctx.Pool(processes=self.njobs, initializer=_init_worker, initargs=(ctx.Value("i", 0),)) as pool:
                payload = [(func, kw) for kw in tasks]
                if self.run_async:
                    self.output = pool.map_async(_worker, payload).get()
                else:
                    self.output = pool.map(_worker, payload)
        else:
            self.output = [func(**kw) for kw in tasks]

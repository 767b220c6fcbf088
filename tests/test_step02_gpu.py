"""The step_02 kernels (pgw_step02.cu, pgw_nanterp.cu) at production shapes and on fields that contain NaN.

Bilinear regridding is compared bit for bit with the one-thread-per-output ``regrid_kernel``
(``PGW_REGRID_PATH=generic``) on every element: all regridding kernels evaluate the same float64 expressions.
Every kernel is also compared with the float64 oracle, run on slices of fields or points to keep host memory and
time small (each oracle operation is independent across fields and points, so slicing changes nothing): for
regridding a spread of fields, for smoothing every NaN series with its neighbours in all grid-stride passes and a
sample of each pass (the NaN mask is checked on every point), for ocean regridding every field.  ``regrid_plan`` restates on the
host which kernel and which specialised body a grid pair runs, so a later edit of a grid cannot move a case
silently onto another body."""
import numpy as np
import pytest
import torch

from oracle import pgw_oracle as O
from test_ops_gpu import _regrid_with

pytestmark = pytest.mark.gpu

# pgw_step02.cu: kRegridChunk, kRegridSrcRows, the walk kernel's CTA size and grid cap, the smoothing grid cap
CHUNK, SRC_ROWS, WALK_THREADS, WALK_CTAS = 32, 10, 384, 148 * 5
SMOOTH_STRIDE = 148 * 8 * 128

ERA_LAT, ERA_LON = np.linspace(-90, 90, 721), 0.25 * np.arange(1440)
DEG1_LAT = np.linspace(-89.5, 89.5, 180)


@pytest.fixture(scope="module")
def F():
    from pgw4era5_b200 import functions
    return functions


def regrid_plan(tb, nx_s, rows=None):
    """The kernel pgw_regrid_bilinear_band_f32 launches for the tables ``tb`` of ``F.regrid_tables`` and the body
    that kernel runs (pgw_step02.cu:580-610 and :423-449), for a 16-byte aligned destination.  Returns
    dict(kernel="walk" | "generic", vec=4 | 1, n1=1..4 for the three-column bodies, 0 for the general body,
    staged=[per chunk: its source rows are staged in shared memory (True) or read from global memory (False)])."""
    ny_t, nx_t = len(tb["wy"]), len(tb["wx"])
    r0, r1 = (0, ny_t) if rows is None else rows
    vec = 4 if nx_t % 4 == 0 else 1
    nchunk = -(-(r1 - r0) // CHUNK)
    if nx_t // vec > WALK_THREADS or nx_s > WALK_THREADS or nchunk > 4096:
        return dict(kernel="generic", vec=vec, n1=None, staged=None)
    # three-column pattern: the first n1 targets of a thread bracket (u0, u1), the rest (u1, u2); n1 equal for all
    n1_of, pattern = [], True
    for t in range(nx_t // vec):
        ia, ib = tb["i0"][t * vec:(t + 1) * vec], tb["i1"][t * vec:(t + 1) * vec]
        u0, u1, u2 = ia[0], ib[0], ib[-1]
        n1 = 0
        for v in range(vec):
            if ia[v] == u0 and ib[v] == u1 and n1 == v:
                n1 = v + 1
            elif not (ia[v] == u1 and ib[v] == u2):
                pattern = False
        n1_of.append(n1)
    uniform = pattern and len(set(n1_of)) == 1
    staged = []
    for c in range(nchunk):
        sl = slice(r0 + c * CHUNK, min(r0 + (c + 1) * CHUNK, r1))
        js = np.concatenate([tb["j0"][sl], tb["j1"][sl]])
        js = js[js >= 0]                                     # negative: a pole row, always in shared memory
        staged.append(bool(len(js) == 0 or js.max() - js.min() + 1 <= SRC_ROWS))
    return dict(kernel="walk", vec=vec, n1=n1_of[0] if uniform and vec == 4 else 0, staged=staged)


def _items_per_cta(nfield, nrow):
    nitem = nfield * -(-nrow // CHUNK)
    return nitem // min(nitem, WALK_CTAS)


def assert_same_bits(a, b):
    """Bit identity of two float32 device tensors; NaN at the same places."""
    assert a.shape == b.shape
    na, nb = torch.isnan(a), torch.isnan(b)
    assert torch.equal(na, nb), "NaN masks differ in %d elements" % int((na != nb).sum())
    ai, bi = a.masked_fill(na, 0).view(torch.int32), b.masked_fill(nb, 0).view(torch.int32)
    assert torch.equal(ai, bi), "%d elements differ" % int((ai != bi).sum())


def assert_regrid_oracle(out, data, lat, lon, tlat, tlon, fields, rows=None):
    """The float64 oracle on the fields ``fields`` (rows ``rows`` of the target), NaN masks exact, values to 5e-7."""
    r0, r1 = (0, len(tlat)) if rows is None else rows
    for f in fields:
        ref = O.regrid_lat_lon(data[f:f + 1], lat, lon, tlat, tlon)[0, r0:r1]
        got = out[f].cpu().numpy()
        np.testing.assert_array_equal(np.isnan(got), np.isnan(ref), err_msg="NaN mask of field %d" % f)
        np.testing.assert_allclose(got, ref, rtol=0, atol=5e-7, equal_nan=True, err_msg="field %d" % f)


def _sample_fields(nfield):
    return sorted({0, 1, nfield // 3, nfield // 2, (2 * nfield) // 3, nfield - 2, nfield - 1})


def _normal_fields(seed, nfield, ny, nx):
    return np.random.default_rng(seed).normal(size=(nfield, ny, nx)).astype(np.float32)


# --------------------------------------------------------------------------------------------------------------
# A. bilinear regridding
# --------------------------------------------------------------------------------------------------------------
BODY_CASES = {
    # 1 degree sources on the ERA5 target: the longitude offset alone picks the body
    "n1_1": (DEG1_LAT, 0.1 + np.arange(360), ERA_LAT, ERA_LON, 100, (4, 1)),
    "n1_2": (DEG1_LAT, 0.25 + np.arange(360), ERA_LAT, ERA_LON, 100, (4, 2)),
    "n1_3": (DEG1_LAT, 0.5 + np.arange(360), ERA_LAT, ERA_LON, 100, (4, 3)),
    "n1_4": (DEG1_LAT, 0.75 + np.arange(360), ERA_LAT, ERA_LON, 100, (4, 4)),
    "general": (DEG1_LAT, np.arange(360.0), ERA_LAT, ERA_LON, 100, (4, 0)),
    # the 201 x 281 European target: odd width, scalar stores
    "vec1": (DEG1_LAT, 0.5 + np.arange(360), 30 + 0.25 * np.arange(201), -20 + 0.25 * np.arange(281), 320, (1, 0)),
}


@pytest.mark.parametrize("case", list(BODY_CASES))
def test_walk_bodies_many_items_per_cta(F, case):
    """Every body of regrid_walk_kernel with at least 3 (field, chunk) items per CTA: the cp.async prefetch into the
    other half of the source rows, the pole means carried from item to item and the table parity across items,
    with the 17-row last chunk of the 721 ERA5 rows.  Also the 8-GPU split of ``parallel.split_rows``: bands of
    about 90 rows whose edges cut chunks and 4-row groups concatenate bit for bit to the whole field."""
    from pgw4era5_b200.parallel import split_rows
    lat, lon, tlat, tlon, nfield, (vec, n1) = BODY_CASES[case]
    tb = F.regrid_tables(lat, lon, tlat, tlon)
    plan = regrid_plan(tb, len(lon))
    assert (plan["kernel"], plan["vec"], plan["n1"]) == ("walk", vec, n1)
    assert all(plan["staged"])
    assert _items_per_cta(nfield, len(tlat)) >= 3
    data = _normal_fields(40 + n1 + vec, nfield, len(lat), len(lon))
    d = torch.from_numpy(data).cuda()
    walk = F.regrid_arrays(d, lat, lon, tlat, tlon)
    assert_same_bits(walk, _regrid_with("generic", F, d, lat, lon, tlat, tlon))
    assert not torch.isnan(walk).any()
    assert_regrid_oracle(walk, data, lat, lon, tlat, tlon, _sample_fields(nfield))
    bounds = split_rows(len(tlat), 8)
    parts = []
    for r0, r1 in bounds:
        p = regrid_plan(tb, len(lon), rows=(r0, r1))
        assert (p["kernel"], p["vec"], p["n1"]) == ("walk", vec, n1)
        parts.append(F.regrid_arrays(d, lat, lon, tlat, tlon, rows=(r0, r1)))
    assert_same_bits(torch.cat(parts, dim=-2), walk)


@pytest.mark.parametrize("poles,n_unstaged", [("exact", 10), ("inner", 4)])
def test_walk_staged_and_unstaged_chunks_interleaved(F, poles, n_unstaged):
    """A CESM-like 192 x 288 source (0.94 degree) on the ERA5 target: chunks whose 32 target rows span more
    than kRegridSrcRows source rows read global memory, the others are staged, and every CTA walks through both
    kinds over many items.

    With rows at exactly -90 and 90 ("exact") the -90 row and the added south-pole row share a latitude, so
    ``_interp_table`` gives the first target row a 0/0 weight and that whole row comes out NaN.  scipy's
    ``_call_linear``, which the reference uses, does the same and so does the oracle: this pins the NaN row as
    parity with the reference, not as a defect to fix on one side only."""
    lat = np.linspace(-90, 90, 192) if poles == "exact" else np.linspace(-89.5, 89.5, 192)
    lon = 1.25 * np.arange(288)
    tb = F.regrid_tables(lat, lon, ERA_LAT, ERA_LON)
    plan = regrid_plan(tb, len(lon))
    assert plan["kernel"] == "walk" and plan["vec"] == 4
    assert len(plan["staged"]) == 23 and plan["staged"].count(False) == n_unstaged
    nfield = 100
    assert _items_per_cta(nfield, len(ERA_LAT)) >= 3
    data = _normal_fields(50 + n_unstaged, nfield, len(lat), len(lon))
    d = torch.from_numpy(data).cuda()
    walk = F.regrid_arrays(d, lat, lon, ERA_LAT, ERA_LON)
    assert_same_bits(walk, _regrid_with("generic", F, d, lat, lon, ERA_LAT, ERA_LON))
    assert_regrid_oracle(walk, data, lat, lon, ERA_LAT, ERA_LON, _sample_fields(nfield))
    nan_rows = torch.isnan(walk).all(dim=-1).all(dim=0).nonzero().flatten().tolist()
    assert nan_rows == ([0] if poles == "exact" else [])
    assert torch.isnan(walk).sum() == (nfield * len(ERA_LON) if poles == "exact" else 0)


def test_regrid_kernel_fallback_whole_and_banded(F):
    """A 0.5 degree source (nx_s = 720 > 384) on the ERA5 target runs regrid_kernel without being forced, and with
    ``rows=`` bands it takes the branch that shifts the row tables; the bands concatenate bit for bit."""
    from pgw4era5_b200.parallel import split_rows
    lat, lon = np.linspace(-89.75, 89.75, 360), 0.25 + 0.5 * np.arange(720)
    tb = F.regrid_tables(lat, lon, ERA_LAT, ERA_LON)
    assert regrid_plan(tb, len(lon))["kernel"] == "generic"
    bounds = split_rows(len(ERA_LAT), 8)
    assert all(regrid_plan(tb, len(lon), rows=b)["kernel"] == "generic" for b in bounds)
    nfield = 6
    data = _normal_fields(60, nfield, len(lat), len(lon))
    d = torch.from_numpy(data).cuda()
    whole = F.regrid_arrays(d, lat, lon, ERA_LAT, ERA_LON)
    parts = [F.regrid_arrays(d, lat, lon, ERA_LAT, ERA_LON, rows=b) for b in bounds]
    assert_same_bits(torch.cat(parts, dim=-2), whole)
    assert not torch.isnan(whole).any()
    assert_regrid_oracle(whole, data, lat, lon, ERA_LAT, ERA_LON, range(nfield))
    r0, r1 = bounds[3]
    assert_regrid_oracle(parts[3], data, lat, lon, ERA_LAT, ERA_LON, range(nfield), rows=(r0, r1))


def test_regrid_nan_in_source(F):
    """NaN in the source field, as in pressure-level ta/hur/ua/va below ground.  The pole rows are
    ``north[var].mean(dim=[lon])`` in the reference (functions.py:833-842), an xarray DataArray.mean, and
    xarray's reductions skip NaN for float data by default (skipna); oracle/xrlite.py restates that with
    np.nanmean.  So a partly missing first or last source row gives a pole row equal to the mean of its
    valid points, and the target rows between that pole and the row stay finite wherever the row is valid;
    an all-NaN row gives a NaN pole row.  Interior NaN spreads to the targets whose brackets touch it.
    Checked against the oracle and across the walk, row and generic kernels, with the NaN fields late in the
    item order of the walk kernel's CTAs."""
    lat, lon = DEG1_LAT, 0.5 + np.arange(360)
    tb = F.regrid_tables(lat, lon, ERA_LAT, ERA_LON)
    assert regrid_plan(tb, len(lon))["n1"] == 3
    nfield = 100
    data = _normal_fields(70, nfield, len(lat), len(lon))
    data[40, 60:63, 100:110] = np.nan                     # interior patches
    data[41, 90, 0:5] = np.nan
    data[41, 91, 355:360] = np.nan                        # across the periodic seam
    data[77, 0, 200:260] = np.nan                         # first row partly missing
    data[78, -1, 10:12] = np.nan                          # last row partly missing
    data[78, -1, 300] = np.nan
    data[99, 0, :] = np.nan                               # first row entirely missing
    d = torch.from_numpy(data).cuda()
    walk = F.regrid_arrays(d, lat, lon, ERA_LAT, ERA_LON)
    gen = _regrid_with("generic", F, d, lat, lon, ERA_LAT, ERA_LON)
    rows = _regrid_with("rows", F, d, lat, lon, ERA_LAT, ERA_LON)
    assert_same_bits(walk, gen)
    assert_same_bits(rows, gen)
    nan_fields = [40, 41, 77, 78, 99]
    assert_regrid_oracle(walk, data, lat, lon, ERA_LAT, ERA_LON, nan_fields + [0, 39, 42, 98])
    bad = torch.isnan(walk).flatten(1).any(dim=1).nonzero().flatten().tolist()
    assert bad == nan_fields
    w = walk.cpu().numpy()
    # partly missing pole-side rows: the rows between pole and source row stay finite where the row is valid
    for f, jt in ((77, [0, 1]), (78, [719, 720])):
        for j in jt:
            assert 0 < np.isnan(w[f, j]).sum() < len(ERA_LON) // 4, (f, j)
    # an all-NaN first row: NaN from the pole up to -88.5 (bracketed with that row), finite from -88.25 on
    assert np.isnan(w[99, :7]).all() and np.isfinite(w[99, 7:]).all()


# --------------------------------------------------------------------------------------------------------------
# B. smoothing of the annual cycle
# --------------------------------------------------------------------------------------------------------------
def _smooth_nan_points(nt, npoint):
    """(point, times) of the NaN placements: at t = 0, inside a ring group, only in the directly read tail
    (t >= 8 floor(nt / 8)), at t = nt - 1 and over a whole series.  Points in the first grid-stride pass (whose
    threads go on to later points), in the second pass and in the partial last pass."""
    last_pass = 2 * SMOOTH_STRIDE if npoint > 2 * SMOOTH_STRIDE else None
    second = SMOOTH_STRIDE if npoint > SMOOTH_STRIDE else None
    pick = lambda base, k, fallback: base + k if base is not None else fallback
    ngroup = nt // 8
    out = [(3, [0]),
           (pick(second, 1000, npoint // 2), [8 * (ngroup - 1) + 3]),
           (70, [8 * (ngroup - 1) + 5]),
           (200, [nt - 1]),
           (pick(last_pass, 76, npoint - 1), list(range(nt)))]
    if nt % 8:
        out.append((pick(last_pass, 10, npoint - 7), [8 * ngroup + (nt % 8) // 2]))
    return out


def _run_smoothing(F, nt, npoint, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn((nt, npoint), generator=g, device="cuda", dtype=torch.float32) + 3.0
    pts = _smooth_nan_points(nt, npoint)
    for p, ts in pts:
        x[ts, p] = float("nan")
    out = F.smooth_annual_cycle(x)
    assert out.shape == x.shape and out.dtype == torch.float32
    # NaN exactly for the series that hold one, the whole series; every other series finite
    bad = torch.isnan(x).any(dim=0)
    assert sorted(bad.nonzero().flatten().tolist()) == sorted(p for p, _ in pts)
    assert torch.equal(torch.isnan(out), bad.expand_as(out)), "NaN outside the series that contain one"
    # the oracle on the NaN series, their neighbours and a sample of every pass
    rng = np.random.default_rng(seed)
    idx = set(range(min(npoint, 512))) | set(rng.integers(0, npoint, 2048).tolist())
    for base in (SMOOTH_STRIDE, 2 * SMOOTH_STRIDE):
        idx |= set(range(base, min(base + 512, npoint)))
    for p, _ in pts:
        idx |= {q for q in range(p - 2, p + 3) if 0 <= q < npoint}
        idx |= {q for q in (p - SMOOTH_STRIDE, p + SMOOTH_STRIDE, p + 2 * SMOOTH_STRIDE) if 0 <= q < npoint}
    idx = torch.tensor(sorted(idx), device="cuda")
    ref = O.filter_data_fast(x[:, idx].cpu().numpy())
    got = out[:, idx].cpu().numpy()
    np.testing.assert_array_equal(np.isnan(got), np.isnan(ref))
    np.testing.assert_allclose(got, ref, rtol=0, atol=2e-6, equal_nan=True)


@pytest.mark.parametrize("nt", [8, 12, 15, 16, 17, 360, 365, 366])
def test_smoothing_many_points_per_thread(F, nt):
    """smooth_kernel's grid is capped at 148 * 8 CTAs of 128 threads: with 2 * 151 552 + 77 points every thread
    makes at least two passes and refills the cp.async ring for each point, and the last pass is partial.  nt < 16
    leaves fewer groups than the ring holds, 8, 16 and 360 leave no directly read tail."""
    npoint = 2 * SMOOTH_STRIDE + 77
    _run_smoothing(F, nt, npoint, seed=nt)


@pytest.mark.parametrize("nt", [1460, 4096])
def test_smoothing_long_series(F, nt):
    """6-hourly series (nt = 1460) need more than 48 KB of shared memory (the pgw_ensure_smem opt-in);
    nt = 4096 is the longest series that fits."""
    assert 8 * 6 * nt + 4 * 16 * 128 > 48 * 1024
    _run_smoothing(F, nt, 2999, seed=nt)


def test_smoothing_limits(F):
    from pgw4era5_b200._native import NativeError
    x = torch.ones((4097, 5), device="cuda")
    with pytest.raises(NativeError, match="shared memory"):
        F.smooth_annual_cycle(x)
    with pytest.raises(NativeError, match="invalid argument"):
        F.smooth_annual_cycle(torch.ones((7, 5), device="cuda"))


# --------------------------------------------------------------------------------------------------------------
# C. NaN-ignoring Gaussian-kernel regridding of ocean fields
# --------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("nfield", [13, 24, 25])
def test_ocean_regridding_more_fields_than_one_launch(F, nfield):
    """nan_ignoring_interp_arrays launches gauss_interp_kernel for at most 12 fields at a time; 13 and 25 fields
    leave a launch of one field.  The NaN masks differ from field to field on both sides of each boundary.  A
    target sits exactly on a source point that is NaN in fields 0, 12 and 24 and valid elsewhere: the exact hit
    locks per field, so the valid fields take that point's value and the others the Gaussian mean of the
    neighbours, as in the oracle."""
    rng = np.random.default_rng(nfield)
    nj, ni = 16, 32                                        # a coarse global curvilinear grid, 0..360, crosses 180
    glat, glon = np.meshgrid(np.linspace(-76, 86, nj), np.arange(ni) * 11.25 + 3.0, indexing="ij")
    glat = glat + 0.8 * np.sin(np.radians(glon) * 2)
    glon = np.mod(glon + 1.5 * np.cos(np.radians(glat) * 3), 360.0)
    tlat, tlon = np.linspace(-90, 90, 13), np.arange(0.0, 360.0, 20.0)
    radius = 2.0e6
    land_fr = ((rng.uniform(size=(len(tlat), len(tlon))) < 0.3) * rng.uniform(0.5, 1.0, (len(tlat), len(tlon)))).astype(np.float32)
    vals = (2.0 + np.cos(np.radians(glat)) + 0.3 * rng.normal(size=(nfield, nj, ni))).astype(np.float32)
    vals[:, rng.uniform(size=(nj, ni)) < 0.2] = np.nan                          # land
    vals[rng.uniform(size=vals.shape) < 0.08] = np.nan                          # field-dependent gaps
    vals[11][glat > 50] = np.nan                          # no source near the north pole: NaN targets there
    vals[nfield - 1][glat < -45] = np.nan                 # the single field of the last launch: none near the south
    a, b, j, i = 8, 12, 10, 21                            # target (30, 240) put exactly on source point (j, i)
    glat[j, i], glon[j, i] = tlat[a], tlon[b]
    land_fr[a, b] = 0.0
    holes = [f for f in (0, 12, 24) if f < nfield]
    vals[:, j, i] = 1.0 + 0.01 * np.arange(nfield)
    vals[holes, j, i] = np.nan
    out = F.nan_ignoring_interp_arrays(land_fr, tlat, tlon, vals, glat, glon, radius, 4.0)
    assert out.shape == (nfield, len(tlat), len(tlon)) and out.dtype == np.float64
    for f in range(nfield):
        ref = O.nan_ignoring_interp(land_fr, tlat, tlon, vals[f], glat, glon, radius, 4.0)
        np.testing.assert_array_equal(np.isnan(out[f]), np.isnan(ref), err_msg="NaN mask of field %d" % f)
        np.testing.assert_allclose(out[f], ref, rtol=0, atol=1e-9, equal_nan=True, err_msg="field %d" % f)
    for f in range(nfield):
        if f in holes:
            assert np.isfinite(out[f, a, b]) and abs(out[f, a, b] - (1.0 + 0.01 * f)) > 1e-3, f
        else:
            assert out[f, a, b] == np.float64(vals[f, j, i]), f
    masks = np.isnan(out).reshape(nfield, -1)
    assert not np.array_equal(masks[11], masks[12]) and not np.array_equal(masks[nfield - 2], masks[nfield - 1])

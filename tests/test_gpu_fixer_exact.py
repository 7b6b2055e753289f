"""The Tmin >= Tmax fixer, the recomputed 1981-2010 normals, se and the int16 quantisation on the device, held to an exact
referee on the device's own unfixed dailies.

twxi_interp_cells with fix_invalid = 0 returns the device's unfixed f8 dailies and with fix_invalid = 1 the fixed ones of
the same cells; the GWR stage is the same in both calls.  So the fixer is judged on its exact input, one fix at a time,
by the referee of test_fixer_exact_host.py (which also proves, on the CPU, that it rejects seeded defects):
  * the fixed days are exactly nonzero(tmin0 >= tmax0), every other day keeps its bits, ninvalid is their count and the
    status is what oracle.tmin_tmax_fixer decides on the unfixed series;
  * each fix is within fix_bound of its exact value on the device's own history (and within a chain bound of the float64
    oracle run on the unfixed series);
  * normals of fixed cells are the exact mean of the monthly means of the fixed 1981-2010 days (NaN for an empty group),
    those of cells without a fix are the kriged normals bit for bit, and se = sqrt(var) bit for bit;
  * twxi_interp_chunk on the same cells gives oracle.quantize_daily of those fixed dailies byte for byte, float32 of the
    f8 normals and se, and fill values wherever the status is not 0; the day windows of the record path give the chunk's
    bytes for windows of 1, 15, 16, 31, 32, 33 days and calendar years.

The crafted records come from "twin" station tables: one station table for both variables, Tmin observations
float32(norm_s(month) + a_d), Tmax observations float32(norm_s(month) + a_d + delta_d), and the Tmax LST planes of the work
chunk a copy of the Tmin planes.  A GWR hat row sums to 1 (X has an intercept), so every cell's Tmax - Tmin on day d is
delta_d up to ~1e-5, and delta_d = 0 gives bit-identical Tmin and Tmax: the inversions fall exactly where the pattern puts
them (checked first, in every cell).  Two realistic records (Fields(dtr_override=0.3) over 1979-1983, 0.05 over
1995-1996) add breadth.  The module runs in about 4 s on a B200 (1 000 W power limit).  Run with -m gpu."""
import importlib.util
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
_spec = importlib.util.spec_from_file_location("fixer_exact_referee", os.path.join(HERE, "test_fixer_exact_host.py"))
R = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(R)

NSTN = 700
CELLS = (2, 3)                          # work chunk of the crafted records (ny, nx)
WINDOWS = (1, 15, 16, 31, 32, 33)
KEYS = ("tmin", "tmax", "tmin_norm", "tmax_norm", "tmin_se", "tmax_se", "ninvalid", "status")
COVERAGE = {}


@pytest.fixture(scope="module")
def stations():
    from topowx_b200 import synth
    f = synth.Fields()
    sd = synth.make_station_db(0, NSTN, synth.tile_bbox(buf=2.0), f, synth.make_days(1995, 1), seed=77)
    wrk = synth.make_wrk_chk(f, synth.TILE_ROW0 + 10, synth.TILE_COL0 + 20, *CELLS)
    wrk[20:32] = wrk[8:20]                                    # both variables see the same LST predictors
    return sd.stns, wrk


def _twin_contexts(stns, days, delta):
    from topowx_b200 import db
    from topowx_b200.context import TwxiContext
    norm = np.stack([stns[db.get_norm_varname(m)] for m in range(1, 13)])
    base = norm[np.asarray(days[db.MONTH]) - 1, :] + R.smooth_anomaly(days.size)[:, None]
    obs = [base.astype(np.float32), (base + delta[:, None]).astype(np.float32)]
    good = np.isnan(stns[db.BAD])
    return [TwxiContext(db.StationSerialDataDb((stns, x, days), v), good) for x, v in zip(obs, ("tmin", "tmax"))]


def _record(ctx, wrk):
    """Unfixed and fixed cells of the chunk, the variances of both variables and the chunk call."""
    from topowx_b200.context import interp_cells, interp_chunk
    lat, lon, elev, tdi, cd = (np.ascontiguousarray(wrk[i].ravel()) for i in (3, 4, 5, 6, 7))
    lst = [np.stack([wrk[p + m].ravel() for m in range(12)], axis=1) for p in (8, 20)]
    r0 = interp_cells(ctx[0], ctx[1], lat, lon, elev, tdi, cd, lst[0], lst[1], fix_invalid=False)
    r1 = interp_cells(ctx[0], ctx[1], lat, lon, elev, tdi, cd, lst[0], lst[1], fix_invalid=True)
    var = [ctx[v].interp_points(lat, lon, elev, tdi, lst[v], daily=False)[3] for v in (0, 1)]
    chunk = {k: np.asarray(v) for k, v in interp_chunk(ctx[0], ctx[1], wrk).items()}
    return r0, r1, var, chunk


def _runs(days_fixed):
    """Lengths of the maximal runs of consecutive fixed days."""
    if days_fixed.size == 0:
        return np.zeros(0, dtype=np.int64)
    cut = np.flatnonzero(np.diff(days_fixed) != 1) + 1
    return np.diff(np.concatenate([[0], cut, [days_fixed.size]]))


def _judge(days, r0, r1, var, chunk, delta=None):
    """Every check of the module docstring on each cell; returns the coverage counts."""
    gs, gl = R.normal_groups(days)
    nd = days.size
    tmin0, tmax0, n0min, n0max, se0min, se0max, ninv0, st0 = r0
    tmin1, tmax1, nmin, nmax, semin, semax, ninv, st = r1
    ny, nx = chunk["status"].shape
    assert np.all(st0 == 0) and np.all(ninv0 == 0)
    cov = dict(cells=ny * nx, fixes=0, start=0, end=0, ballot_edge=0, ties=0, runs3=0, longest_run=0, fixer_empty=0,
               nan_normals=0, worst_step=0.0)
    for i in range(ny * nx):
        r, c = divmod(i, nx)
        a0, b0 = tmin0[i], tmax0[i]
        if delta is not None:                                 # the construction reproduces the pattern in every cell
            assert np.array_equal(np.flatnonzero(a0 >= b0), np.flatnonzero(delta <= 0)), i
            assert np.array_equal(a0[delta == 0], b0[delta == 0]), i
            live = delta > 0
            assert np.all(np.abs((b0 - a0)[live] - delta[live]) < 1e-3), i
            assert np.all(np.abs((b0 - a0)[delta < 0] + 2.0) < 1e-3), i
        want = R.oracle_status(a0, b0)
        assert st[i] == want, "cell %d: status %d, the oracle decides %d" % (i, st[i], want)
        assert chunk["status"][r, c] == st[i]
        if want != R.ST_OK:
            cov["fixer_empty"] += 1
            for arr in (tmin1[i], tmax1[i], nmin[i], nmax[i], semin[i], semax[i]):
                assert np.all(arr == R.FILL_F8), i
            assert ninv[i] == R.FILL_I4 and chunk["ninvalid"][r, c] == R.FILL_I4
            assert np.all(chunk["tmin"][:, r, c] == R.FILL_I2) and np.all(chunk["tmax"][:, r, c] == R.FILL_I2)
            for k in ("tmin_norm", "tmax_norm", "tmin_se", "tmax_se"):
                assert np.all(chunk[k][:, r, c] == R.FILL_F4), (i, k)
            continue
        fixed, worst = R.check_fixes(a0, b0, tmin1[i], tmax1[i], ninv[i])
        R.check_against_oracle(a0, b0, tmin1[i], tmax1[i])
        cov["worst_step"] = max(cov["worst_step"], worst)
        runs = _runs(fixed)
        cov["fixes"] += fixed.size
        cov["start"] += int((fixed < R.TAIL).sum())
        cov["end"] += int((fixed >= nd - R.TAIL).sum())
        cov["ballot_edge"] += int(np.isin(fixed % 32, (31, 0, 1)).sum())
        cov["ties"] += int((a0[fixed] == b0[fixed]).sum())
        cov["runs3"] += int((runs >= 3).sum())
        cov["longest_run"] = max(cov["longest_run"], int(runs.max()) if runs.size else 0)
        # normals: recomputed from the fixed 1981-2010 days, or the kriged ones bit for bit
        for t1, n1, n0 in ((tmin1[i], nmin[i], n0min[i]), (tmax1[i], nmax[i], n0max[i])):
            if fixed.size:
                cov["nan_normals"] += R.check_normals(t1, gs, gl, n1)
            else:
                assert R._same_bits(n1, n0), i
        # se = sqrt(var), 0 for a negative variance, in both calls
        for se1, se_0, v in ((semin[i], se0min[i], var[0][i]), (semax[i], se0max[i], var[1][i])):
            want_se = np.where(v >= 0, np.sqrt(np.maximum(v, 0.0)), 0.0)
            assert R._same_bits(se1, want_se) and R._same_bits(se_0, want_se), i
        # the chunk call: quantised fixed dailies, float32 of the f8 normals and se, the same count
        R.check_quantized(chunk["tmin"][:, r, c], tmin1[i])
        R.check_quantized(chunk["tmax"][:, r, c], tmax1[i])
        for k, f8 in (("tmin_norm", nmin[i]), ("tmax_norm", nmax[i]), ("tmin_se", semin[i]), ("tmax_se", semax[i])):
            assert np.array_equal(chunk[k][:, r, c], f8.astype(np.float32), equal_nan=True), (i, k)
        assert chunk["ninvalid"][r, c] == ninv[i]
    return cov


def _partitions(days):
    nd = days.size
    out = {}
    for k in WINDOWS:
        sizes = [k] * (nd // k) + ([nd % k] if nd % k else [])
        out.setdefault(tuple(sizes), "%d-day windows" % k)
    out.setdefault(tuple(np.unique(np.asarray(days["YEAR"]), return_counts=True)[1].tolist()), "calendar years")
    return out


def _check_record_path(ctx, wrk, days, chunk):
    """The day windows of twxi_tile_begin / _days / _end give the chunk's bytes for every partition."""
    from topowx_b200.context import tile_begin, tile_days, tile_end
    for sizes, what in _partitions(days).items():
        shape = tile_begin(ctx[0], ctx[1], wrk)
        parts = [tile_days(ctx[0], ctx[1], n, shape) for n in sizes]
        out = dict(tile_end(ctx[0], ctx[1], shape))
        for k in ("tmin", "tmax"):
            out[k] = np.concatenate([p[k] for p in parts])
        for k in KEYS:
            assert np.array_equal(chunk[k], np.asarray(out[k]), equal_nan=chunk[k].dtype.kind == "f"), (what, k)
    return len(_partitions(days))


# What each crafted record must exercise (coverage counts that must be > 0, and the ones that must be 0).
INTENT = {
    "y1995": (("start", "end", "ballot_edge", "ties", "runs3"), ("fixer_empty", "nan_normals")),
    "rec1980": (("start", "end", "ballot_edge", "ties", "runs3", "nan_normals"), ("fixer_empty",)),
    "empty_start": (("fixer_empty",), ("fixes",)),
    "all_tied": (("fixer_empty",), ("fixes",)),
    "short20": (("start", "end", "runs3", "nan_normals"), ("fixer_empty",)),
    "short31": (("start", "end", "ties", "ballot_edge", "nan_normals"), ("fixer_empty",)),
    "short32": (("start", "end", "ties", "ballot_edge", "nan_normals"), ("fixer_empty",)),
    "short33": (("start", "end", "ties", "ballot_edge", "nan_normals"), ("fixer_empty",)),
}


@pytest.mark.parametrize("name", sorted(R.CRAFTED))
def test_crafted_record(stations, name):
    stns, wrk = stations
    days, delta = R.crafted_days(name), R.crafted_delta(name)
    ctx = _twin_contexts(stns, days, delta)
    r0, r1, var, chunk = _record(ctx, wrk)
    cov = _judge(days, r0, r1, var, chunk, delta)
    cov["partitions"] = _check_record_path(ctx, wrk, days, chunk)
    COVERAGE[name] = cov
    print("%s (%d days): %s" % (name, days.size, cov))
    must, never = INTENT[name]
    for k in must:
        assert cov[k] > 0, (name, k)
    for k in never:
        assert cov[k] == 0, (name, k)
    if name == "y1995" or name == "rec1980":
        assert cov["longest_run"] >= 40
    if name in ("empty_start", "all_tied"):
        assert cov["fixer_empty"] == cov["cells"]


@pytest.mark.parametrize("dtr,year0,nyears", [(0.3, 1979, 5), (0.05, 1995, 2)])
def test_realistic_record(dtr, year0, nyears):
    """Fields with a forced diurnal range: 0.3 C over 1979-1983 (groups start mid-record, leap year), and 0.05 C over
    1995-1996 (dense inversions: fixes within 15 days of both ends of the record, runs)."""
    from topowx_b200 import synth, db
    from topowx_b200.context import TwxiContext
    f = synth.Fields(dtr_override=dtr)
    days = synth.make_days(year0, nyears)
    da = [synth.make_station_db(w, NSTN, synth.tile_bbox(buf=2.0), f, days, seed=77) for w in (0, 1)]
    ctx = [TwxiContext(d, np.isnan(d.stns[db.BAD])) for d in da]
    wrk = synth.make_wrk_chk(f, synth.TILE_ROW0 + 10, synth.TILE_COL0 + 20, 3, 4)
    r0, r1, var, chunk = _record(ctx, wrk)
    cov = _judge(days, r0, r1, var, chunk)
    cov["partitions"] = _check_record_path(ctx, wrk, days, chunk)
    print("dtr %.2f, %d-%d: %s" % (dtr, year0, year0 + nyears - 1, cov))
    assert cov["fixes"] > 0 and np.all(r1[6][r1[7] == 0] > 0)
    if dtr < 0.1:
        assert cov["start"] > 0 and cov["end"] > 0 and cov["runs3"] > 0

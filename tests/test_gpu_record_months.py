"""Monthly means of the daily product (twxi_tile_days_mth): bit for bit the numpy statement of the contract
float32((S / n) * float64(float32(0.01))) over the emitted int16 dailies, for any partition of the record into windows,
with the dailies of twxi_tile_days unchanged, fill for cells that are not ok, partial months at the record's ends, and
misuse reported without touching the tile.  Run with -m gpu."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

FILL_F4 = np.float32(9.969209968386869e+36)
ERR_ARG, ERR_STATE = -1, -3


@pytest.fixture(scope="module")
def rec():
    """1979-1983 (1 826 days, leap year 1980) with the fixer heavily active, masked cells and cells failed at begin."""
    from topowx_b200 import synth, db
    from topowx_b200.context import TwxiContext, interp_chunk
    f = synth.Fields(dtr_override=0.3)
    days = synth.make_days(1979, 5)
    da = [synth.make_station_db(w, 700, synth.tile_bbox(buf=2.0), f, days, seed=77) for w in (0, 1)]
    ctx = [TwxiContext(d, np.isnan(d.stns[db.BAD])) for d in da]
    wrk = synth.make_wrk_chk(f, synth.TILE_ROW0 + 10, synth.TILE_COL0 + 20, 12, 15)
    wrk[2, 3:5, 4:7] = 0                                              # masked cells
    wrk[7, 0, 0:2] = 1e6                                              # climate division unknown to the DB: fail at begin
    ref = interp_chunk(ctx[0], ctx[1], wrk)
    assert (ref["status"] == 255).sum() == 6 and (ref["status"] == 6).sum() == 2
    assert ref["ninvalid"][ref["status"] == 0].min() > 0              # the fixer really ran
    return dict(days=days, da=da, ctx=ctx, wrk=wrk, ref=ref)


def expected_months(days, tmin, tmax, status):
    """The contract in numpy: per month run, the exact sum of the int16 counts over its n days,
    float32((S / n) * float64(float32(0.01))); fill for every cell whose status is not ok."""
    from topowx_b200 import db
    start, ndays, year, month = db.month_runs(days)
    bad = np.asarray(status) != 0
    out = {}
    for k, q in (("tmin", tmin), ("tmax", tmax)):
        q = np.asarray(q)
        m = np.empty((start.size,) + q.shape[1:], np.float32)
        for g, (s, n) in enumerate(zip(start, ndays)):
            S = q[s:s + n].astype(np.int64).sum(axis=0)
            assert np.abs(S).max() < 2 ** 31 or bad.all()
            m[g] = ((S.astype(np.float64) / np.float64(n)) * np.float64(np.float32(0.01))).astype(np.float32)
        m[:, bad] = FILL_F4
        out[k] = m
    return out, [(int(y), int(mo), int(n)) for y, mo, n in zip(year, month, ndays)]


def run_months(ctx, wrk, days, sizes, device=False):
    """tile_begin, twxi_tile_days_mth over `sizes`, tile_end; per-window results on the host."""
    import torch
    from topowx_b200.context import tile_begin, tile_days_mth, tile_end, MonthGroups
    w = torch.from_numpy(wrk).cuda() if device else wrk
    dev = w.device if device else None
    host = (lambda a: a.cpu().numpy()) if device else np.asarray
    shape = tile_begin(ctx[0], ctx[1], w)
    groups = MonthGroups(days)
    parts = []
    for n in sizes:
        o = tile_days_mth(ctx[0], ctx[1], n, shape, groups, device=dev)
        parts.append(dict({k: host(o[k]) for k in ("tmin", "tmax", "tmin_mth", "tmax_mth")}, mth_groups=o["mth_groups"]))
    fin = {k: host(v) for k, v in tile_end(ctx[0], ctx[1], shape, device=dev).items()}
    cat = {k: np.concatenate([p[k] for p in parts]) for k in ("tmin", "tmax", "tmin_mth", "tmax_mth")}
    return cat, parts, fin


def run_days(ctx, wrk, sizes):
    from topowx_b200.context import tile_begin, tile_days, tile_end
    shape = tile_begin(ctx[0], ctx[1], wrk)
    parts = [tile_days(ctx[0], ctx[1], n, shape) for n in sizes]
    tile_end(ctx[0], ctx[1], shape)
    return {k: np.concatenate([p[k] for p in parts]) for k in ("tmin", "tmax")}


def same_bits(a, b):
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    return a.shape == b.shape and np.array_equal(a.view(np.int32), b.view(np.int32))


def check_windows(days, sizes, parts, exp_groups):
    """nmth and the (year, month, ndays) of every window: the runs whose last day falls inside it, in order."""
    from topowx_b200 import db
    start, ndays, _, _ = db.month_runs(days)
    ends = start + ndays
    d0 = 0
    for n, p in zip(sizes, parts):
        want = [exp_groups[g] for g in np.flatnonzero((ends > d0) & (ends <= d0 + n))]
        assert p["mth_groups"] == want, (d0, n)
        assert p["tmin_mth"].shape[0] == p["tmax_mth"].shape[0] == len(want)
        d0 += n


def test_partitions_bitwise_against_numpy(rec):
    days, ref, ctx, wrk = rec["days"], rec["ref"], rec["ctx"], rec["wrk"]
    nd = days.size
    exp, groups = expected_months(days, ref["tmin"], ref["tmax"], ref["status"])
    assert len(groups) == 60
    yrs = np.unique(days["YEAR"], return_counts=True)[1].tolist()
    feb81 = int(np.flatnonzero((days["YEAR"] == 1981) & (days["MONTH"] == 2))[0])
    mar81 = int(np.flatnonzero((days["YEAR"] == 1981) & (days["MONTH"] == 3))[0])
    ends = [feb81, mar81 + 1, mar81 + 11]          # a window ending on Jan 31, on Mar 1, on Mar 11
    parts = {
        "one window": [nd],
        "calendar years": yrs,
        "1-day windows over 70 days, then the rest": [1] * 70 + [nd - 70],
        "97-day windows": [97] * (nd // 97) + [nd % 97],
        "month's last day, first day, inside a month": [ends[0], ends[1] - ends[0], ends[2] - ends[1], nd - ends[2]],
    }
    first = None
    for what, sizes in parts.items():
        assert sum(sizes) == nd
        cat, win, fin = run_months(ctx, wrk, days, sizes)
        check_windows(days, sizes, win, groups)
        for k in ("tmin", "tmax"):
            assert same_bits(cat[k + "_mth"], exp[k]), (what, k)
        # the dailies are those of twxi_tile_days for the same windows, and the end is unchanged
        plain = run_days(ctx, wrk, sizes)
        for k in ("tmin", "tmax"):
            assert np.array_equal(cat[k], plain[k]) and np.array_equal(cat[k], ref[k]), (what, k)
        for k, v in fin.items():
            assert np.array_equal(v, ref[k]), (what, k)
        blob = b"".join(cat[k + "_mth"].tobytes() for k in ("tmin", "tmax"))
        first = blob if first is None else first
        assert blob == first, what
    bad = ref["status"] != 0
    assert np.all(exp["tmin"][:, bad] == FILL_F4) and np.all(exp["tmin"][:, ~bad] != FILL_F4)


def test_fill_for_masked_and_failed_cells(rec):
    ref = rec["ref"]
    cat, _, _ = run_months(rec["ctx"], rec["wrk"], rec["days"], [rec["days"].size])
    for st in (255, 6):                                                # masked, failed at begin
        sel = ref["status"] == st
        assert sel.any()
        for k in ("tmin_mth", "tmax_mth"):
            assert np.all(cat[k][:, sel] == FILL_F4)
    ok = ref["status"] == 0
    assert np.all(np.abs(cat["tmin_mth"][:, ok]) < 100) and np.all(cat["tmin_mth"][:, ok] < cat["tmax_mth"][:, ok])


def test_stream_months_and_memory_spaces(rec):
    """PtInterpTair.interp_chunk_stream(months=True).years() with host buffers and with device buffers: the same bytes."""
    import torch
    from topowx_b200.interp import PtInterpTair
    days, ref, da, wrk = rec["days"], rec["ref"], rec["da"], rec["wrk"]
    exp, groups = expected_months(days, ref["tmin"], ref["tmax"], ref["status"])
    pti = PtInterpTair(da[0], da[1])
    got = {}
    for where, w in (("host", wrk), ("device", torch.from_numpy(wrk).cuda())):
        s = pti.interp_chunk_stream(w, months=True)
        host = (lambda a: a.cpu().numpy()) if where == "device" else np.asarray
        parts = [dict({k: host(o[k]) for k in ("tmin", "tmax", "tmin_mth", "tmax_mth")}, mth_groups=o["mth_groups"])
                 for _, o in s.years()]
        fin = s.finish()
        assert np.array_equal(host(fin["status"]), ref["status"])
        assert sum((p["mth_groups"] for p in parts), []) == groups
        assert all(len(p["mth_groups"]) == 12 for p in parts)
        got[where] = {k: np.concatenate([p[k] for p in parts]) for k in ("tmin", "tmax", "tmin_mth", "tmax_mth")}
        for k in ("tmin", "tmax"):
            assert same_bits(got[where][k + "_mth"], exp[k]) and np.array_equal(got[where][k], ref[k]), (where, k)
    for k in got["host"]:
        assert got["host"][k].tobytes() == got["device"][k].tobytes(), k
    # the default stream returns no monthly grids
    s = pti.interp_chunk_stream(wrk)
    o = s.days(days.size)
    assert "tmin_mth" not in o
    s.finish()


def _pair(days, dtr, seed, wrk_at, shape=(2, 3)):
    from topowx_b200 import synth, db
    from topowx_b200.context import TwxiContext, interp_chunk
    f = synth.Fields(dtr_override=dtr)
    da = [synth.make_station_db(w, 700, synth.tile_bbox(buf=2.0), f, days, seed=seed) for w in (0, 1)]
    ctx = [TwxiContext(d, np.isnan(d.stns[db.BAD])) for d in da]
    wrk = synth.make_wrk_chk(f, synth.TILE_ROW0 + wrk_at[0], synth.TILE_COL0 + wrk_at[1], *shape)
    return ctx, wrk, interp_chunk(ctx[0], ctx[1], wrk)


def test_fixer_failure_gives_fill_in_months_completed_by_the_deciding_window():
    """'No valid tmin/tmax in window' is decided by the first window's fixer.  The record starts on Jan 31, so the one-day
    first window also completes January: that month is fill for the failed cells, like every later month."""
    from topowx_b200 import synth
    days = synth.make_days(1995, 2)[30:]
    assert days["DAY"][0] == 31
    ctx, wrk, ref = _pair(days, -1.2, 78, (30, 40))
    bad = ref["status"] == 5
    assert bad.any()
    exp, groups = expected_months(days, ref["tmin"], ref["tmax"], ref["status"])
    ys = np.unique(days["YEAR"], return_counts=True)[1].tolist()
    for sizes in ([1, ys[0] - 1, ys[1]], [days.size]):
        cat, parts, fin = run_months(ctx, wrk, days, sizes)
        assert np.array_equal(fin["status"], ref["status"])
        check_windows(days, sizes, parts, groups)
        if sizes[0] == 1:
            assert parts[0]["mth_groups"] == [(1995, 1, 1)]
            assert np.all(parts[0]["tmin_mth"][:, bad] == FILL_F4) and np.all(parts[0]["tmax_mth"][:, bad] == FILL_F4)
        for k in ("tmin", "tmax"):
            assert same_bits(cat[k + "_mth"], exp[k]) and np.all(cat[k + "_mth"][:, bad] == FILL_F4)
            assert np.array_equal(cat[k], ref[k])


def test_partial_months_at_the_ends_of_the_record():
    """A record from 1980-01-10 to 1981-06-20: the first and the last month average the days the record has."""
    from topowx_b200 import synth
    days = synth.make_days(1980, 2)
    i0 = int(np.flatnonzero(days["YMD"] == 19800110)[0])
    i1 = int(np.flatnonzero(days["YMD"] == 19810620)[0])
    days = days[i0:i1 + 1]
    ctx, wrk, ref = _pair(days, 0.3, 79, (60, 70), (3, 4))
    assert (ref["status"] == 0).all()
    exp, groups = expected_months(days, ref["tmin"], ref["tmax"], ref["status"])
    assert groups[0] == (1980, 1, 22) and groups[-1] == (1981, 6, 20) and len(groups) == 18
    # the value of the partial months is the mean of their days, not of a whole month
    q = np.asarray(ref["tmin"])
    assert np.allclose(exp["tmin"][0], q[:22].mean(axis=0) * 0.01, rtol=0, atol=1e-5)
    for sizes in ([days.size], [5, 30, 200, days.size - 235]):
        cat, parts, _ = run_months(ctx, wrk, days, sizes)
        check_windows(days, sizes, parts, groups)
        for k in ("tmin", "tmax"):
            assert same_bits(cat[k + "_mth"], exp[k]), (sizes, k)


def _raw_mth(ctx, n, ny, nx, max_mth, null_nmth=False):
    """twxi_tile_days_mth with host buffers, straight through ctypes.  Returns (rc, dailies, months, nmth)."""
    from topowx_b200 import _lib
    tmin, tmax = np.empty((n, ny, nx), np.int16), np.empty((n, ny, nx), np.int16)
    fmin, fmax = np.empty((max(max_mth, 1), ny, nx), np.float32), np.empty((max(max_mth, 1), ny, nx), np.float32)
    nm = C.c_int32(-7)
    rc = _lib.lib.twxi_tile_days_mth(ctx[0].handle, ctx[1].handle, n, _lib.ptr(tmin), _lib.ptr(tmax), max_mth,
                                     _lib.ptr(fmin), _lib.ptr(fmax), None if null_nmth else C.byref(nm), _lib.MEM_HOST)
    return rc, (tmin, tmax), (fmin[:nm.value], fmax[:nm.value]) if nm.value >= 0 else None, nm.value


def test_errors_leave_the_tile_as_it_was(rec):
    from topowx_b200 import _lib
    from topowx_b200.context import tile_begin, tile_days, tile_end, tile_days_mth, MonthGroups
    days, ref, ctx, wrk = rec["days"], rec["ref"], rec["ctx"], rec["wrk"]
    nd = days.size
    exp, _ = expected_months(days, ref["tmin"], ref["tmax"], ref["status"])
    ny, nx = wrk.shape[1:]
    # no open tile (the fixture's tiles were all ended)
    rc, _, _, _ = _raw_mth(ctx, 10, ny, nx, 1)
    assert rc == ERR_STATE
    # max_mth one too small, a NULL nmth: nothing happens, the retry gives the bytes of an uninterrupted run
    tile_begin(ctx[0], ctx[1], wrk)
    n1 = 100                                                          # Jan 1 .. Apr 10 1979: 3 months
    assert _raw_mth(ctx, n1, ny, nx, 2)[0] == ERR_ARG
    assert "more than max_mth" in _lib.lib.twxi_last_error().decode()
    assert _raw_mth(ctx, n1, ny, nx, 3, null_nmth=True)[0] == ERR_ARG
    rc, (a, b), (fa, fb), nm = _raw_mth(ctx, n1, ny, nx, 3)
    assert rc == 0 and nm == 3
    assert np.array_equal(a, ref["tmin"][:n1]) and np.array_equal(b, ref["tmax"][:n1])
    assert same_bits(fa, exp["tmin"][:3]) and same_bits(fb, exp["tmax"][:3])
    assert _raw_mth(ctx, nd - n1, ny, nx, 56)[0] == ERR_ARG           # 57 months remain
    rc, (a, b), (fa, fb), nm = _raw_mth(ctx, nd - n1, ny, nx, 57)
    assert rc == 0 and nm == 57
    assert np.array_equal(a, ref["tmin"][n1:]) and same_bits(fa, exp["tmin"][3:]) and same_bits(fb, exp["tmax"][3:])
    fin = tile_end(ctx[0], ctx[1], (ny, nx))
    assert np.array_equal(fin["tmin_norm"], ref["tmin_norm"])
    # a plain twxi_tile_days window earlier in the tile: the carry misses it
    shape = tile_begin(ctx[0], ctx[1], wrk)
    tile_days(ctx[0], ctx[1], 40, shape)
    g = MonthGroups(days)
    g.day0 = 40
    with pytest.raises(_lib.TwxiError, match="libtwxi error %d:" % ERR_STATE):
        tile_days_mth(ctx[0], ctx[1], 40, shape, g)
    last = tile_days(ctx[0], ctx[1], nd - 40, shape)                   # the daily calls still go on
    assert np.array_equal(last["tmin"], ref["tmin"][40:])
    tile_end(ctx[0], ctx[1], shape)
    # a new begin makes the monthly call valid again
    cat, _, _ = run_months(ctx, wrk, days, [nd])
    assert same_bits(cat["tmin_mth"], exp["tmin"])


def test_split_month_record_is_refused_while_daily_calls_work():
    """Jan 1-15, Feb, Jan 16-31, Mar .. Dec 1979: January falls in two runs.  twxi_ctx_set_obs and the daily calls accept
    the record (the 1981-2010 groups are unaffected); the monthly call returns TWXI_ERR_ARG and leaves the tile as it was."""
    from topowx_b200 import synth, db, _lib
    from topowx_b200.context import TwxiContext, interp_chunk, tile_begin, tile_days, tile_end, tile_days_mth, MonthGroups
    days = synth.make_days(1979, 1)
    perm = np.concatenate([np.arange(0, 15), np.arange(31, 59), np.arange(15, 31), np.arange(59, days.size)])
    f = synth.Fields(dtr_override=0.3)
    da = [synth.make_station_db(w, 700, synth.tile_bbox(buf=2.0), f, days, seed=80) for w in (0, 1)]
    da = [db.StationSerialDataDb((d.stns, np.asarray(d.var)[perm], days[perm]), ("tmin", "tmax")[w]) for w, d in enumerate(da)]
    ctx = [TwxiContext(d, np.isnan(d.stns[db.BAD])) for d in da]
    wrk = synth.make_wrk_chk(f, synth.TILE_ROW0 + 80, synth.TILE_COL0 + 90, 2, 3)
    ref = interp_chunk(ctx[0], ctx[1], wrk)
    assert (ref["status"] == 0).any()
    shape = tile_begin(ctx[0], ctx[1], wrk)
    with pytest.raises(_lib.TwxiError, match="libtwxi error %d:.*not consecutive" % ERR_ARG):
        tile_days_mth(ctx[0], ctx[1], 20, shape, MonthGroups(days[perm]))
    a = tile_days(ctx[0], ctx[1], 20, shape)
    b = tile_days(ctx[0], ctx[1], days.size - 20, shape)
    fin = tile_end(ctx[0], ctx[1], shape)
    assert np.array_equal(np.concatenate([a["tmin"], b["tmin"]]), ref["tmin"])
    assert np.array_equal(fin["status"], ref["status"])

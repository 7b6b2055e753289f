"""twxi_xval_overall (XvalTairOverall.run_xval_batch): the leave-one-out interpolation of step 24 with its bias / MAE / r^2
computed on the device, over a 2 000-station table with a one-year record and with a 32-year record that spans 1981-2010.
Run on the B200 box with -m gpu."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from oracle import twx_oracle as o          # noqa: E402  (checker only)

TOL_C = 1e-4
NAN_BITS = np.float64(np.nan).view(np.int64)


def _same(a, b):
    """Byte identity of two float arrays (NaN payloads included)."""
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and a.dtype == b.dtype and a.tobytes() == b.tobytes()


@pytest.fixture(scope="module", params=[(1995, 1), (1980, 32)], ids=["1995", "1980-2011"])
def rec(request):
    from topowx_b200 import synth, db
    from topowx_b200.interp import XvalTairOverall
    year0, nyears = request.param
    days = synth.make_days(year0, nyears)
    da = synth.make_station_db(0, 2000, synth.tile_bbox(), synth.Fields(), days)
    xv = XvalTairOverall(da, "tmin")
    cand = da.stn_ids[np.isnan(da.stns[db.BAD]) & np.isfinite(da.stns[db.MASK])]
    return dict(da=da, xv=xv, ctx=xv.interp_tair.gwr_tair.stn_slct.ctx, cand=cand, db=db, synth=synth)


def _obs(da, ids):
    """The stations' own observations, float32 widened to float64, [n, ndays]."""
    return np.asarray(da.var[:, [da.stn_idxs[s] for s in ids]], dtype=np.float64).T


def _numpy_stats(da, dly, obs):
    """bias, MAE, r^2 [n, 12] of the dailies against the observations over every record day of each month."""
    n = dly.shape[0]
    bias, mae, r2 = np.full((n, 12), np.nan), np.full((n, 12), np.nan), np.full((n, 12), np.nan)
    for m in range(1, 13):
        i = da.mth_idx[m]
        if i.size == 0:
            continue
        x, y = dly[:, i], obs[:, i]
        bias[:, m - 1] = np.mean(x - y, axis=1)
        mae[:, m - 1] = np.mean(np.abs(x - y), axis=1)
        xm, ym = x - x.mean(axis=1, keepdims=True), y - y.mean(axis=1, keepdims=True)
        r2[:, m - 1] = ((xm * ym).sum(1) / np.sqrt((xm * xm).sum(1) * (ym * ym).sum(1))) ** 2
    return bias, mae, r2


def _oracle_xval(oxv, oda, sid):
    """Skill of the oracle's leave-one-out interpolation: the statistics of oracle.XvalTairOverall.run_interp against
    load_obs, written the way oracle.XvalTairAnom.run_xval (optimize.py:520-531) is, over the full series."""
    dly, _, _ = oxv.run_interp(sid)
    obs = oda.load_obs(np.array([sid]))[:, 0].astype(np.float64)
    bias, mae, r2 = np.zeros(12), np.zeros(12), np.zeros(12)
    for mth in range(1, 13):
        x, y = dly[oda.mth_idx[mth]], obs[oda.mth_idx[mth]]
        difs = x - y
        bias[mth - 1] = np.mean(difs)
        mae[mth - 1] = np.mean(np.abs(difs))
        r2[mth - 1] = np.corrcoef(x, y)[0, 1] ** 2
    return bias, mae, r2


def test_same_bytes_as_interp_batch_and_numpy_statistics(rec):
    """1. daily, norms, se byte-identical to run_interp_batch; 2. bias / MAE within 1e-10 C and r^2 within 1e-9 of numpy
    statistics of those dailies against the stations' observations; 4. daily=False gives the same bytes."""
    xv, da, ids = rec["xv"], rec["da"], rec["cand"]
    dly0, norms0, se0, st0 = xv.run_interp_batch(ids)
    bias, mae, r2, norms, se, st, dly = xv.run_xval_batch(ids, daily=True)
    assert np.mean(st == 0) > 0.95
    assert _same(st, st0) and _same(dly, dly0) and _same(norms, norms0) and _same(se, se0)
    ok = st == 0
    assert np.all(np.isnan(bias[~ok])) and np.all(np.isnan(mae[~ok])) and np.all(np.isnan(r2[~ok]))
    nb, nm, nr = _numpy_stats(da, dly[ok], _obs(da, ids[ok]))
    assert np.all(np.isfinite(bias[ok])) and np.all(np.isfinite(r2[ok]))
    assert np.abs(bias[ok] - nb).max() < 1e-10
    assert np.abs(mae[ok] - nm).max() < 1e-10
    assert np.abs(r2[ok] - nr).max() < 1e-9
    lean = xv.run_xval_batch(ids)
    assert len(lean) == 6
    for a, b in zip(lean, (bias, mae, r2, norms, se, st)):
        assert _same(a, b)


def test_statistics_vs_oracle(rec):
    """3. Against the oracle's leave-one-out interpolation at three stations: bias / MAE within 1e-4 C, r^2 within 1e-6;
    run_xval is the batch's row."""
    da, xv, ids = rec["da"], rec["xv"], rec["cand"]
    oda = o.StationDb(da.stns, da.var, da.days)
    oxv = o.XvalTairOverall(oda)
    sel = ids[[5, 333, 1207]]
    bias, mae, r2, norms, se, st = xv.run_xval_batch(sel)
    assert np.all(st == 0)
    for i, sid in enumerate(sel):
        ob, om, orr = _oracle_xval(oxv, oda, sid)
        assert np.abs(bias[i] - ob).max() < TOL_C
        assert np.abs(mae[i] - om).max() < TOL_C
        assert np.abs(r2[i] - orr).max() < 1e-6
        one = xv.run_xval(sid)
        for a, b in zip(one, (bias[i], mae[i], r2[i])):
            assert _same(a, b)


def test_permuting_stations_permutes_outputs(rec):
    """5. The outputs of a permuted station list are the permuted outputs, byte for byte."""
    xv, ids = rec["xv"], rec["cand"][:700]
    ref = xv.run_xval_batch(ids, daily=True)
    perm = np.random.default_rng(24).permutation(ids.size)
    got = xv.run_xval_batch(ids[perm], daily=True)
    for a, b in zip(got, ref):
        assert _same(a, b[perm])


def test_colocated_twin_is_left_out(rec):
    """6. A station with a co-located twin is left out together with it: the results equal the point batch with the
    station left out and rm_zero, and the point batch with both stations left out explicitly."""
    from topowx_b200.db import StationSerialDataDb
    from topowx_b200.interp import XvalTairOverall
    db, da, cand = rec["db"], rec["da"], rec["cand"]
    stns = da.stns.copy()
    a, b = da.stn_idxs[cand[40]], da.stn_idxs[cand[41]]
    stns[db.LON][b], stns[db.LAT][b] = stns[db.LON][a], stns[db.LAT][a]
    da2 = StationSerialDataDb((stns, np.asarray(da.var), da.days), "tmin")
    xv = XvalTairOverall(da2, "tmin")
    ctx = xv.interp_tair.gwr_tair.stn_slct.ctx
    la, lb = int(ctx.local_of_db[a]), int(ctx.local_of_db[b])
    assert la >= 0 and lb >= 0
    bias, mae, r2, norms, se, st, dly = ctx.xval_overall([la, lb], daily=True)
    assert np.all(st == 0) and np.all(np.isfinite(r2))
    s = stns[[a, b]]
    lst = np.stack([s[db.get_lst_varname(m)] for m in range(1, 13)], axis=1)
    pts = (s[db.LAT], s[db.LON], s[db.ELEV], s[db.TDI], lst)
    d1, n1, s1, _, st1 = ctx.interp_points(*pts, rm_idx=np.array([[la], [lb]]), rm_zero=True)
    d2, n2, s2, _, st2 = ctx.interp_points(*pts, rm_idx=np.array([[la, lb], [lb, la]]), rm_zero=False)
    for dd, nn, ss, stt in ((d1, n1, s1, st1), (d2, n2, s2, st2)):
        assert _same(stt, st) and _same(dd, dly) and _same(nn, norms) and _same(ss, se)


def test_failures_are_per_station(rec):
    """7. An index outside the table gives TWXI_ST_TOO_FEW_STNS, NaN statistics and fill values, and the other stations of
    the batch keep their bytes; every station of a table too small for its neighbour count fails the same way; before
    set_obs the call returns TWXI_ERR_STATE."""
    from topowx_b200 import _lib, synth, db
    from topowx_b200.context import TwxiContext
    ctx = rec["ctx"]
    good = ctx.local_of_db[[rec["da"].stn_idxs[s] for s in rec["cand"][[3, 50, 900]]]].astype(np.int32)
    ref = ctx.xval_overall(good, daily=True)
    batch = np.array([good[0], ctx.n, good[1], -1, good[2]], dtype=np.int32)
    bias, mae, r2, norms, se, st, dly = ctx.xval_overall(batch, daily=True)
    bad, ok = np.array([1, 3]), np.array([0, 2, 4])
    assert np.all(st[bad] == _lib.ST_TOO_FEW_STNS)
    for arr in (bias, mae, r2):
        assert np.all(arr[bad].view(np.int64) == NAN_BITS)
    assert np.all(norms[bad] == _lib.FILL_F8) and np.all(se[bad] == _lib.FILL_F8) and np.all(dly[bad] == _lib.FILL_F8)
    for a, b in zip((bias, mae, r2, norms, se, st, dly), ref):
        assert _same(a[ok], b)

    f = synth.Fields()
    small = synth.make_station_db(0, 90, synth.tile_bbox(buf=1.0), f, synth.make_days(1995, 1), frac_bad=0.0)
    sctx = TwxiContext(small, np.isnan(small.stns[db.BAD]))
    bias, mae, r2, norms, se, st, dly = sctx.xval_overall(np.arange(sctx.n, dtype=np.int32), daily=True)
    assert np.all(st == _lib.ST_TOO_FEW_STNS)
    assert np.all(np.isnan(bias)) and np.all(np.isnan(mae)) and np.all(np.isnan(r2))
    assert np.all(norms == _lib.FILL_F8) and np.all(se == _lib.FILL_F8) and np.all(dly == _lib.FILL_F8)

    nobs = TwxiContext(small, np.isnan(small.stns[db.BAD]), with_obs=False)
    idx = np.zeros(1, dtype=np.int32)
    out = [np.empty(12) for _ in range(5)]
    stb = np.empty(1, dtype=np.uint8)
    rc = _lib.lib.twxi_xval_overall(nobs.handle, 1, _lib.ptr(idx), None, *[_lib.ptr(x) for x in out], _lib.ptr(stb),
                                    _lib.MEM_HOST)
    assert rc == -3
    assert ctx.xval_overall(np.zeros(0, dtype=np.int32))[5].size == 0

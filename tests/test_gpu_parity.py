"""Parity of the CUDA path (through the C ABI) against the CPU oracle and the committed golden vectors.
Run on the B200 box:  python -m pytest tests -m gpu"""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from oracle import twx_oracle as o          # noqa: E402  (checker only)

TOL_C = 1e-4          # deg C, north_star tolerance on interpolated values
TOL_VAR_REL = 1e-6    # relative, north_star tolerance on the kriging variance


@pytest.fixture(scope="module")
def env():
    from topowx_b200 import synth, db
    from topowx_b200.context import TwxiContext
    f = synth.Fields()
    days = synth.make_days(1995, 1)
    bbox = synth.tile_bbox()
    da = [synth.make_station_db(w, 2000, bbox, f, days) for w in (0, 1)]
    ctx = [TwxiContext(d, np.isnan(d.stns[db.BAD])) for d in da]
    oda = [o.StationDb(d.stns, d.var, d.days) for d in da]
    return dict(f=f, days=days, da=da, ctx=ctx, oda=oda, synth=synth, db=db)


def _pts(env, n, seed):
    synth = env["synth"]
    r = np.random.default_rng(seed)
    rows = r.integers(synth.TILE_ROW0, synth.TILE_ROW0 + synth.TILE_SIZE, n)
    cols = r.integers(synth.TILE_COL0, synth.TILE_COL0 + synth.TILE_SIZE, n)
    lat, lon = synth.grid_lats(rows), synth.grid_lons(cols)
    f = env["f"]
    elev, tdi = f.elev(lon, lat), f.tdi(lon, lat)
    lst = [np.stack([f.lst(w, m, lon, lat, elev) for m in range(1, 13)], axis=1) for w in (0, 1)]
    return lat, lon, elev, tdi, lst, f.climdiv(lon, lat)


def test_knn_bit_exact_vs_oracle(env):
    lat, lon, *_ = _pts(env, 300, 1)
    ctx, oda = env["ctx"][0], env["oda"][0]
    idx, dist, wgt, st = ctx.knn(lat, lon, 147)
    assert np.all(st == 0)
    ss = o.StationSelect(oda, ctx.mask)
    for i in range(lat.size):
        ss._set_pt(lat[i], lon[i])
        assert np.array_equal(ss.pt_sort_idx[:148], idx[i])                 # bit-exact neighbour order
        np.testing.assert_allclose(dist[i], ss.pt_sort_stn_dists[:148], rtol=1e-12, atol=0)
        d = ss.pt_sort_stn_dists
        w = np.square(1.0 - np.square(d[:148] / d[147]))
        np.testing.assert_allclose(wgt[i], w, rtol=0, atol=1e-11)
        gaps = np.diff(d[:150])
        assert gaps.min() > 1e-9                                            # fixture has no near ties


def test_knn_matches_reference_golden(env, golden_dir):
    """Neighbour sets of the reference's own StationSelect (golden vectors) incl. leave-one-out cases."""
    from topowx_b200 import db
    from topowx_b200.context import TwxiContext
    g = np.load(os.path.join(golden_dir, "station_select.npz"))
    n = g["stn_lon"].size
    stns = np.zeros(n, dtype=db.station_dtype())
    stns[db.STN_ID] = ["SYN%06d" % i for i in range(n)]
    stns[db.LON], stns[db.LAT] = g["stn_lon"], g["stn_lat"]
    for nm in stns.dtype.names[6:]:
        stns[nm] = 1.0
    sd = db.StationSerialDataDb((stns, g["obs_all"], env["days"][:g["month"].size]), "tmin")   # obs of the year's first days
    ctx = TwxiContext(sd, g["good"])
    for meta, gidx, gd, gw in zip(g["meta"], g["idx"], g["dists"], g["wgt"]):
        lat, lon, nn, rm, rm0 = meta[0], meta[1], int(meta[2]), int(meta[3]), int(meta[4])
        rm_idx = None if rm < 0 else np.array([[ctx.local_of_db[rm]]], dtype=np.int32)
        idx, dist, wgt, st = ctx.knn(lat, lon, nn, rm_idx=rm_idx, rm_zero=bool(rm0))
        assert st[0] == 0
        sel = ctx.gidx[idx[0, :nn]]
        order = np.argsort(sel)                                             # station-id order (:179-182)
        assert np.array_equal(sel[order], gidx[:nn])
        np.testing.assert_allclose(dist[0, :nn][order], gd[:nn], rtol=1e-12)
        np.testing.assert_allclose(wgt[0, :nn][order], gw[:nn], rtol=0, atol=1e-11)


def test_knn_too_few_stations(env):
    ctx = env["ctx"][0]
    lat, lon, *_ = _pts(env, 2, 5)
    # ask for more neighbours than the limit allows -> argument error, not a crash
    from topowx_b200._lib import TwxiError
    with pytest.raises(TwxiError):
        ctx.knn(lat, lon, 400)


def test_nngh_params_vs_oracle(env):
    lat, lon, elev, tdi, lst, _ = _pts(env, 120, 2)
    for w in (0, 1):
        ctx, oda = env["ctx"][w], env["oda"][w]
        kn, ka, vario, st = ctx.nngh_params(lat, lon)
        assert np.all(st == 0)
        ss = o.StationSelect(oda, ctx.mask)
        kt, gt = o.KrigTair(ss), o.GwrTairAnom(ss)
        pt = o.build_empty_pt()
        for i in range(0, lat.size, 3):
            pt[o.LAT], pt[o.LON] = lat[i], lon[i]
            for m in range(1, 13):
                k = kt.get_nnghs(pt, m)
                assert k == kn[i, m - 1]
                assert gt.get_nnghs(pt, m) == ka[i, m - 1]
                ss.set_ngh_stns(lat[i], lon[i], k, load_obs=False)
                np.testing.assert_allclose(vario[i, m - 1], kt.get_vario_params(pt, m), rtol=1e-11)


def test_krig_vs_oracle(env):
    lat, lon, elev, tdi, lst, _ = _pts(env, 60, 3)
    for w in (0, 1):
        ctx, oda = env["ctx"][w], env["oda"][w]
        mean, var, st = ctx.krig(lat, lon, elev, lst[w], mth=0)
        assert np.all(st == 0)
        ss = o.StationSelect(oda, ctx.mask)
        kt = o.KrigTair(ss)
        pt = o.build_empty_pt()
        worst = 0.0
        for i in range(0, lat.size, 2):
            pt[o.LAT], pt[o.LON], pt[o.ELEV] = lat[i], lon[i], elev[i]
            for m in range(1, 13):
                pt[o.lst_name(m)] = lst[w][i, m - 1]
                om, ov = kt.krig(pt, m)
                worst = max(worst, abs(om - mean[i, m - 1]))
                assert abs(om - mean[i, m - 1]) < TOL_C
                assert abs(ov - var[i, m - 1]) <= TOL_VAR_REL * abs(ov)
        print("krig worst |dmean| = %.3e C" % worst)


def test_krig_overrides_and_single_month(env):
    lat, lon, elev, tdi, lst, _ = _pts(env, 8, 4)
    ctx, oda = env["ctx"][1], env["oda"][1]
    mean, var, st = ctx.krig(lat, lon, elev, lst[1], mth=7, nnghs=41, vario=(0.3, 1.4, 75.0))
    assert np.all(st == 0) and mean.shape == (8, 1)
    ss = o.StationSelect(oda, ctx.mask)
    kt = o.KrigTair(ss)
    pt = o.build_empty_pt()
    for i in range(lat.size):
        pt[o.LAT], pt[o.LON], pt[o.ELEV] = lat[i], lon[i], elev[i]
        pt[o.lst_name(7)] = lst[1][i, 6]
        om, ov = kt.krig(pt, 7, nnghs=41, vario_params=(0.3, 1.4, 75.0))
        assert abs(om - mean[i, 0]) < TOL_C and abs(ov - var[i, 0]) <= TOL_VAR_REL * abs(ov)
    # pure nugget model (range == 0, interp.R:223-227)
    mean, var, st = ctx.krig(lat, lon, elev, lst[1], mth=2, nnghs=60, vario=(0.4, 0.9, 0.0))
    for i in range(lat.size):
        pt[o.LAT], pt[o.LON], pt[o.ELEV] = lat[i], lon[i], elev[i]
        pt[o.lst_name(2)] = lst[1][i, 1]
        om, ov = kt.krig(pt, 2, nnghs=60, vario_params=(0.4, 0.9, 0.0))
        assert abs(om - mean[i, 0]) < TOL_C and abs(ov - var[i, 0]) <= TOL_VAR_REL * abs(ov)


def test_krig_every_size_class_vs_oracle(env):
    """Neighbour counts from the smallest system to the reference's maximum (147 = size class NB 19), with and without
    padding of the last tile row (n a multiple of 8): each count exercises another launch of the kriging stage."""
    lat, lon, elev, tdi, lst, _ = _pts(env, 3, 11)
    ctx, oda = env["ctx"][0], env["oda"][0]
    ss = o.StationSelect(oda, ctx.mask)
    kt = o.KrigTair(ss)
    pt = o.build_empty_pt()
    for n in (6, 8, 9, 16, 35, 40, 64, 71, 80, 88, 96, 100, 104, 128, 147):
        mean, var, st = ctx.krig(lat, lon, elev, lst[0], mth=5, nnghs=n, vario=(0.2, 1.1, 120.0))
        assert np.all(st == 0), n
        for i in range(lat.size):
            pt[o.LAT], pt[o.LON], pt[o.ELEV] = lat[i], lon[i], elev[i]
            pt[o.lst_name(5)] = lst[0][i, 4]
            om, ov = kt.krig(pt, 5, nnghs=n, vario_params=(0.2, 1.1, 120.0))
            assert abs(om - mean[i, 0]) < TOL_C, (n, i, om, mean[i, 0])
            assert abs(ov - var[i, 0]) <= TOL_VAR_REL * abs(ov), (n, i, ov, var[i, 0])


def test_empty_batch_is_a_no_op(env):
    ctx = env["ctx"][0]
    z = np.zeros(0)
    mean, var, st = ctx.krig(z, z, z, np.zeros((0, 12)), mth=0)
    assert mean.shape[0] == 0 and var.shape[0] == 0 and st.shape[0] == 0
    idx, dist, wgt, st = ctx.knn(z, z, 35)
    assert idx.shape[0] == 0 and st.shape[0] == 0


def test_krig_colocated_stations_are_singular():
    """Two stations at the same location make the kriging covariance matrix singular: gstat stops, the drivers leave
    the fill value (step25:154-160).  The library decides it exactly (a zero station-station distance inside the
    point's neighbour set) instead of by the sign of a rounded pivot; points that do not see the pair are unaffected."""
    from topowx_b200 import synth, db, _lib
    from topowx_b200.context import TwxiContext
    f = synth.Fields()
    days = synth.make_days(1995, 1)
    da = synth.make_station_db(1, 600, synth.tile_bbox(buf=2.0), f, days)
    good = np.flatnonzero(np.isnan(da.stns[db.BAD]))
    lon0, lat0 = synth.grid_lons(synth.TILE_COL0), synth.grid_lats(synth.TILE_ROW0)
    d = o.grt_circle_dist(lon0, lat0, da.stns[db.LON][good], da.stns[db.LAT][good])
    a, b = good[np.argsort(d)[:2]]                        # the two stations nearest the tile's first cell
    da.stns[db.LON][b], da.stns[db.LAT][b] = da.stns[db.LON][a], da.stns[db.LAT][a]
    ctx = TwxiContext(da, np.isnan(da.stns[db.BAD]))
    oda = o.StationDb(da.stns, da.var, da.days)
    rows = np.array([0, 2, 10, 7, 249, 240]) + synth.TILE_ROW0
    cols = np.array([0, 3, 4, 12, 249, 200]) + synth.TILE_COL0
    lat, lon = synth.grid_lats(rows), synth.grid_lons(cols)
    elev = f.elev(lon, lat)
    lst = np.stack([f.lst(1, m, lon, lat, elev) for m in range(1, 13)], axis=1)
    kn, _, _, st0 = ctx.nngh_params(lat, lon)
    idx, _, _, _ = ctx.knn(lat, lon, 147)
    mean, var, st = ctx.krig(lat, lon, elev, lst, mth=0)
    ia, ib = int(np.flatnonzero(good == a)[0]), int(np.flatnonzero(good == b)[0])
    ss = o.StationSelect(oda, ctx.mask)
    kt = o.KrigTair(ss)
    pt = o.build_empty_pt()
    nsing = 0
    for i in range(lat.size):
        nmax = kn[i].max()
        sees_pair = ia in idx[i, :nmax] and ib in idx[i, :nmax]
        assert (st[i] == _lib.ST_SINGULAR) == sees_pair
        pt[o.LAT], pt[o.LON], pt[o.ELEV] = lat[i], lon[i], elev[i]
        if sees_pair:
            nsing += 1
            raised = 0                                    # (numpy's Cholesky lets some months through on a rounded pivot)
            for m in range(1, 13):
                pt[o.lst_name(m)] = lst[i, m - 1]
                try:
                    kt.krig(pt, m)
                except o.OracleError as e:
                    assert e.status == o.ST_SINGULAR
                    raised += 1
            assert raised >= 1                            # the point fails in the reference loop (interp_tair.py:396-439)
        else:
            assert st[i] == 0
            for m in (1, 7):
                pt[o.lst_name(m)] = lst[i, m - 1]
                om, ov = kt.krig(pt, m)
                assert abs(om - mean[i, m - 1]) < TOL_C and abs(ov - var[i, m - 1]) <= TOL_VAR_REL * abs(ov)
    assert 3 <= nsing < lat.size


def test_gwr_hat_and_daily_vs_oracle(env):
    lat, lon, elev, tdi, lst, _ = _pts(env, 40, 6)
    ctx, oda = env["ctx"][0], env["oda"][0]
    ss = o.StationSelect(oda, ctx.mask)
    gt = o.GwrTairAnom(ss)
    pt = o.build_empty_pt()
    for m in (1, 6, 11):
        k, idx, z, st = ctx.gwr_hat(lat, lon, elev, tdi, lst[0], m)
        ptn = np.linspace(-5, 20, lat.size)
        out, st2 = ctx.gwr_mth(lat, lon, elev, tdi, lst[0], m, ptn)
        assert np.all(st == 0) and np.all(st2 == 0)
        for i in range(lat.size):
            pt[o.LAT], pt[o.LON], pt[o.ELEV], pt[o.TDI] = lat[i], lon[i], elev[i], tdi[i]
            pt[o.lst_name(m)] = lst[0][i, m - 1]
            pt[o.norm_name(m)] = ptn[i]
            vals = gt.gwr_mth(pt, m)
            assert gt.last["nnghs"] == k[i]
            zz = np.zeros(ctx.n); zz[idx[i, :k[i]]] = z[i, :k[i]]
            zo = np.zeros(ctx.n); zo[gt.last["idx"]] = gt.last["z"]
            assert np.abs(zz - zo).max() < 1e-9
            assert np.abs(vals - out[i]).max() < TOL_C


def test_interp_points_loo_vs_oracle(env):
    """step24-style leave-one-out at station locations (optimize.py:579-604)."""
    db = env["db"]
    w = 1
    ctx, oda, da = env["ctx"][w], env["oda"][w], env["da"][w]
    xv = o.XvalTairOverall(oda)
    cand = np.nonzero(np.isnan(da.stns[db.BAD]) & np.isfinite(da.stns[db.MASK]))[0]
    sel = cand[np.random.default_rng(8).choice(cand.size, 12, replace=False)]
    s = da.stns[sel]
    lst = np.stack([s[db.get_lst_varname(m)] for m in range(1, 13)], axis=1)
    rm = ctx.local_of_db[sel].astype(np.int32).reshape(-1, 1)
    dly, norms, se, var, st = ctx.interp_points(s[db.LAT], s[db.LON], s[db.ELEV], s[db.TDI], lst, rm_idx=rm, rm_zero=True)
    assert np.all(st == 0)
    for i, sid in enumerate(s[db.STN_ID]):
        od, on, ose = xv.run_interp(sid)
        assert np.abs(on - norms[i]).max() < TOL_C
        assert np.abs(ose - se[i]).max() < 1e-6
        assert np.abs(od - dly[i]).max() < TOL_C


def test_interp_chunk_vs_oracle(env):
    """A small work chunk through twxi_interp_chunk against the oracle's step25 loop, incl. a masked cell,
    an unknown climate division and the int16 quantisation."""
    from topowx_b200.context import interp_chunk
    synth = env["synth"]
    wrk = synth.make_wrk_chk(env["f"], synth.TILE_ROW0 + 40, synth.TILE_COL0 + 60, 6, 8)
    wrk[2, 0, 0] = 0.0                       # masked
    wrk[7, 1, 1] = 9999.0                    # KeyError climdiv
    out = interp_chunk(env["ctx"][0], env["ctx"][1], wrk)
    pti = o.PtInterpTair(env["oda"][0], env["oda"][1])
    ref = o.interp_chunk(pti, wrk)
    assert out["status"][0, 0] == 255 and out["status"][1, 1] == o.ST_CLIMDIV
    st = out["status"].copy(); st[0, 0] = 0
    assert np.array_equal(st, ref["status"])
    for k in ("tmin", "tmax"):
        d = np.abs(out[k].astype(np.int32) - ref[k].astype(np.int32))
        assert d.max() <= 1                                           # 0.01 C count, x.xx5 boundaries
        assert (d > 0).mean() < 1e-3
        assert np.all(out[k][:, 0, 0] == -32767) and np.all(out[k][:, 1, 1] == -32767)
    for k in ("tmin_norm", "tmax_norm", "tmin_se", "tmax_se"):
        good = ref["status"] == 0
        good[0, 0] = False
        assert np.abs(out[k][:, good] - ref[k][:, good]).max() < TOL_C
        assert out[k][0, 0, 0] == ref[k][0, 0, 0]                     # fill value
    assert np.array_equal(out["ninvalid"], ref["ninvalid"])


def test_conus_scale_station_table():
    """BASELINE configs 3-5 use ~10 000 stations over CONUS: the neighbour search scans / prunes a 5x larger table,
    the station-station distance table is 800 MB, and land/ocean mask plus out-of-domain stations (NaN optim /
    variogram columns) come into play.  A chunk in the interior and a leave-one-out batch against the oracle."""
    from topowx_b200 import synth, db
    from topowx_b200.context import TwxiContext, interp_chunk
    f = synth.Fields()
    days = synth.make_days(1995, 1)
    da = [synth.make_station_db(w, 10000, synth.conus_bbox(), f, days) for w in (0, 1)]
    oda = [o.StationDb(d.stns, d.var, d.days) for d in da]
    ctx = [TwxiContext(d, np.isnan(d.stns[db.BAD])) for d in da]
    wrk = synth.make_wrk_chk(f, 1500, 3400, 30, 40)
    out = interp_chunk(ctx[0], ctx[1], wrk)
    pti = o.PtInterpTair(oda[0], oda[1])
    land = np.argwhere(wrk[2] != 0)
    assert land.size > 0
    r = np.random.default_rng(5)
    cells = [tuple(int(v) for v in land[i]) for i in r.choice(len(land), min(5, len(land)), replace=False)]
    ref = o.interp_chunk(pti, wrk, cells=cells)
    for (a, b) in cells:
        assert out["status"][a, b] == ref["status"][a, b]
        if ref["status"][a, b] != 0:
            continue
        for k in ("tmin", "tmax"):
            assert np.abs(out[k][:, a, b].astype(int) - ref[k][:, a, b].astype(int)).max() <= 1
        for k in ("tmin_norm", "tmax_norm", "tmin_se", "tmax_se"):
            assert np.abs(out[k][:, a, b] - ref[k][:, a, b]).max() < TOL_C
    # step24-style LOO at 4 in-domain stations of the tmax DB
    w = 1
    xv = o.XvalTairOverall(oda[w])
    cand = np.nonzero(np.isnan(da[w].stns[db.BAD]) & np.isfinite(da[w].stns[db.MASK]))[0]
    sel = cand[r.choice(cand.size, 4, replace=False)]
    s = da[w].stns[sel]
    lst = np.stack([s[db.get_lst_varname(m)] for m in range(1, 13)], axis=1)
    rm = ctx[w].local_of_db[sel].astype(np.int32).reshape(-1, 1)
    dly, norms, se, var, st = ctx[w].interp_points(s[db.LAT], s[db.LON], s[db.ELEV], s[db.TDI], lst, rm_idx=rm, rm_zero=True)
    for i, sid in enumerate(s[db.STN_ID]):
        try:
            od, on, ose = xv.run_interp(sid)
        except o.OracleError as e:
            assert st[i] == e.status
            continue
        assert st[i] == 0
        assert np.abs(on - norms[i]).max() < TOL_C and np.abs(od - dly[i]).max() < TOL_C

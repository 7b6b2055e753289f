"""Every GWR kernel instance against an extended-precision solve of the reference's formula.

gwr_kernel is compiled for the daily values (gwr_mth), the leave-one-out statistics (xval_anom) and the hat rows of the
record path (tile_begin), each with the separate-array gather and with the packed 64-byte station rows used above
TWXI_GWR_PACKED_MIN_N stations; tile_apply_kernel repeats the day loop.  The referee here is not the float64 oracle
(which inverts the uncentred X'WX, condition up to ~1e15 on these neighbourhoods, and is itself off by up to 2e-6 C) but
``gwr_exact``: the same formula in 40-digit arithmetic, rounded once.  Each tolerance comes from the problem's own
conditioning, so a kernel that drops precision anywhere (a float accumulator, a wrong constant, a lost neighbour) fails.

Neighbour counts cover k mod 8 and k mod 16 (the 8-, 4- and 1-wide passes of the day loop, the padded DMMA staging),
the extremes 6 and TWXI_MAX_NNGHS = 255, and k = 1..5 (fewer stations than the six coefficients: TWXI_ST_SINGULAR).
Months 1, 2, 4 and 12 of 1995-1996 give 57-62 days: two lane passes, the second one partial, and a leap February.
Run with -m gpu; the reference's own checks at the end run on the CPU."""
import multiprocessing as mp
import os
import re
from fractions import Fraction

import numpy as np
import pytest

try:
    import mpmath
except ImportError:                     # mpmath comes with torch (through sympy); exact rationals otherwise
    mpmath = None

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DPS = 40
EPS = 2.0 ** -53
C_BOUND = 64                            # bound = C_BOUND * eps * (conditioning terms), see _hat_bound / _daily_bound
R2_TOL = 1e-9
ABS_TOL_C = 1e-8                        # DESIGN.md §2: GWR dailies <= 1e-8 C (k >= 35, the counts the DB holds)
COUNTS = list(range(6, 23)) + [31, 32, 33, 63, 64, 65, 127, 128, 129, 147, 168, 169] + list(range(240, 256))
MONTHS = (1, 2, 4, 12)
REC_COUNTS = (6, 13, 64, 128, 241, 254, 255)
ST_OK, ST_SINGULAR, ST_MASKED = 0, 4, 255
FILL_I2, FILL_I4, FILL_F4 = -32767, -2147483647, np.float32(9.969209968386869e+36)


# ---- the reference --------------------------------------------------------------------------------------------------
def _num(x):
    """A float64 as an exact number of the working precision."""
    return mpmath.mpf(float(x)) if mpmath else Fraction(float(x))


def _dot(a, b):
    return mpmath.fdot(a, b) if mpmath else sum(x * y for x, y in zip(a, b))


def _solve(A, b):
    """Gaussian elimination with partial pivoting (6x6, working precision)."""
    n = len(b)
    M = [list(A[i]) + [b[i]] for i in range(n)]
    for c in range(n):
        p = max(range(c, n), key=lambda r: abs(M[r][c]))
        M[c], M[p] = M[p], M[c]
        for r in range(c + 1, n):
            f = M[r][c] / M[c][c]
            M[r] = [M[r][i] - f * M[c][i] for i in range(n + 1)]
    u = [None] * n
    for c in reversed(range(n)):
        u[c] = (M[c][n] - sum(M[c][i] * u[i] for i in range(c + 1, n))) / M[c][c]
    return u


def _hat_exact(X, x0, w):
    """z_j = w_j x_j' (X'WX)^-1 x0 with the uncentred X = [1, lon, lat, elev, tdi, lst_m] of interp_tair.py:1128-1140.
    ``w`` holds exact numbers; returns z as exact numbers (not rounded)."""
    one = _num(1.0)
    rows = [[one] + [_num(v) for v in r] for r in np.asarray(X)]
    cols = [[r[a] for r in rows] for a in range(6)]
    wcols = [[wj * v for wj, v in zip(w, c)] for c in cols]
    A = [[_dot(wcols[a], cols[b]) for b in range(6)] for a in range(6)]
    u = _solve(A, [one] + [_num(v) for v in x0])
    return [wj * _dot(r, u) for wj, r in zip(w, rows)]


def gwr_exact(X, x0, dist, k, obs, norm, ptn, own=None):
    """The GWR value of every day of one (point, month) in DPS-digit arithmetic, rounded once at the end.

    X [k][5] station predictors (lon, lat, elev, tdi, lst_m), x0 [5] the point's, dist [k+1] the library's kNN distances
    (bisquare weights w = (1 - (d_j / d_k)^2)^2), obs [D][k] float32 observations, norm [k] station normals, ptn the
    point's normal:  v_d = sum_j z_j obs_dj + (ptn - sum_j z_j norm_j).
    Returns dict(z [k], v [D]); with ``own`` [D] (the held-out station's observations, XvalTairAnom) also bias, mae, r2
    of the interpolated anomaly v - ptn against own - ptn (optimize.py:520-531)."""
    ctx = mpmath.workdps(DPS) if mpmath else _NoCtx()
    with ctx:
        d = [_num(v) for v in dist[:k + 1]]
        w = []
        for j in range(k):
            r = d[j] / d[k]
            w.append((1 - r * r) ** 2)
        z = _hat_exact(np.asarray(X)[:k], x0, w)
        P = _num(ptn)
        off = P - _dot(z, [_num(v) for v in norm[:k]])
        obs = np.asarray(obs, dtype=np.float64)[:, :k]
        v = [_dot(z, [_num(o) for o in row]) + off for row in obs]
        out = dict(z=np.array([float(t) for t in z]), v=np.array([float(t) for t in v]))
        if own is not None:
            x = [t - P for t in v]
            y = [_num(o) - P for o in np.asarray(own, dtype=np.float64)]
            n = len(x)
            dif = [a - b for a, b in zip(x, y)]
            xm, ym = sum(x) / n, sum(y) / n
            cxy = sum((a - xm) * (b - ym) for a, b in zip(x, y))
            cxx = sum((a - xm) ** 2 for a in x)
            cyy = sum((b - ym) ** 2 for b in y)
            out.update(bias=float(sum(dif) / n), mae=float(sum(abs(t) for t in dif) / n),
                       r2=float(cxy * cxy / (cxx * cyy)))
    return out


class _NoCtx(object):
    def __enter__(self):
        return self

    def __exit__(self, *a):
        return False


def _weights(dist, k):
    return np.square(1.0 - np.square(dist[:k] / dist[k]))


def _kappa(X, x0, w):
    """cond_2 of X_e'WX_e, X_e = [1, predictors centred on the point, each scaled to unit weighted RMS]."""
    Xc = np.asarray(X, dtype=np.float64) - np.asarray(x0, dtype=np.float64)
    Xc = Xc / np.sqrt((w[:, None] * Xc * Xc).sum(0) / w.sum())
    Xe = np.column_stack([np.ones(len(w)), Xc])
    return float(np.linalg.cond((Xe.T * w) @ Xe))


def _hat_bound(kappa, z):
    return C_BOUND * EPS * kappa * np.abs(z).max()


def _daily_bound(kappa, z, obs, norm, ptn):
    az = np.abs(z)
    obs = np.asarray(obs, dtype=np.float64)
    return C_BOUND * EPS * (kappa * (np.abs(obs - norm) @ az) + (np.abs(obs) + np.abs(norm)) @ az + abs(ptn))


def _ref_task(args):
    return gwr_exact(*args)


def _farm(tasks):
    """gwr_exact over every host core (fork pool, as oracle/cpu_farm.py)."""
    n = max(1, os.cpu_count() or 1)
    with mp.get_context("fork").Pool(n) as pool:
        return pool.map(_ref_task, tasks, chunksize=max(1, len(tasks) // (8 * n)))


# ---- fixture --------------------------------------------------------------------------------------------------------
def _packed_min_n():
    src = open(os.path.join(ROOT, "topowx_b200", "csrc", "gwr.cu")).read()
    return int(re.search(r"#define\s+TWXI_GWR_PACKED_MIN_N\s+(\d+)", src).group(1))


class _Stats(object):
    """Worst error / bound ratio and worst absolute error per (instance, layout, k >= 35)."""

    def __init__(self):
        self.d = {}

    def add(self, key, ratio, err):
        r, e = self.d.get(key, (0.0, 0.0))
        self.d[key] = (max(r, float(ratio)), max(e, float(err)))

    def report(self, title):
        print("\n" + title)
        for key in sorted(self.d):
            print("  %-44s worst error/bound %.3g   worst |error| %.3g" % (" ".join(map(str, key)), *self.d[key]))


@pytest.fixture(scope="module")
def env():
    from topowx_b200 import synth, db
    from topowx_b200.context import TwxiContext
    f = synth.Fields()
    days = synth.make_days(1995, 2)
    da = [synth.make_station_db(w, 3200, synth.tile_bbox(), f, days) for w in (0, 1)]
    nsep = _packed_min_n()
    mid_r, mid_c = synth.TILE_ROW0 + synth.TILE_SIZE // 2, synth.TILE_COL0 + synth.TILE_SIZE // 2
    lat_c, lon_c = float(synth.grid_lats(mid_r)), float(synth.grid_lons(mid_c))
    rng = np.random.default_rng(20261020)
    rows = rng.integers(synth.TILE_ROW0 + 20, synth.TILE_ROW0 + synth.TILE_SIZE - 20, 6)
    cols = rng.integers(synth.TILE_COL0 + 20, synth.TILE_COL0 + synth.TILE_SIZE - 20, 6)
    cell_lat, cell_lon = synth.grid_lats(rows), synth.grid_lons(cols)
    V = []
    for w, d in enumerate(da):
        s = d.stns
        good = np.nonzero(np.isnan(s[db.BAD]))[0]
        far = np.hypot(s[db.LAT][good] - lat_c, (s[db.LON][good] - lon_c) * np.cos(np.radians(lat_c)))
        order = good[np.argsort(far, kind="stable")]
        assert order.size > nsep
        sep = np.zeros(s.size, dtype=bool)
        sep[order[:nsep]] = True
        packed = sep.copy()
        extra = int(order[-1])                                        # the good station farthest from the tile
        packed[extra] = True
        ctx = dict(sep=TwxiContext(d, sep), packed=TwxiContext(d, packed))
        assert ctx["sep"].n == nsep and ctx["packed"].n == nsep + 1
        # points: 6 tile cells, and 2 stations of the table queried without rm_zero (a neighbour at d = 0)
        on = order[[3, 40]]
        lat = np.concatenate([cell_lat, s[db.LAT][on]])
        lon = np.concatenate([cell_lon, s[db.LON][on]])
        elev = np.concatenate([f.elev(cell_lon, cell_lat), s[db.ELEV][on]])
        tdi = np.concatenate([f.tdi(cell_lon, cell_lat), s[db.TDI][on]])
        lst = np.stack([np.concatenate([f.lst(w, m, cell_lon, cell_lat, elev[:6]), s[db.get_lst_varname(m)][on]])
                        for m in range(1, 13)], axis=1)
        ptn = np.stack([np.linspace(-6.0, 21.0, lat.size) + 0.37 * m for m in range(1, 13)], axis=1)
        # leave-one-out stations of the cross validation: near the tile centre, context indices of each layout
        xv_db = order[[0, 7, 19]]
        V.append(dict(da=d, ctx=ctx, extra=extra, on=on, lat=lat, lon=lon, elev=elev, tdi=tdi, lst=lst, ptn=ptn, xv_db=xv_db))
    return dict(f=f, days=days, da=da, V=V, synth=synth, db=db)


def _station_arrays(v, m, sel):
    """Predictors [k][5] (lon, lat, elev, tdi, lst_m) and normals of the DB stations ``sel``."""
    from topowx_b200 import db
    s = v["da"].stns[sel]
    X = np.column_stack([s[db.LON], s[db.LAT], s[db.ELEV], s[db.TDI], s[db.get_lst_varname(m)]])
    return X, np.asarray(s[db.get_norm_varname(m)], dtype=np.float64)


@pytest.fixture(scope="module")
def hat_ref(env):
    """Reference of test 1: per variable, the kNN of the points (separate layout, k1 = 256, DB indices) and gwr_exact of
    every (point, month, count)."""
    out = []
    for v in env["V"]:
        sep = v["ctx"]["sep"]
        idx, dist, _, st = sep.knn(v["lat"], v["lon"], 255)
        assert np.all(st == 0)
        gidx = sep.gidx[idx]
        assert not np.isin(v["extra"], gidx)                         # the packed table's extra station is never used
        assert np.array_equal(gidx[6:, 0], v["on"]) and np.all(dist[6:, 0] < 1e-9)    # station points: d = 0 first
        tasks, meta = [], []
        for m in MONTHS:
            days = sep.mth_idx[m]
            for q in range(v["lat"].size):
                x0 = [v["lon"][q], v["lat"][q], v["elev"][q], v["tdi"][q], v["lst"][q, m - 1]]
                for k in COUNTS:
                    X, norm = _station_arrays(v, m, gidx[q, :k])
                    obs = v["da"].var[days][:, gidx[q, :k]]
                    tasks.append((X, x0, dist[q], k, obs, norm, v["ptn"][q, m - 1]))
                    meta.append((m, q, k))
        res = _farm(tasks)
        ref = {}
        for (m, q, k), t, r in zip(meta, tasks, res):
            X, x0, dq, _, obs, norm, ptn = t
            kap = _kappa(X, x0, _weights(dq, k))
            ref[m, q, k] = dict(r, kappa=kap, hb=_hat_bound(kap, r["z"]), db=_daily_bound(kap, r["z"], obs, norm, ptn))
        out.append(dict(gidx=gidx, ref=ref))
    return out


def _batch(v, m):
    """Every (point, count) of test 1 as one batch: point q, count k at row q * len(COUNTS) + i."""
    nc, npt = len(COUNTS), v["lat"].size
    rep = lambda a: np.repeat(a, nc, axis=0)
    return (rep(v["lat"]), rep(v["lon"]), rep(v["elev"]), rep(v["tdi"]), rep(v["lst"]),
            np.tile(np.asarray(COUNTS, dtype=np.int32), npt), rep(v["ptn"][:, m - 1]))


# ---- 1. hat rows and dailies, both layouts --------------------------------------------------------------------------
@pytest.mark.gpu
def test_hat_rows_and_dailies_vs_exact(env, hat_ref):
    """gwr_hat and gwr_mth of both gather layouts against gwr_exact: hat rows within 64 eps kappa max|z*|, dailies within
    the daily bound, and within 1e-8 C for k >= 35.  The packed instance gives bitwise the values of the separate one."""
    stats, bad = _Stats(), []
    for w, (v, hr) in enumerate(zip(env["V"], hat_ref)):
        for m in MONTHS:
            lat, lon, elev, tdi, lst, nn, ptn = _batch(v, m)
            got = {}
            for lay in ("sep", "packed"):
                ctx = v["ctx"][lay]
                k, idx, z, st = ctx.gwr_hat(lat, lon, elev, tdi, lst, m, nnghs=nn)
                daily, st2 = ctx.gwr_mth(lat, lon, elev, tdi, lst, m, ptn, nnghs=nn)
                assert np.all(st == ST_OK) and np.all(st2 == ST_OK), (w, m, lay)
                assert np.array_equal(k, nn), (w, m, lay)
                got[lay] = (k, ctx.gidx[idx], z, daily)
                for r in range(nn.size):
                    q, kk = divmod(r, len(COUNTS))
                    kk = COUNTS[kk]
                    ref = hr["ref"][m, q, kk]
                    assert np.array_equal(ctx.gidx[idx[r, :kk]], hr["gidx"][q, :kk]), (w, m, lay, q, kk)
                    assert np.all(z[r, kk:] == 0.0)
                    ez = np.abs(z[r, :kk] - ref["z"]).max()
                    ed = np.abs(daily[r] - ref["v"])
                    big = "k>=35" if kk >= 35 else "k<35"
                    stats.add(("hat", lay, big), ez / ref["hb"], ez)
                    stats.add(("daily", lay, big), (ed / ref["db"]).max(), ed.max())
                    if ez > ref["hb"]:
                        bad.append(("hat row", w, m, lay, q, kk, ez, ref["hb"], ref["kappa"]))
                    if np.any(ed > ref["db"]) or (kk >= 35 and ed.max() > ABS_TOL_C):
                        bad.append(("daily", w, m, lay, q, kk, ed.max(), ref["db"].min(), ref["kappa"]))
            for a, b, what in zip(got["sep"], got["packed"], ("k", "idx", "z", "daily")):
                if not np.array_equal(a, b):
                    bad.append(("packed != sep", w, m, what))
    stats.report("GWR daily / hat-row instances against gwr_exact")
    assert not bad, (len(bad), bad[:10])


# ---- 2. cross validation, both layouts ------------------------------------------------------------------------------
@pytest.mark.gpu
def test_xval_vs_exact(env):
    """xval_anom (leave-one-out at 3 stations, every count of test 1, 12 months) of both layouts against gwr_exact:
    bias and MAE within the month's largest daily bound, r2 within 1e-9."""
    from topowx_b200 import db
    stats, bad = _Stats(), []
    counts = np.asarray(COUNTS, dtype=np.int32)
    for w, v in enumerate(env["V"]):
        sep = v["ctx"]["sep"]
        loc = sep.local_of_db[v["xv_db"]].astype(np.int32)
        s = v["da"].stns[v["xv_db"]]
        idx, dist, _, st = sep.knn(s[db.LAT], s[db.LON], 255, rm_idx=loc[:, None], rm_zero=True)
        assert np.all(st == 0)
        gidx = sep.gidx[idx]
        assert not np.isin(v["extra"], gidx) and not np.any(gidx == v["xv_db"][:, None])
        tasks, meta = [], []
        for m in range(1, 13):
            days = sep.mth_idx[m]
            for i in range(loc.size):
                x0 = [s[db.LON][i], s[db.LAT][i], s[db.ELEV][i], s[db.TDI][i], s[db.get_lst_varname(m)][i]]
                ptn = float(s[db.get_norm_varname(m)][i])
                own = v["da"].var[days, v["xv_db"][i]]
                for k in COUNTS:
                    X, norm = _station_arrays(v, m, gidx[i, :k])
                    obs = v["da"].var[days][:, gidx[i, :k]]
                    tasks.append((X, x0, dist[i], k, obs, norm, ptn, own))
                    meta.append((m, i, k))
        res = _farm(tasks)
        ref = {}
        for (m, i, k), t, r in zip(meta, tasks, res):
            X, x0, di, _, obs, norm, ptn, _ = t
            kap = _kappa(X, x0, _weights(di, k))
            ref[m, i, k] = dict(r, db=_daily_bound(kap, r["z"], obs, norm, ptn).max())
        got = {}
        for lay in ("sep", "packed"):
            ctx = v["ctx"][lay]
            li = ctx.local_of_db[v["xv_db"]].astype(np.int32)
            bias, mae, r2, st = ctx.xval_anom(li, counts)
            assert np.all(st == ST_OK)
            got[lay] = (bias, mae, r2)
            for (m, i, k), r in ref.items():
                c = COUNTS.index(k)
                eb, em = abs(bias[i, c, m - 1] - r["bias"]), abs(mae[i, c, m - 1] - r["mae"])
                er = abs(r2[i, c, m - 1] - r["r2"])
                big = "k>=35" if k >= 35 else "k<35"
                stats.add(("xval bias/mae", lay, big), max(eb, em) / r["db"], max(eb, em))
                stats.add(("xval r2", lay, big), er / R2_TOL, er)
                if eb > r["db"] or em > r["db"] or er > R2_TOL:
                    bad.append(("xval", w, lay, m, i, k, eb, em, r["db"], er))
        for a, b, what in zip(got["sep"], got["packed"], ("bias", "mae", "r2")):
            if not np.array_equal(a, b):
                bad.append(("packed != sep", w, what))
    stats.report("GWR cross-validation instances against gwr_exact")
    assert not bad, (len(bad), bad[:10])


# ---- 3. record path on packed tables at TWXI_MAX_NNGHS --------------------------------------------------------------
def _with_anom_counts(env, w, counts_by_month):
    """Copies of variable w's station DB whose optim_nnghs_anom is counts_by_month[m - 1] at every station, and the
    contexts of both layouts on them."""
    from topowx_b200 import db
    from topowx_b200.context import TwxiContext
    v = env["V"][w]
    s = v["da"].stns.copy()
    for m in range(1, 13):
        s[db.get_optim_anom_varname(m)] = float(counts_by_month[m - 1])
    d = db.StationSerialDataDb((s, v["da"].var, v["da"].days), v["da"].var_name)
    return {lay: TwxiContext(d, v["ctx"][lay].mask) for lay in ("sep", "packed")}


def _chunk(env):
    synth = env["synth"]
    wrk = synth.make_wrk_chk(env["f"], synth.TILE_ROW0 + 117, synth.TILE_COL0 + 109, 10, 12)
    wrk[2, 4, 5] = 0                                                  # one masked cell
    return wrk


def _tile(cmin, cmax, wrk, sizes):
    from topowx_b200.context import tile_begin, tile_days, tile_end
    shape = tile_begin(cmin, cmax, wrk)
    parts = [tile_days(cmin, cmax, n, shape) for n in sizes]
    out = dict(tile_end(cmin, cmax, shape))
    for k in ("tmin", "tmax"):
        out[k] = np.concatenate([p[k] for p in parts])
    return out


KEYS = ("tmin", "tmax", "tmin_norm", "tmax_norm", "tmin_se", "tmax_se", "ninvalid", "status")


@pytest.mark.gpu
def test_record_path_packed_at_max_nnghs(env):
    """Smoothed k_anom per month from {6, 13, 64, 128, 241, 254, 255} (hat rows of kh = 255): interp_chunk of both layouts
    and the day windows of the packed layout give the same bytes for every partition of 1995-1996."""
    from topowx_b200.context import interp_chunk
    vals = list(REC_COUNTS)
    counts = ([vals[(m * 3) % 7] for m in range(12)], [vals[(m * 5 + 6) % 7] for m in range(12)])
    assert all(set(c) == set(vals) for c in counts)
    c0, c1 = _with_anom_counts(env, 0, counts[0]), _with_anom_counts(env, 1, counts[1])
    for w, c in enumerate((c0, c1)):
        for lay in ("sep", "packed"):
            _, ka, _, st = c[lay].nngh_params(env["V"][0]["lat"][:6], env["V"][0]["lon"][:6])
            assert np.all(st == 0) and np.all(ka == np.asarray(counts[w])), (w, lay)
    wrk = _chunk(env)
    cells_lat, cells_lon = wrk[3].ravel(), wrk[4].ravel()
    for w, c in enumerate((c0, c1)):
        idx, _, _, _ = c["packed"].knn(cells_lat, cells_lon, 255)
        assert not np.isin(env["V"][w]["extra"], c["packed"].gidx[idx])
    ref = interp_chunk(c0["sep"], c1["sep"], wrk)
    assert np.all(ref["status"][wrk[2] != 0] == ST_OK) and ref["status"][4, 5] == ST_MASKED
    nd = env["days"].size
    feb96 = 365 + 31 + 14
    runs = {"interp_chunk packed": interp_chunk(c0["packed"], c1["packed"], wrk),
            "windows 1, 58, rest of 1995, 1996": _tile(c0["packed"], c1["packed"], wrk, [1, 58, 365 - 59, nd - 365]),
            "split inside February 1996": _tile(c0["packed"], c1["packed"], wrk, [feb96, nd - feb96]),
            "one window": _tile(c0["packed"], c1["packed"], wrk, [nd])}
    for what, out in runs.items():
        for k in KEYS:
            assert np.array_equal(np.asarray(ref[k]), np.asarray(out[k])), (what, k)


# ---- 4. fewer neighbours than coefficients --------------------------------------------------------------------------
@pytest.mark.gpu
def test_fewer_neighbours_than_coefficients_is_singular(env):
    """k = 1..5 < 6 coefficients: X'WX has rank <= k, so any finite output would be rounding noise.  gwr_hat / gwr_mth
    report TWXI_ST_SINGULAR, and a chunk whose smoothed k_anom is 5 in one month gets status 4 and fill values from
    interp_chunk and from the day windows."""
    from topowx_b200.context import interp_chunk
    for v in env["V"]:
        lat, lon, elev, tdi, lst, ptn = v["lat"], v["lon"], v["elev"], v["tdi"], v["lst"], v["ptn"]
        for lay in ("sep", "packed"):
            ctx = v["ctx"][lay]
            for k in range(1, 6):
                for m in (2, 7):
                    *_, st = ctx.gwr_hat(lat, lon, elev, tdi, lst, m, nnghs=k)
                    out, st2 = ctx.gwr_mth(lat, lon, elev, tdi, lst, m, ptn[:, m - 1], nnghs=k)
                    assert np.all(st == ST_SINGULAR) and np.all(st2 == ST_SINGULAR), (lay, k, m, st, st2)
                    assert np.all(np.isnan(out))
    counts = [64] * 12
    counts[8] = 5                                                      # September
    c0 = _with_anom_counts(env, 0, counts)
    c1 = _with_anom_counts(env, 1, [64] * 12)
    wrk = _chunk(env)
    live = wrk[2] != 0
    for lay in ("sep", "packed"):
        outs = [interp_chunk(c0[lay], c1[lay], wrk), _tile(c0[lay], c1[lay], wrk, [200, env["days"].size - 200])]
        for out in outs:
            st = np.asarray(out["status"])
            assert np.all(st[live] == ST_SINGULAR) and np.all(st[~live] == ST_MASKED), lay
            assert np.all(np.asarray(out["tmin"])[:, live] == FILL_I2) and np.all(np.asarray(out["tmax"])[:, live] == FILL_I2)
            assert np.all(np.asarray(out["ninvalid"])[live] == FILL_I4)
            for k in ("tmin_norm", "tmax_norm", "tmin_se", "tmax_se"):
                assert np.all(np.asarray(out[k])[:, live] == FILL_F4), (lay, k)
        for k in KEYS:
            assert np.array_equal(np.asarray(outs[0][k]), np.asarray(outs[1][k])), (lay, k)


# ---- 5. the reference itself (CPU) ----------------------------------------------------------------------------------
def test_exact_reference_matches_gwr_series_golden(golden_dir):
    """gwr_exact's solve against the reference's own _gwr_series vectors (tests/golden/gwr_series.npz): those are float64
    LAPACK results, so they agree to their own rounding (measured: <= 3.7e-12)."""
    g = np.load(os.path.join(golden_dir, "gwr_series.npz"))
    ctx = mpmath.workdps(DPS) if mpmath else _NoCtx()
    for c in range(6):
        with ctx:
            z = _hat_exact(g["X%d" % c], g["x%d" % c], [_num(t) for t in g["w%d" % c]])
            p = np.array([float(_dot(z, [_num(t) for t in row])) for row in g["y%d" % c]])
        np.testing.assert_allclose(p, g["p%d" % c], rtol=0, atol=1e-10)


def test_exact_reference_reproduces_constants_and_predictors():
    """On random neighbourhoods (k = 6 .. 255, elevations in metres, near-collinear lst) the hat row of gwr_exact
    reproduces the intercept and every predictor at the point: sum z = 1 and sum z_j x_j = x0 to 1e-30."""
    rng = np.random.default_rng(7)
    ctx = mpmath.workdps(DPS) if mpmath else _NoCtx()
    for k in (6, 7, 11, 40, 147, 255):
        lon, lat = rng.uniform(-101, -95, k), rng.uniform(36, 42, k)
        elev, tdi = rng.uniform(100, 3000, k), rng.uniform(0, 1, k)
        lst = 6.0 - 0.0055 * elev + rng.normal(0, 0.05, k)
        X = np.column_stack([lon, lat, elev, tdi, lst])
        x0 = [-98.0, 39.0, 1200.0, 0.4, -0.6]
        d = np.sort(rng.uniform(0, 150, k + 1))
        with ctx:
            w = [(1 - (_num(a) / _num(d[k])) ** 2) ** 2 for a in d[:k]]
            z = _hat_exact(X, x0, w)
            assert abs(sum(z) - 1) < 1e-30, k
            for a in range(5):
                assert abs(_dot(z, [_num(t) for t in X[:, a]]) - _num(x0[a])) < 1e-30, (k, a)
